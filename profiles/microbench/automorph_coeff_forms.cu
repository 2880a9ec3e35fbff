// automorph_coeff_forms.cu -- the two coefficient-domain Galois automorphism forms the library
// does not use at a given N, for tools/bench_rns_automorph.py.  It builds this file into a
// temporary shared object, calls it through ctypes on the same buffers as
// nttb200_rns_automorphism, times both in one run and compares the outputs word for word.
//
//   auto_coeff_cluster  N = 2^14..2^16: the row staged across a thread-block cluster of N / 2^13
//                       CTAs, each holding a contiguous 32 KiB slice; after cluster.sync() each CTA
//                       produces its slice of every output by gathering through distributed shared
//                       memory (map_shared_rank), and a final cluster.sync() keeps every slice alive
//                       until the peers are done.  (The library gathers from L2 at these sizes.)
//   auto_coeff_l2       any N: every source word gathered from L2 with a 4-byte __ldg, the form the
//                       library uses for N >= 2^14.  (At N <= 2^13 the library stages the row in
//                       one CTA's shared memory.)
// Both: out[c][row][j] = in[row][e] for e = j g_c^-1 mod 2N < N, q_l - in[row][e - N] otherwise.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cg = cooperative_groups;

struct Consts {
    uint32_t ginv[64];   // g^-1 mod 2N
    uint32_t q[32];
};

__device__ __forceinline__ uint32_t neg_if(uint32_t x, bool neg, uint32_t q) { return neg && x ? q - x : x; }

template <int CS>
__global__ void __launch_bounds__(256)
cluster_kernel(const uint4 *in, uint4 *out, uint64_t rows, uint64_t out_elem, uint32_t limbs, uint32_t count,
               const __grid_constant__ Consts k) {
    constexpr uint32_t kSlice = 8192, kN = kSlice * CS;
    constexpr int kVecs = kSlice / 4 / 256;
    __shared__ uint4 s4[kSlice / 4];
    uint32_t *s = reinterpret_cast<uint32_t *>(s4);
    cg::cluster_group cl = cg::this_cluster();
    const uint32_t rank = cl.block_rank();
    const uint64_t cid = blockIdx.x / CS, clusters = gridDim.x / CS;
    for (uint64_t row = cid; row < rows; row += clusters) {
        const uint32_t q = k.q[row % limbs];
        const uint64_t base = (row * kN + rank * kSlice) / 4;
        uint4 v[kVecs];
#pragma unroll
        for (int i = 0; i < kVecs; i++) v[i] = __ldcs(in + base + threadIdx.x + i * 256);
#pragma unroll
        for (int i = 0; i < kVecs; i++) s4[threadIdx.x + i * 256] = v[i];
        cl.sync();
        for (uint32_t c = 0; c < count; c++) {
            const uint32_t ginv = k.ginv[c];
#pragma unroll
            for (int i = 0; i < kVecs; i++) {
                const uint32_t j0 = rank * kSlice + (threadIdx.x + i * 256) * 4;
                uint32_t r[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const uint32_t src = ((j0 + e) * ginv) & (2 * kN - 1), w = src & (kN - 1);
                    r[e] = neg_if(*cl.map_shared_rank(s + (w & (kSlice - 1)), w / kSlice), src & kN, q);
                }
                __stcs(out + c * (out_elem / 4) + base + threadIdx.x + i * 256, make_uint4(r[0], r[1], r[2], r[3]));
            }
        }
        cl.sync();
    }
}

__global__ void __launch_bounds__(256)
l2_kernel(const uint32_t *__restrict__ in, uint4 *out, uint64_t items, uint64_t out_elem, uint32_t logn,
          uint32_t limbs, uint32_t count, const __grid_constant__ Consts k) {
    const uint32_t n = 1u << logn, log_c = logn - 12;
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint64_t row = it >> log_c;
        const uint32_t q = k.q[row % limbs];
        const uint32_t *src = in + (row << logn);
        for (uint32_t c = 0; c < count; c++) {
            const uint32_t ginv = k.ginv[c];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const uint32_t j0 = (((uint32_t) it & ((1u << log_c) - 1)) << 12) + (threadIdx.x + i * 256) * 4;
                uint32_t r[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const uint32_t s = ((j0 + e) * ginv) & (2 * n - 1);
                    r[e] = neg_if(__ldg(src + (s & (n - 1))), s & n, q);
                }
                __stcs(out + (c * out_elem + (row << logn) + j0) / 4, make_uint4(r[0], r[1], r[2], r[3]));
            }
        }
    }
}

static Consts consts(uint32_t logn, uint32_t limbs, const uint32_t *qs, const uint32_t *galois, uint32_t count) {
    Consts k = {};
    for (uint32_t c = 0; c < count; c++) {
        uint32_t x = galois[c];
        for (int i = 0; i < 5; i++) x *= 2u - galois[c] * x;   // g^-1 mod 2^32
        k.ginv[c] = x & ((2u << logn) - 1);
    }
    for (uint32_t l = 0; l < limbs; l++) k.q[l] = qs[l];
    return k;
}

template <int CS>
static cudaError_t cluster_launch(const int32_t *in, int32_t *out, uint64_t rows, uint32_t limbs, uint32_t count,
                                  const Consts &k, int sm_count) {
    const uint64_t cap = (uint64_t) sm_count * 6 / CS;   // clusters: 6 CTAs of 32 KiB per SM
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned) ((rows < cap ? rows : cap) * CS));
    cfg.blockDim = dim3(256);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, cluster_kernel<CS>, reinterpret_cast<const uint4 *>(in),
                              reinterpret_cast<uint4 *>(out), rows, rows * 8192 * CS, limbs, count, k);
}

extern "C" int auto_coeff_cluster(const int32_t *in, int32_t *out, uint64_t rows, uint32_t logn, uint32_t limbs,
                                  const uint32_t *qs, const uint32_t *galois, uint32_t count, int sm_count) {
    const Consts k = consts(logn, limbs, qs, galois, count);
    cudaError_t e;
    switch (logn) {
        case 14: e = cluster_launch<2>(in, out, rows, limbs, count, k, sm_count); break;
        case 15: e = cluster_launch<4>(in, out, rows, limbs, count, k, sm_count); break;
        case 16: e = cluster_launch<8>(in, out, rows, limbs, count, k, sm_count); break;
        default: return (int) cudaErrorInvalidValue;
    }
    return e != cudaSuccess ? (int) e : (int) cudaGetLastError();
}

extern "C" int auto_coeff_l2(const int32_t *in, int32_t *out, uint64_t rows, uint32_t logn, uint32_t limbs,
                             const uint32_t *qs, const uint32_t *galois, uint32_t count, int sm_count) {
    const Consts k = consts(logn, limbs, qs, galois, count);
    const uint64_t items = rows << (logn - 12), cap = (uint64_t) sm_count * 8;
    l2_kernel<<<(unsigned) (items < cap ? items : cap), 256>>>(reinterpret_cast<const uint32_t *>(in),
                                                              reinterpret_cast<uint4 *>(out), items, rows << logn,
                                                              logn, limbs, count, k);
    return (int) cudaGetLastError();
}
