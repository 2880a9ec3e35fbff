// kernels_generic.cu -- stage-pass kernels that serve EVERY (logn, stage range).
//
// One pass = one HBM read + one HBM write of the data.  A pass applies a run of
// consecutive butterfly stages [s0, s0+ns) to tiles held in shared memory:
//   tile = 2^ns rows (the bits s0..s0+ns-1 of the coefficient index, i.e. the
//          bits those stages pair up) x 2^logc contiguous columns (the lowest
//          index bits, so every global access is a coalesced >=128 B run).
// This is the CUDA successor of the reference's tiling plan (src/aie2.py:161-317:
// tile-local stages on a contiguous slice, then cross-tile stages on strided
// partners) with shared memory in the role of the AIE tile memory and the pass
// structure in the role of the neighbour-memory exchanges + swap_buff
// (src/aie_core.cc:133-143).  Butterfly arithmetic follows the golden exactly
// (src/test.cpp:46-50); twiddle index is table[h + i] (src/test.cpp:45).
//
// These kernels keep every intermediate canonical; they are the always-correct
// path (any N up to 2^27, partial depth via stage_limit, CT and GS) and the
// second pass of large transforms.  The throughput path for the benchmark sizes
// is kernels_fused.cu.
#include "modarith.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kGenThreads = 512;
constexpr int kGenLogTile = 12;  // 4096 words = 16 KiB of shared memory per CTA

struct PassParams {
    uint32_t logn;
    uint32_t s0;      // first (lowest-stride) stage of the pass
    uint32_t ns;      // number of stages in the pass
    uint32_t logc;    // log2 columns
    uint32_t q;
    uint32_t permute;  // apply ans_order on store (src/test.cpp:69-71,212-219)
    uint64_t tiles;    // total tiles over the whole batch
};

// ans_order = {0,2,1,3,8,10,9,11,4,6,5,7,12,14,13,15}: swap the two bits inside
// each bit pair of the 4-bit block index (b3b2b1b0 -> b2b3b0b1).
__device__ __forceinline__ uint32_t ans_order_block(uint32_t b) {
    return ((b & 0x5u) << 1) | ((b & 0xAu) >> 1);
}

template <bool CT>
__global__ void __launch_bounds__(kGenThreads)
stage_pass_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out,
                  const uint2 *__restrict__ tw, PassParams pp) {
    extern __shared__ uint32_t sm[];
    const uint32_t q = pp.q;
    const uint32_t logtile = pp.ns + pp.logc;
    const uint32_t tile = 1u << logtile;
    // the tile's 2^ns - 1 twiddles, staged once per tile so the per-stage dependent
    // global loads (one L2 round trip per stage) leave the critical path:
    // ltw[(R >> (k+1)) + blk] = table[(n >> (s0+k+1)) + (high << (ns-k-1)) + blk]
    uint2 *ltw = reinterpret_cast<uint2 *>(sm + tile);
    const uint32_t rows = 1u << pp.ns;
    const uint32_t cmask = (1u << pp.logc) - 1u;
    const uint32_t lowhi_bits = pp.s0 - pp.logc;          // index bits between columns and rows
    const uint32_t tiles_per_poly_log = pp.logn - logtile;
    const uint32_t n = 1u << pp.logn;

    for (uint64_t t = blockIdx.x; t < pp.tiles; t += gridDim.x) {
        const uint64_t poly = t >> tiles_per_poly_log;
        const uint32_t tin = (uint32_t) (t & ((1ull << tiles_per_poly_log) - 1ull));
        const uint32_t lowhi = tin & ((1u << lowhi_bits) - 1u);
        const uint32_t high = tin >> lowhi_bits;
        // global index of tile element (r, c):
        //   (high << (s0+ns)) | (r << s0) | (lowhi << logc) | c
        const uint32_t base = (high << (pp.s0 + pp.ns)) | (lowhi << pp.logc);
        const uint32_t *src = in + poly * n;
        uint32_t *dst = out + poly * n;

        for (uint32_t e = threadIdx.x; e < tile; e += kGenThreads) {
            uint32_t r = e >> pp.logc, c = e & cmask;
            sm[e] = src[base | (r << pp.s0) | c];
        }
        for (uint32_t e = threadIdx.x + 1; e < rows; e += kGenThreads) {
            // entry e = hk + blk with hk = rows >> (k+1) the leading power of two of e
            uint32_t lvl = 31u - __clz(e);               // hk = 1 << lvl, k = ns - 1 - lvl
            uint32_t blk = e - (1u << lvl);
            uint32_t k = pp.ns - 1u - lvl;
            ltw[e] = __ldg(&tw[(n >> (pp.s0 + k + 1)) + (high << lvl) + blk]);
        }
        __syncthreads();

        for (uint32_t kk = 0; kk < pp.ns; kk++) {
            const uint32_t k = CT ? (pp.ns - 1 - kk) : kk;  // CT: large stride first
            const uint32_t hk = rows >> (k + 1);
            for (uint32_t b = threadIdx.x; b < (tile >> 1); b += kGenThreads) {
                uint32_t rr = b >> pp.logc, c = b & cmask;
                uint32_t r0 = ((rr >> k) << (k + 1)) | (rr & ((1u << k) - 1u));
                uint32_t i0 = (r0 << pp.logc) | c;
                uint32_t i1 = i0 + (1u << (k + pp.logc));
                uint2 w = ltw[hk + (r0 >> (k + 1))];
                uint32_t x = sm[i0], y = sm[i1];
                if (CT) {
                    uint32_t v = shoup_mul(y, w.x, w.y, q);
                    sm[i0] = add_mod(x, v, q);
                    sm[i1] = sub_mod(x, v, q);
                } else {
                    sm[i0] = add_mod(x, y, q);
                    sm[i1] = shoup_mul(x + q - y, w.x, w.y, q);
                }
            }
            __syncthreads();
        }

        for (uint32_t e = threadIdx.x; e < tile; e += kGenThreads) {
            uint32_t r = e >> pp.logc, c = e & cmask;
            uint32_t g = base | (r << pp.s0) | c;
            if (pp.permute) {
                uint32_t sh = pp.logn - 4;
                g = (ans_order_block(g >> sh) << sh) | (g & ((1u << sh) - 1u));
            }
            dst[g] = sm[e];
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
pointwise_kernel(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b,
                 uint32_t *__restrict__ c, size_t count4, size_t count, uint32_t q, uint64_t mu) {
    size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t) gridDim.x * blockDim.x;
    for (size_t v = i; v < count4; v += stride) {
        uint4 x = reinterpret_cast<const uint4 *>(a)[v];
        uint4 y = reinterpret_cast<const uint4 *>(b)[v];
        uint4 z;
        z.x = barrett_mul(x.x, y.x, q, mu);
        z.y = barrett_mul(x.y, y.y, q, mu);
        z.z = barrett_mul(x.z, y.z, q, mu);
        z.w = barrett_mul(x.w, y.w, q, mu);
        reinterpret_cast<uint4 *>(c)[v] = z;
    }
    for (size_t v = count4 * 4 + i; v < count; v += stride) {
        c[v] = barrett_mul(a[v], b[v], q, mu);
    }
}

__global__ void __launch_bounds__(256)
scale_kernel(const uint32_t *__restrict__ a, uint32_t *__restrict__ c, size_t count4, size_t count,
             uint32_t q, uint32_t s, uint32_t sp) {
    size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t) gridDim.x * blockDim.x;
    for (size_t v = i; v < count4; v += stride) {
        uint4 x = reinterpret_cast<const uint4 *>(a)[v];
        x.x = shoup_mul(x.x, s, sp, q);
        x.y = shoup_mul(x.y, s, sp, q);
        x.z = shoup_mul(x.z, s, sp, q);
        x.w = shoup_mul(x.w, s, sp, q);
        reinterpret_cast<uint4 *>(c)[v] = x;
    }
    for (size_t v = count4 * 4 + i; v < count; v += stride) {
        c[v] = shoup_mul(a[v], s, sp, q);
    }
}

static int grid_for(uint64_t work_items, int sm_count, int per_sm) {
    uint64_t cap = (uint64_t) sm_count * per_sm;
    return (int) (work_items < cap ? (work_items ? work_items : 1) : cap);
}

// per-device one-time setup (called from plan creation with the plan's device current):
// 16 KiB of data + up to 32 KiB of staged twiddles per CTA
int generic_prepare() {
    NTTB200_CUDA(cudaFuncSetAttribute(stage_pass_kernel<true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, 49152));
    NTTB200_CUDA(cudaFuncSetAttribute(stage_pass_kernel<false>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, 49152));
    return NTTB200_OK;
}

int launch_generic(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch, int sb,
                   int se, bool ct, bool permute_out, cudaStream_t st) {
    if (batch == 0 || sb >= se) {
        return NTTB200_OK;
    }

    // split [sb, se) into passes, each as deep as a 4096-word tile allows
    struct Pass {
        int s0, ns, logc;
    } passes[32];
    int np = 0;
    for (int s = sb; s < se;) {
        int logc = s < 5 ? s : 5;
        int ns = kGenLogTile - logc;
        if (ns > se - s) ns = se - s;
        passes[np++] = {s, ns, logc};
        s += ns;
    }
    // The ans_order store permutes the top four index bits.  It is race-free in
    // place only when those bits are row bits of the storing tile (the tile then
    // writes exactly the addresses it read), i.e. the last pass needs >= 4 stages.
    if (permute_out && np >= 2 && passes[np - 1].ns < 4) {
        int take = 4 - passes[np - 1].ns;
        passes[np - 2].ns -= take;
        passes[np - 1].s0 -= take;
        passes[np - 1].ns = 4;
        passes[np - 1].logc = passes[np - 1].s0 < 5 ? passes[np - 1].s0 : 5;
    }
    const uint32_t *src = reinterpret_cast<const uint32_t *>(d_in);
    uint32_t *dst = reinterpret_cast<uint32_t *>(d_out);
    for (int k = 0; k < np; k++) {
        const Pass &ps = ct ? passes[np - 1 - k] : passes[k];  // CT: largest strides first
        PassParams pp;
        pp.logn = p->logn;
        pp.s0 = (uint32_t) ps.s0;
        pp.ns = (uint32_t) ps.ns;
        pp.logc = (uint32_t) ps.logc;
        pp.q = p->q;
        pp.permute = (permute_out && k == np - 1) ? 1u : 0u;
        pp.tiles = (uint64_t) batch << (p->logn - (uint32_t) (ps.ns + ps.logc));
        size_t smem = (sizeof(uint32_t) << (ps.ns + ps.logc)) + (sizeof(uint2) << ps.ns);
        int grid = grid_for(pp.tiles, p->sm_count, 8);
        if (ct) {
            stage_pass_kernel<true><<<grid, kGenThreads, smem, st>>>(src, dst, p->d_tw, pp);
        } else {
            stage_pass_kernel<false><<<grid, kGenThreads, smem, st>>>(src, dst, p->d_tw, pp);
        }
        g_launches.fetch_add(1, std::memory_order_relaxed);
        NTTB200_CUDA(cudaGetLastError());
        src = dst;  // later passes run in place on the output
    }
    return NTTB200_OK;
}

// The uint4 loop of pointwise/scale needs every pointer 16-byte aligned; any other
// 4-byte-aligned views (t[1:], one RNS channel, ...) take the scalar loop only.
static bool vec_ok(const void *x, const void *y, const void *z) {
    return !(((uintptr_t) x | (uintptr_t) y | (uintptr_t) z) & 15u);
}

int launch_pointwise(nttb200_plan *p, const int32_t *a, const int32_t *b, int32_t *c, size_t count,
                     cudaStream_t st) {
    if (count == 0) return NTTB200_OK;
    const bool vec = vec_ok(a, b, c);
    size_t count4 = vec ? count / 4 : 0;
    int grid = grid_for(((vec ? count4 : count) + 255) / 256 + 1, p->sm_count, 16);
    pointwise_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const uint32_t *>(a),
                                           reinterpret_cast<const uint32_t *>(b),
                                           reinterpret_cast<uint32_t *>(c), count4, count, p->q,
                                           p->mu);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

int launch_scale(nttb200_plan *p, const int32_t *a, int32_t *c, size_t count, uint32_t s,
                 uint32_t s_shoup, cudaStream_t st) {
    if (count == 0) return NTTB200_OK;
    const bool vec = vec_ok(a, a, c);
    size_t count4 = vec ? count / 4 : 0;
    int grid = grid_for(((vec ? count4 : count) + 255) / 256 + 1, p->sm_count, 16);
    scale_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const uint32_t *>(a),
                                       reinterpret_cast<uint32_t *>(c), count4, count, p->q, s,
                                       s_shoup);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

}  // namespace nttb200
