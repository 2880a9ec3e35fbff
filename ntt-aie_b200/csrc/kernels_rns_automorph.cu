// kernels_rns_automorph.cu -- Galois automorphisms sigma_g : a(X) -> a(X^g) mod (X^N + 1) on RNS
// batches ([batch][L][N] rows), count automorphisms of the same input in one launch (hoisting).
//
//   rns_auto_eval_kernel       evaluation domain (the order of nttb200_rns_ct_batch: index k holds
//                              a(psi^(2 brev(k) + 1))): out[k] = in[brev((g brev(k) + (g-1)/2) mod N)],
//                              one permutation for every channel and every psi.  Output block t
//                              (4096 words) gathers from input block brev_s((g brev_s(t) + (g-1)/2)
//                              mod 2^s) only, s = logn - 12.  Work item = one source block of one
//                              row, loaded once into 16 KiB of shared memory; for each of the count
//                              elements the block writes the output block whose source it is:
//                              brev_s(g^-1 (brev_s(src) - (g-1)/2) mod 2^s).  The input is read
//                              once per call whatever count is.
//   rns_auto_coeff_kernel<LOGN>, rns_auto_coeff_l2_kernel
//                              coefficient domain: e = j g^-1 mod 2N, out[j] = in[e] for e < N,
//                              q_l - in[e - N] (0 for 0) otherwise.  The source of a word can be
//                              anywhere in its row.  N <= 2^13: one CTA stages the row (16 or 32
//                              KiB) in shared memory and gathers from there.  N >= 2^14: each
//                              word is gathered straight from L2.  The alternative above 2^13,
//                              a row staged across a cluster of N / 2^13 CTAs and gathered
//                              through distributed shared memory, measured 1.6-4x slower on the
//                              B200 (DESIGN 3.6) and is kept only in profiles/microbench.
// Streamed loads and stores are 128-bit with evict-first hints.  Every pointer is 16-byte aligned
// (checked by the host), every index 64-bit.
#include "modarith.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kA_Threads = 256;
constexpr int kA_BlockWords = 4096;                          // evaluation-domain work item
constexpr int kA_BlockVecs = kA_BlockWords / 4 / kA_Threads;   // uint4 per thread

// items = rows << (logn - 12); out_elem = words of one output element (rows * N)
__global__ void __launch_bounds__(kA_Threads)
rns_auto_eval_kernel(const uint4 *in, uint4 *out, uint64_t items, uint64_t out_elem, uint32_t logn,
                     uint32_t count, const __grid_constant__ RnsAutoConsts k) {
    __shared__ uint4 s4[kA_BlockWords / 4];
    const uint32_t *s = reinterpret_cast<const uint32_t *>(s4);
    const uint32_t log_b = logn - 12, bmask = (1u << log_b) - 1, nmask = (1u << logn) - 1;
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        uint4 v[kA_BlockVecs];
#pragma unroll
        for (int i = 0; i < kA_BlockVecs; i++) v[i] = __ldcs(in + it * (kA_BlockWords / 4) + threadIdx.x + i * kA_Threads);
        __syncthreads();   // the previous item's gathers are done
#pragma unroll
        for (int i = 0; i < kA_BlockVecs; i++) s4[threadIdx.x + i * kA_Threads] = v[i];
        __syncthreads();
        const uint64_t row_base = (it >> log_b) << logn;   // first word of the row
        const uint32_t src_r = log_b ? __brev((uint32_t) it & bmask) >> (32 - log_b) : 0;
        for (uint32_t c = 0; c < count; c++) {
            const uint32_t g = k.g[c] & nmask, off = k.off[c];
            const uint32_t t = log_b ? __brev(((src_r - off) * k.ginv[c]) & bmask) >> (32 - log_b) : 0;
            uint4 *dst = out + (c * out_elem + row_base + ((uint64_t) t << 12)) / 4;
#pragma unroll
            for (int i = 0; i < kA_BlockVecs; i++) {
                const uint32_t k0 = (t << 12) + (threadIdx.x + i * kA_Threads) * 4;
                uint32_t r[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    r[e] = s[brev_n((g * brev_n(k0 + e, logn) + off) & nmask, logn) & (kA_BlockWords - 1)];
                }
                __stcs(dst + threadIdx.x + i * kA_Threads, make_uint4(r[0], r[1], r[2], r[3]));
            }
        }
    }
}

// N <= 2^13: the row (2^LOGN words, at most 32 KiB) is staged in the block's shared memory.
template <int LOGN>
__global__ void __launch_bounds__(kA_Threads)
rns_auto_coeff_kernel(const uint4 *in, uint4 *out, uint64_t rows, uint64_t out_elem, uint32_t limbs,
                      uint32_t count, const __grid_constant__ RnsAutoConsts k) {
    constexpr uint32_t kN = 1u << LOGN;
    constexpr int kVecs = kN / 4 / kA_Threads;   // uint4 of the row per thread
    __shared__ uint4 s4[kN / 4];
    const uint32_t *s = reinterpret_cast<const uint32_t *>(s4);
    for (uint64_t row = blockIdx.x; row < rows; row += gridDim.x) {
        const uint32_t q = k.q[row % limbs];
        uint4 v[kVecs];
#pragma unroll
        for (int i = 0; i < kVecs; i++) v[i] = __ldcs(in + row * (kN / 4) + threadIdx.x + i * kA_Threads);
        __syncthreads();   // the previous row's gathers are done
#pragma unroll
        for (int i = 0; i < kVecs; i++) s4[threadIdx.x + i * kA_Threads] = v[i];
        __syncthreads();
        for (uint32_t c = 0; c < count; c++) {
            const uint32_t ginv = k.ginv[c];
            uint4 *dst = out + (c * out_elem + row * kN) / 4;
#pragma unroll
            for (int i = 0; i < kVecs; i++) {
                const uint32_t j0 = (threadIdx.x + i * kA_Threads) * 4;
                uint32_t r[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const uint32_t src = ((j0 + e) * ginv) & (2 * kN - 1);   // mod 2^32 first: 2N | 2^32
                    const uint32_t x = s[src & (kN - 1)];
                    r[e] = (src & kN) ? sub_mod(0, x, q) : x;
                }
                __stcs(dst + threadIdx.x + i * kA_Threads, make_uint4(r[0], r[1], r[2], r[3]));
            }
        }
    }
}

// N >= 2^14: every source word gathered from L2 (4-byte __ldg).  Work item = 4096 consecutive
// output words of one row; consecutive blocks take consecutive chunks of the same row, so the rows
// in flight (about 1184 chunks, 18 MiB at N = 2^16) stay L2-resident while they are gathered.
__global__ void __launch_bounds__(kA_Threads)
rns_auto_coeff_l2_kernel(const uint32_t *__restrict__ in, uint4 *out, uint64_t items, uint64_t out_elem,
                         uint32_t logn, uint32_t limbs, uint32_t count, const __grid_constant__ RnsAutoConsts k) {
    const uint32_t n = 1u << logn, log_c = logn - 12;
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint64_t row = it >> log_c;
        const uint32_t q = k.q[row % limbs];
        const uint32_t *src = in + (row << logn);
        const uint32_t chunk = ((uint32_t) it & ((1u << log_c) - 1)) << 12;
        for (uint32_t c = 0; c < count; c++) {
            const uint32_t ginv = k.ginv[c];
#pragma unroll
            for (int i = 0; i < kA_BlockVecs; i++) {
                const uint32_t j0 = chunk + (threadIdx.x + i * kA_Threads) * 4;
                uint32_t r[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const uint32_t s = ((j0 + e) * ginv) & (2 * n - 1);
                    const uint32_t x = __ldg(src + (s & (n - 1)));
                    r[e] = (s & n) ? sub_mod(0, x, q) : x;
                }
                __stcs(out + (c * out_elem + (row << logn) + j0) / 4, make_uint4(r[0], r[1], r[2], r[3]));
            }
        }
    }
}

int launch_rns_automorph(const nttb200_rns_plan *rp, const int32_t *in, int32_t *out, size_t batch,
                         const uint32_t *galois, uint32_t count, bool eval, cudaStream_t st) {
    const uint32_t logn = rp->logn;
    const uint32_t two_n_mask = (2u << logn) - 1;
    RnsAutoConsts k{};
    for (uint32_t c = 0; c < count; c++) {
        k.g[c] = galois[c];
        k.ginv[c] = inv_mod_2_32(galois[c]) & two_n_mask;   // g^-1 mod 2^32 is g^-1 mod 2N
        k.off[c] = ((galois[c] - 1) / 2) & (two_n_mask >> 1);
    }
    for (uint32_t l = 0; l < rp->limbs; l++) k.q[l] = rp->pos[l].x;
    const uint64_t rows = (uint64_t) batch * rp->limbs, out_elem = rows << logn;
    if (eval) {
        const uint64_t items = rows << (logn - 12);
        const uint64_t cap = (uint64_t) rp->sm_count * 8;
        rns_auto_eval_kernel<<<(unsigned) (items < cap ? items : cap), kA_Threads, 0, st>>>(
            reinterpret_cast<const uint4 *>(in), reinterpret_cast<uint4 *>(out), items, out_elem, logn, count, k);
    } else {
        const uint4 *in4 = reinterpret_cast<const uint4 *>(in);
        uint4 *out4 = reinterpret_cast<uint4 *>(out);
        const uint64_t cap = (uint64_t) rp->sm_count * 8;
        if (logn <= 13) {
            const unsigned grid = (unsigned) (rows < cap ? rows : cap);
            if (logn == 12) {
                rns_auto_coeff_kernel<12><<<grid, kA_Threads, 0, st>>>(in4, out4, rows, out_elem, rp->limbs, count, k);
            } else {
                rns_auto_coeff_kernel<13><<<grid, kA_Threads, 0, st>>>(in4, out4, rows, out_elem, rp->limbs, count, k);
            }
        } else {
            const uint64_t items = rows << (logn - 12);
            rns_auto_coeff_l2_kernel<<<(unsigned) (items < cap ? items : cap), kA_Threads, 0, st>>>(
                reinterpret_cast<const uint32_t *>(in), out4, items, out_elem, logn, rp->limbs, count, k);
        }
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

}  // namespace nttb200
