// kernels_rns_eval.cu -- evaluation-domain arithmetic on RNS batches ([batch][L][N], channel l
// of polynomial b at (b*L + l)*N, modulo q_l).
//
//   rns_stream_kernel<OP, BCAST>  c = a + b, a - b, a * b (OP 0..2) or a * s_l (OP 3), one
//                                 launch for every channel.  Work item = one 16 KiB tile
//                                 (1024 uint4) of one channel row: N >= 4096, so a tile never
//                                 straddles two channels, and the channel -- hence q_l and its
//                                 constants, read from the kernel-parameter bank -- is uniform
//                                 across the block.  BCAST: b is one [L][N] operand shared by
//                                 the batch (at most 8 MiB, read through L2; the streamed a and
//                                 c carry evict-first hints so that they do not push it out).
//   rns_dot_kernel<G, WB>         c = (acc ? c : 0) + sum_k a_k * w_k: the products are summed
//                                 exactly in 64 bits and folded (reduced mod q_l) every 16
//                                 terms:  q + 16 (q-1)^2 < 2^30 + 2^64 - 2^35 < 2^64 for
//                                 q <= 2^30.  A thread keeps the accumulators of G polynomials
//                                 at the same (l, i); with WB (one key for the whole batch) each
//                                 key word is loaded once per group instead of once per
//                                 polynomial.
// Every pointer is 16-byte aligned (checked by the host), every index 64-bit.
#include "modarith.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kE_Threads = 256;
constexpr int kE_TileVecs = 1024;               // uint4 per streaming work item (4096 words)
constexpr int kE_PerThread = kE_TileVecs / kE_Threads;
constexpr int kE_MaxChannels = 32;
constexpr int kE_DotGroupShared = 8;            // G of rns_dot with one shared key (ptxas: no spills)
constexpr int kE_DotGroupOwn = 2;               // G with one key per polynomial

// per-channel constants, kernel parameters: q_l, floor(2^64 / q_l) for reduce64, and the
// scalar of rns_scale with its Shoup companion
struct RnsEvalConsts {
    uint64_t mu[kE_MaxChannels];
    uint32_t q[kE_MaxChannels];
    uint32_t s[kE_MaxChannels];
    uint32_t sp[kE_MaxChannels];
};

template <int OP>
__device__ __forceinline__ uint32_t stream_op(uint32_t a, uint32_t b, uint32_t q, uint64_t mu, uint32_t s,
                                              uint32_t sp) {
    if (OP == 0) return add_mod(a, b, q);
    if (OP == 1) return sub_mod(a, b, q);
    if (OP == 2) return reduce64((uint64_t) a * b, q, mu);
    return shoup_mul(a, s, sp, q);
}

template <int OP>
__device__ __forceinline__ uint4 stream_op4(uint4 a, uint4 b, uint32_t q, uint64_t mu, uint32_t s,
                                            uint32_t sp) {
    return make_uint4(stream_op<OP>(a.x, b.x, q, mu, s, sp), stream_op<OP>(a.y, b.y, q, mu, s, sp),
                      stream_op<OP>(a.z, b.z, q, mu, s, sp), stream_op<OP>(a.w, b.w, q, mu, s, sp));
}

// tiles = batch * L * N / 4096; a row (one channel of one polynomial) is 2^log_g tiles
template <int OP, bool BCAST>
__global__ void __launch_bounds__(kE_Threads)
rns_stream_kernel(const uint4 *a, const uint4 *b, uint4 *c, uint64_t tiles, uint32_t log_g, uint32_t limbs,
                  const __grid_constant__ RnsEvalConsts k) {
    const uint64_t chan_tiles = (uint64_t) limbs << log_g;   // tiles of one polynomial
    for (uint64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        const uint32_t l = (uint32_t) ((t >> log_g) % limbs);
        const uint32_t q = k.q[l], s = k.s[l], sp = k.sp[l];
        const uint64_t mu = k.mu[l];
        const uint64_t base = t * kE_TileVecs + threadIdx.x;
        const uint64_t b_base = (BCAST ? t % chan_tiles : t) * kE_TileVecs + threadIdx.x;
        uint4 x[kE_PerThread], y[kE_PerThread];
#pragma unroll
        for (int i = 0; i < kE_PerThread; i++) {
            x[i] = __ldcs(a + base + i * kE_Threads);
            if (OP == 3) {
                y[i] = x[i];
            } else if (BCAST) {
                y[i] = __ldg(b + b_base + i * kE_Threads);
            } else {
                y[i] = __ldcs(b + b_base + i * kE_Threads);
            }
        }
#pragma unroll
        for (int i = 0; i < kE_PerThread; i++) {
            __stcs(c + base + i * kE_Threads, stream_op4<OP>(x[i], y[i], q, mu, s, sp));
        }
    }
}

// Work item = (group of G polynomials, channel l, chunk of 256 uint4 of the row); a row holds
// N/1024 >= 4 chunks (2^log_c).  a: [terms][batch][L][N], w: [terms][WB ? 1 : batch][L][N].
template <int G, bool WB>
__global__ void __launch_bounds__(kE_Threads)
rns_dot_kernel(const uint4 *a, const uint4 *w, uint4 *c, uint32_t terms, uint64_t batch, uint32_t limbs,
               uint32_t log_c, uint64_t items, int accumulate, const __grid_constant__ RnsEvalConsts k) {
    const uint64_t row_vecs = (uint64_t) kE_Threads << log_c;   // N / 4
    const uint64_t poly_vecs = row_vecs * limbs;
    const uint64_t a_term = poly_vecs * batch, w_term = WB ? poly_vecs : a_term;
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint64_t rest = it >> log_c;
        const uint32_t l = (uint32_t) (rest % limbs);
        const uint64_t b0 = rest / limbs * G;
        const uint32_t q = k.q[l];
        const uint64_t mu = k.mu[l];
        const uint64_t v = (uint64_t) l * row_vecs + ((it & ((1u << log_c) - 1)) << 8) + threadIdx.x;
        const int gn = batch - b0 < (uint64_t) G ? (int) (batch - b0) : G;   // uniform: ragged last group
        uint64_t acc[G][4];
#pragma unroll
        for (int g = 0; g < G; g++) {
            uint4 x = make_uint4(0, 0, 0, 0);
            if (accumulate && g < gn) x = c[(b0 + g) * poly_vecs + v];
            acc[g][0] = x.x;
            acc[g][1] = x.y;
            acc[g][2] = x.z;
            acc[g][3] = x.w;
        }
        for (uint32_t k0 = 0; k0 < terms; k0 += 16) {
            const uint32_t k1 = terms - k0 < 16u ? terms : k0 + 16;
            for (uint32_t kk = k0; kk < k1; kk++) {
                // every load of the term is issued before the first product: the last polynomial
                // of a ragged group stands in for the missing ones (their sums are not stored), so
                // the loads need no branch
                uint4 x[G], y[WB ? 1 : G];
#pragma unroll
                for (int g = 0; g < G; g++) {
                    const uint64_t pg = (b0 + (g < gn ? g : gn - 1)) * poly_vecs + v;
                    x[g] = __ldcs(a + kk * a_term + pg);
                    if (!WB) y[g] = __ldcs(w + kk * w_term + pg);
                }
                if (WB) y[0] = __ldg(w + kk * w_term + v);
#pragma unroll
                for (int g = 0; g < G; g++) {
                    const uint4 yg = y[WB ? 0 : g];
                    acc[g][0] += (uint64_t) x[g].x * yg.x;
                    acc[g][1] += (uint64_t) x[g].y * yg.y;
                    acc[g][2] += (uint64_t) x[g].z * yg.z;
                    acc[g][3] += (uint64_t) x[g].w * yg.w;
                }
            }
#pragma unroll
            for (int g = 0; g < G; g++) {   // fold: every accumulator back below q
#pragma unroll
                for (int e = 0; e < 4; e++) acc[g][e] = reduce64(acc[g][e], q, mu);
            }
        }
#pragma unroll
        for (int g = 0; g < G; g++) {
            if (g < gn) {
                __stcs(c + (b0 + g) * poly_vecs + v, make_uint4((uint32_t) acc[g][0], (uint32_t) acc[g][1],
                                                                (uint32_t) acc[g][2], (uint32_t) acc[g][3]));
            }
        }
    }
}

static RnsEvalConsts eval_consts(const nttb200_rns_plan *rp, const uint32_t *scalars) {
    RnsEvalConsts k{};
    for (uint32_t l = 0; l < rp->limbs; l++) {
        const uint32_t q = rp->pos[l].x;
        k.q[l] = q;
        k.mu[l] = (uint64_t) ((((unsigned __int128) 1) << 64) / q);
        if (scalars) {
            k.s[l] = scalars[l];
            k.sp[l] = (uint32_t) (((uint64_t) scalars[l] << 32) / q);
        }
    }
    return k;
}

static int eval_grid(const nttb200_rns_plan *rp, uint64_t items) {
    const uint64_t cap = (uint64_t) rp->sm_count * 8;
    return (int) (items < cap ? items : cap);
}

template <int OP, bool BCAST>
static void stream_launch(int grid, const int32_t *a, const int32_t *b, int32_t *c, uint64_t tiles,
                          uint32_t log_g, uint32_t limbs, const RnsEvalConsts &k, cudaStream_t st) {
    rns_stream_kernel<OP, BCAST><<<grid, kE_Threads, 0, st>>>(
        reinterpret_cast<const uint4 *>(a), reinterpret_cast<const uint4 *>(b), reinterpret_cast<uint4 *>(c),
        tiles, log_g, limbs, k);
}

// op 0..2: add / sub / mul with b; 3: scale by scalars[l] (b unused)
int launch_rns_stream(const nttb200_rns_plan *rp, uint32_t op, const int32_t *a, const int32_t *b, int32_t *c,
                      size_t batch, bool bcast, const uint32_t *scalars, cudaStream_t st) {
    const uint32_t log_g = rp->logn - 12;
    const uint64_t tiles = ((uint64_t) batch * rp->limbs) << log_g;
    if (tiles == 0) return NTTB200_OK;
    const RnsEvalConsts k = eval_consts(rp, scalars);
    const int grid = eval_grid(rp, tiles);
    switch (op * 2 + (bcast ? 1 : 0)) {
        case 0: stream_launch<0, false>(grid, a, b, c, tiles, log_g, rp->limbs, k, st); break;
        case 1: stream_launch<0, true>(grid, a, b, c, tiles, log_g, rp->limbs, k, st); break;
        case 2: stream_launch<1, false>(grid, a, b, c, tiles, log_g, rp->limbs, k, st); break;
        case 3: stream_launch<1, true>(grid, a, b, c, tiles, log_g, rp->limbs, k, st); break;
        case 4: stream_launch<2, false>(grid, a, b, c, tiles, log_g, rp->limbs, k, st); break;
        case 5: stream_launch<2, true>(grid, a, b, c, tiles, log_g, rp->limbs, k, st); break;
        case 6: stream_launch<3, false>(grid, a, a, c, tiles, log_g, rp->limbs, k, st); break;
        default: return NTTB200_ERR_INVALID_ARG;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

int launch_rns_dot(const nttb200_rns_plan *rp, const int32_t *a, const int32_t *w, int32_t *c, uint32_t terms,
                   size_t batch, bool w_shared, bool accumulate, cudaStream_t st) {
    if (batch == 0) return NTTB200_OK;
    const uint32_t log_c = rp->logn - 10;   // chunks of 256 uint4 per row
    const uint64_t group = w_shared ? kE_DotGroupShared : kE_DotGroupOwn;
    const uint64_t items = (((uint64_t) batch + group - 1) / group * rp->limbs) << log_c;
    const RnsEvalConsts k = eval_consts(rp, nullptr);
    const int grid = eval_grid(rp, items);
    const uint4 *a4 = reinterpret_cast<const uint4 *>(a), *w4 = reinterpret_cast<const uint4 *>(w);
    uint4 *c4 = reinterpret_cast<uint4 *>(c);
    if (w_shared) {
        rns_dot_kernel<kE_DotGroupShared, true><<<grid, kE_Threads, 0, st>>>(
            a4, w4, c4, terms, batch, rp->limbs, log_c, items, accumulate ? 1 : 0, k);
    } else {
        rns_dot_kernel<kE_DotGroupOwn, false><<<grid, kE_Threads, 0, st>>>(
            a4, w4, c4, terms, batch, rp->limbs, log_c, items, accumulate ? 1 : 0, k);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

}  // namespace nttb200
