// kernels_polymul.cu -- one kernel per negacyclic product at N = 4096.
//
//   c = a (*) b mod (x^4096 + 1, q):  CT(a), CT(b), pointwise product, GS, N^-1
//
// The three-kernel pipeline (CT(a) -> scratch, CT(b) (*) scratch -> scratch, GS -> c) moves
// 28 N bytes per product through HBM; here both operands enter the SM once and the
// product leaves once: 12 N bytes, the algorithmic minimum (SURVEY 7.5).  A team of 64
// threads (kernels_fused.cu) owns one product at a time:
//
//   TMA a -> buffer | columns: CT stages 11..6 (uniform twiddles, constant bank)
//                   | exchange through the buffer | TMA b -> buffer (lands behind the rows)
//                   | rows: CT stages 5..0 (private twiddles from TENSOR MEMORY)
//                   | a^ made canonical and PARKED IN TENSOR MEMORY (64 columns per warp)
//   same for b      | b^ stays in registers
//   product         | a^ comes back from TMEM 16 words at a time: Montgomery a^*b^*2^-32
//   inverse         | GS stages 0..5 (private twiddles from TMEM), exchange, TMA of the
//                   | NEXT a -> buffer, GS stages 6..11 (constant bank), * N^-1 2^32, store
//
// Tensor Memory holds what would otherwise cost 80 KiB of shared memory per CTA and would
// cap the CTA at 5 teams: the two 32 KiB private-twiddle tables (columns 0..255, lanes =
// threads) and the 16 KiB parking space of every team (columns 256..511); all 512 columns
// are in use.  With one 16 KiB buffer per team left in shared memory the kernel keeps the
// 8 teams x 128 registers shape of the transform kernels.  No tensor-core instruction is
// issued: tcgen05.st / tcgen05.ld only (SASS STTM / LDTM).
//
// Reference counterpart: none (the reference has only the forward network,
// src/test.cpp:34-60); the networks are nttb200_ct_batch / nttb200_gs_batch, bit for bit.
#include <cuda.h>

#include "tile_common.cuh"

namespace nttb200 {

constexpr int kP_Teams = 8;
constexpr int kP_Threads = kP_Teams * kF_Team;
constexpr int kP_SmemBytes = kP_Teams * kF_PolyBytes + 128 + 1024;
constexpr uint32_t kP_ColFwd = 0, kP_ColInv = 128, kP_ColPark = 256;

struct PolymulParams {
    uint32_t *out;
    const uint4 *tw_fwd;   // [32 slots][64 threads] private pairs of the forward rows (CT stages 5..0)
    const uint4 *tw_inv;   // same layout, inverse round 1 (GS stages 0..5)
    uint32_t batch;
    uint32_t q;
    uint32_t zero;
    uint32_t qinv;         // q^-1 mod 2^32
    uint32_t scale;        // N^-1 * 2^32 mod q and its Shoup companion
    uint32_t scale_shoup;
    uint32_t four_q;       // opaque 4q for the 4q-lazy butterflies (q < 2^29)
    uint32_t out_words;    // distance between consecutive products in `out`: 4096, or L * 4096 for one
                           // channel of an RNS batch (the operand views are strided by their tensor maps)
};

// CT stage K on registers pairing rows i and i + 2^K of one column, uniform twiddles
template <int K, bool REDUCE_X>
__device__ __forceinline__ void pm_ct_uniform(uint32_t (&v)[64], const UniformTw &u, uint32_t q,
                                              uint32_t two_q, uint32_t zero) {
    constexpr int kStride = 1 << K;
#pragma unroll
    for (int b = 0; b < (32 >> K); b++) {
        const uint32_t w = u.w[(32 >> K) + b], wp = u.wp[(32 >> K) + b];
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            ct_bfly<REDUCE_X>(v[i0], v[i0 + kStride], w, wp, q, two_q, zero);
        }
    }
}

// GS stage 6+K on registers pairing rows i and i + 2^K; LAST: outputs stay lazy
// (x + y in [0, 4q), product in [0, 2q)) because the N^-1 multiplication that follows
// accepts any 32-bit value
template <int K, bool LAST>
__device__ __forceinline__ void pm_gs_uniform(uint32_t (&v)[64], const UniformTw &u, uint32_t q,
                                              uint32_t two_q, uint32_t zero) {
    constexpr int kStride = 1 << K;
#pragma unroll
    for (int b = 0; b < (32 >> K); b++) {
        const uint32_t w = u.w[(32 >> K) + b], wp = u.wp[(32 >> K) + b];
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            gs_bfly<!LAST>(v[i0], v[i0 + kStride], w, wp, q, two_q, zero);
        }
    }
}

// 4q-lazy form (q < 2^29): inputs below 4q whatever the thread (they come out of round 1)
template <int K>
__device__ __forceinline__ void pm_gs_uniform_l4(uint32_t (&v)[64], const UniformTw &u, uint32_t q,
                                                 uint32_t two_q, uint32_t four_q, uint32_t zero) {
    constexpr int kStride = 1 << K;
#pragma unroll
    for (int b = 0; b < (32 >> K); b++) {
        const uint32_t w = u.w[(32 >> K) + b], wp = u.wp[(32 >> K) + b];
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            gs_bfly_l4(l4_bound(K, e, 4), v[i0], v[i0 + kStride], w, wp, q, two_q, four_q, zero);
        }
    }
}

// LOCKSTEP: the loop body is ~90 KB of straight-line code, twice the instruction-cache reach,
// and 16 warps streaming it at their own pace stall on instruction fetch (ncu: no_instruction
// 0.88 stall cycles per issue).  Widening the team barriers makes warps run in step and share
// every fetch: the barriers span the two teams that share a pair of schedulers (t, t^2)
// instead of one team.  Measured per 16,384 products: team 0.458 ms, team pair 0.417, the four
// teams of a scheduler pair 0.417, the whole CTA 0.423.  Needs batch % 8 == 0 so that all teams
// of a CTA have the same trip count.
// L4 (q < 2^29): 4q-lazy butterflies in both halves.
template <bool LOCKSTEP, bool L4>
__global__ void __launch_bounds__(kP_Threads, 1)
polymul4096_kernel(const __grid_constant__ CUtensorMap a_lo, const __grid_constant__ CUtensorMap a_hi,
                   const __grid_constant__ CUtensorMap b_lo, const __grid_constant__ CUtensorMap b_hi,
                   const __grid_constant__ UniformTw uni_fwd, const __grid_constant__ UniformTw uni_inv,
                   const PolymulParams prm) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t data_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = data_base + kP_Teams * kF_PolyBytes;
    const uint32_t tmem_slot = bar_base + 64;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int team = warp >> 1;   // warp-uniform for the compiler (see kernels_fused.cu)
    const int j = tid & 63;
    const uint32_t q = prm.q, two_q = 2u * prm.q, four_q = prm.four_q, zero = prm.zero;
    constexpr int kBCol = ct_l4_out_n(1, 6), kBRow = ct_l4_out_n(kBCol, 6);   // forward bounds when L4

    if (warp == 0) tmem_alloc_512(tmem_slot);
    if (tid < kP_Teams) mbar_init(bar_base + tid * 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    const uint32_t tmem_base = lds32(tmem_slot);
    // TMEM lane of this thread: 32 * (warp % 4) + lane = 64 * (team % 2) + j
    const uint32_t lane_base = tmem_base + ((uint32_t) (warp & 3) << 21);
    const uint32_t tw_fwd = lane_base + kP_ColFwd, tw_inv = lane_base + kP_ColInv;
    const uint32_t park = lane_base + kP_ColPark + (uint32_t) (warp >> 2) * 64u;

    // both private-twiddle tables, every warp its share of its own lanes
    tmem_fill_table(lane_base + kP_ColFwd, prm.tw_fwd + j, kF_Team, warp);
    tmem_fill_table(lane_base + kP_ColInv, prm.tw_inv + j, kF_Team, warp);
    tmem_wait_st();
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();

    const uint32_t buf = data_base + team * kF_PolyBytes;
    const uint32_t bar = bar_base + team * 8;
    const uint32_t stride = gridDim.x * kP_Teams;
    uint32_t poly = blockIdx.x * kP_Teams + team;
    uint32_t parity = 0;
    if (j == 0 && poly < prm.batch) {
        mbar_expect_tx(bar, kF_PolyBytes);
        tma_load_3d(buf, &a_lo, bar, 0, 0, (int) poly);
        tma_load_3d(buf + kF_PolyBytes / 2, &a_hi, bar, 0, 0, (int) poly);
    }
    // buffer layout as TMA writes it: two halves of [64 rows][32 words], 128 B swizzle
    const uint32_t r1_row = buf + j * 128;
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t r2_col = buf + (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;
    const int pair_id = 9 + ((team & 1) | ((team >> 2) << 1));
    auto sync = [&]() {
        if (LOCKSTEP) {
            asm volatile("bar.sync %0, %1;" ::"r"(pair_id), "n"(128) : "memory");
        } else {
            team_sync(team);
        }
    };

    for (; poly < prm.batch; poly += stride) {
        uint32_t v[64];
#pragma unroll 1
        for (int operand = 0; operand < 2; operand++) {
            mbar_wait(bar, parity);
            parity ^= 1;
            // ---- columns: register i = x[j + 64 i]; CT stages 11..6
#pragma unroll
            for (int i = 0; i < 64; i++) {
                v[i] = lds32(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4)));
            }
            if (L4) {
                ct_round_uniform_l4<1>(v, uni_fwd, q, two_q, four_q, zero);
            } else {
                pm_ct_uniform<5, false>(v, uni_fwd, q, two_q, zero);
                pm_ct_uniform<4, true>(v, uni_fwd, q, two_q, zero);
                pm_ct_uniform<3, true>(v, uni_fwd, q, two_q, zero);
                pm_ct_uniform<2, true>(v, uni_fwd, q, two_q, zero);
                pm_ct_uniform<1, true>(v, uni_fwd, q, two_q, zero);
                pm_ct_uniform<0, true>(v, uni_fwd, q, two_q, zero);
            }
            // ---- exchange: column write, row read (thread j owns x[64j .. 64j+63])
#pragma unroll
            for (int i = 0; i < 64; i++) {
                asm volatile("st.shared.u32 [%0], %1;" ::"r"(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4))),
                             "r"(v[i])
                             : "memory");
            }
            sync();
#pragma unroll
            for (int c = 0; c < 16; c++) {
                uint4 t = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
                v[4 * c + 0] = t.x;
                v[4 * c + 1] = t.y;
                v[4 * c + 2] = t.z;
                v[4 * c + 3] = t.w;
            }
            if (operand == 0) {
                // the buffer is idle during the row stages: fetch b behind them
                fence_proxy_async();
                sync();
                if (j == 0) {
                    mbar_expect_tx(bar, kF_PolyBytes);
                    tma_load_3d(buf, &b_lo, bar, 0, 0, (int) poly);
                    tma_load_3d(buf + kF_PolyBytes / 2, &b_hi, bar, 0, 0, (int) poly);
                }
            }
            // ---- rows: CT stages 5..0, private twiddles from tensor memory
            if (L4) {
                ct_round_tmem_l4<kBCol>(v, tw_fwd, q, two_q, four_q, zero);
            } else {
                ct_round_tmem<true>(v, tw_fwd, q, two_q, zero);
            }
            if (operand == 0) {
                // a^ canonical, parked in this warp's 64 TMEM columns
#pragma unroll
                for (int i = 0; i < 64; i++) {
                    if (L4) {
                        v[i] = canon_l4(kBRow, v[i], q, two_q, four_q);
                    } else {
                        uint32_t r = min(v[i] - two_q, v[i]);
                        v[i] = min(r - q, r);
                    }
                }
#pragma unroll
                for (int g = 0; g < 4; g++) tmem_st16(park + 16 * g, &v[16 * g]);
            }
        }
        // ---- pointwise: b^ (any word) times canonical a^ as a Montgomery product in (0, 2q)
        tmem_wait_st();
#pragma unroll
        for (int g = 0; g < 4; g++) {
            uint32_t t[16];
            tmem_ld16(park + 16 * g, t);
            tmem_wait_ld16(t);
#pragma unroll
            for (int e = 0; e < 16; e++) {
                const uint64_t prod = (uint64_t) v[16 * g + e] * t[e];   // < 2^32 q: no reduction first
                const uint32_t m = (uint32_t) prod * prm.qinv;
                v[16 * g + e] = (uint32_t) (prod >> 32) - __umulhi(m, q) + q;
            }
        }
        // ---- inverse: GS stages 0..5 (private twiddles from tensor memory)
        if (L4) {
            gs_round_tmem_l4<2>(v, tw_inv, q, two_q, four_q, zero);
        } else {
            gs_round_tmem<true>(v, tw_inv, q, two_q, zero);
        }
#pragma unroll
        for (int c = 0; c < 16; c++) {
            sts128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor), v[4 * c],
                   v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
        }
        sync();
#pragma unroll
        for (int i = 0; i < 64; i++) {
            v[i] = lds32(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4)));
        }
        fence_proxy_async();
        sync();
        // ---- the buffer is free: prefetch the next product's a
        const uint32_t next = poly + stride;
        if (j == 0 && next < prm.batch) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &a_lo, bar, 0, 0, (int) next);
            tma_load_3d(buf + kF_PolyBytes / 2, &a_hi, bar, 0, 0, (int) next);
        }
        // ---- GS stages 6..11 (uniform twiddles), N^-1 * 2^32 at the store
        if (L4) {   // the N^-1 multiplication below accepts any word: no canonicalisation
            pm_gs_uniform_l4<0>(v, uni_inv, q, two_q, four_q, zero);
            pm_gs_uniform_l4<1>(v, uni_inv, q, two_q, four_q, zero);
            pm_gs_uniform_l4<2>(v, uni_inv, q, two_q, four_q, zero);
            pm_gs_uniform_l4<3>(v, uni_inv, q, two_q, four_q, zero);
            pm_gs_uniform_l4<4>(v, uni_inv, q, two_q, four_q, zero);
            pm_gs_uniform_l4<5>(v, uni_inv, q, two_q, four_q, zero);
        } else {
            pm_gs_uniform<0, false>(v, uni_inv, q, two_q, zero);
            pm_gs_uniform<1, false>(v, uni_inv, q, two_q, zero);
            pm_gs_uniform<2, false>(v, uni_inv, q, two_q, zero);
            pm_gs_uniform<3, false>(v, uni_inv, q, two_q, zero);
            pm_gs_uniform<4, false>(v, uni_inv, q, two_q, zero);
            pm_gs_uniform<5, true>(v, uni_inv, q, two_q, zero);
        }
        uint32_t *dst = prm.out + (size_t) poly * prm.out_words + j;
#pragma unroll
        for (int i = 0; i < 64; i++) {
            const uint32_t r = shoup_mul_lazy(v[i], prm.scale, prm.scale_shoup, q);
            dst[i * 64] = min(r - q, r);
        }
    }
    tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc_512(tmem_base);
}

// --------------------------------------------------------------------- host side
int tile_maps(CUtensorMap *lo, CUtensorMap *hi, const int32_t *base, size_t tiles);  // kernels_fused.cu
int tile_maps_strided(CUtensorMap *lo, CUtensorMap *hi, const int32_t *base, size_t tiles, uint32_t tile_mul);

int polymul_prepare() {
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    NTTB200_CUDA(cudaFuncSetAttribute(polymul4096_kernel<false, false>, attr, kP_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(polymul4096_kernel<true, false>, attr, kP_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(polymul4096_kernel<false, true>, attr, kP_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(polymul4096_kernel<true, true>, attr, kP_SmemBytes));
    return NTTB200_OK;
}

// c = a (*) b for `batch` products of N = 4096 in one launch.  fwd / inv: plans of the
// psi^bitrev / psi^-bitrev tables with their N = 4096 layouts built (fused_prepare).
int launch_polymul4096(nttb200_plan *fwd, nttb200_plan *inv, const int32_t *d_a, const int32_t *d_b,
                       int32_t *d_c, size_t batch, cudaStream_t st) {
    return launch_polymul4096_strided(fwd, inv, d_a, d_b, d_c, batch, 1, 0, st);
}

// The same for the products p * tile_mul + tile_off, p < batch, of buffers that hold
// batch * tile_mul tiles: channel tile_off of an RNS batch [batch][tile_mul][4096].
int launch_polymul4096_strided(nttb200_plan *fwd, nttb200_plan *inv, const int32_t *d_a,
                               const int32_t *d_b, int32_t *d_c, size_t batch, uint32_t tile_mul,
                               uint32_t tile_off, cudaStream_t st) {
    if (fwd->logn != 12 || inv->logn != 12 || !fwd->d_tw_r1 || !inv->d_tw_r1 || !(fwd->q & 1u)) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    if (batch == 0) return NTTB200_OK;
    if (batch * tile_mul > 0x7fffffffull || ((uintptr_t) d_a & 15u) || ((uintptr_t) d_b & 15u) ||
        ((uintptr_t) d_c & 3u)) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    CUtensorMap a_lo, a_hi, b_lo, b_hi;
    if (tile_maps_strided(&a_lo, &a_hi, d_a + (size_t) tile_off * 4096, batch, tile_mul) != NTTB200_OK ||
        tile_maps_strided(&b_lo, &b_hi, d_b + (size_t) tile_off * 4096, batch, tile_mul) != NTTB200_OK) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    PolymulParams prm;
    prm.out = reinterpret_cast<uint32_t *>(d_c) + (size_t) tile_off * 4096;
    prm.tw_fwd = fwd->d_tw_r1;
    prm.tw_inv = inv->d_tw_r1;
    prm.batch = (uint32_t) batch;
    prm.q = fwd->q;
    prm.zero = 0;
    prm.qinv = inv_mod_2_32(fwd->q);
    const uint64_t sc = ((uint64_t) inv->n_inv << 32) % inv->q;
    prm.scale = (uint32_t) sc;
    prm.scale_shoup = (uint32_t) ((sc << 32) / inv->q);
    prm.four_q = 4u * fwd->q;
    prm.out_words = tile_mul * 4096u;
    const uint64_t ctas = (batch + kP_Teams - 1) / kP_Teams;
    const int grid = (int) (ctas < (uint64_t) fwd->sm_count ? ctas : (uint64_t) fwd->sm_count);
    const bool lockstep = batch % kP_Teams == 0;
    if (lockstep && use_l4(fwd)) {
        polymul4096_kernel<true, true><<<grid, kP_Threads, kP_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi,
                                                                               fwd->uni_gs, inv->uni_gs, prm);
    } else if (lockstep) {
        polymul4096_kernel<true, false><<<grid, kP_Threads, kP_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi,
                                                                                fwd->uni_gs, inv->uni_gs, prm);
    } else if (use_l4(fwd)) {
        polymul4096_kernel<false, true><<<grid, kP_Threads, kP_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi,
                                                                                fwd->uni_gs, inv->uni_gs, prm);
    } else {
        polymul4096_kernel<false, false><<<grid, kP_Threads, kP_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi,
                                                                                 fwd->uni_gs, inv->uni_gs, prm);
    }
    inv->last_path = lockstep ? "polymul4096_one_kernel_tmem_lockstep" : "polymul4096_one_kernel_tmem";
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

}  // namespace nttb200
