// tile_common.cuh -- pieces shared by the tile / polynomial kernels (kernels_multi.cu,
// kernels_poly.cu): team geometry, twiddle sources, the per-stage register routines.
#pragma once
#include "fused_common.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kM_Teams = 8;
constexpr int kM_Threads = kF_Team * kM_Teams;
constexpr int kM_TwRow = 65;                    // 64 round-1 threads + 1 round-2 entry
constexpr int kM_TwTile = 32 * kM_TwRow;        // uint4s of twiddles per tile position
constexpr int kM_SmemBytes = kM_Teams * kF_PolyBytes + 64 + 1024;

__device__ __forceinline__ uint4 ldg128(const uint4 *p) { return __ldg(p); }

// Where a team's twiddle slots come from: global memory (LDG, L1-resident across a
// batch) or a shared-memory copy of one position's table (N = 4096, or a run of tiles
// at the same position).
struct TwGlobal {
    const uint4 *p;
    __device__ __forceinline__ uint4 slot(int s) const { return ldg128(p + s * 65); }
};
struct TwShared {
    uint32_t addr;
    __device__ __forceinline__ uint4 slot(int s) const { return lds128(addr + s * (65 * 16)); }
};

// One stage on the thread's 64 registers (pairs i, i + 2^S); the two (w, w') pairs of
// blocks b, b+1 come as one uint4 from tw[slot * 65] (slot = 0,16,24,28,30,31 + b/2).
template <int S, bool REDUCE, class TW>
__device__ __forceinline__ void gs_stage_t(uint32_t (&v)[64], const TW tw, uint32_t q,
                                           uint32_t two_q, uint32_t zero) {
    constexpr int kBlocks = 32 >> S;
    constexpr int kSlot0 = 32 - (kBlocks >= 2 ? kBlocks : 1);
    constexpr int kStride = 1 << S;
#pragma unroll
    for (int b = 0; b < kBlocks; b += 2) {
        uint4 t = tw.slot(kSlot0 + b / 2);
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            gs_bfly<REDUCE>(v[i0], v[i0 + kStride], t.x, t.y, q, two_q, zero);
        }
        if (kBlocks >= 2) {
#pragma unroll
            for (int e = 0; e < kStride; e++) {
                int i0 = (b + 1) * 2 * kStride + e;
                gs_bfly<REDUCE>(v[i0], v[i0 + kStride], t.z, t.w, q, two_q, zero);
            }
        }
    }
}


// CT stage on the thread's 64 registers (pairs i, i + 2^S), same twiddle slots as GS
template <int S, bool REDUCE_X, class TW>
__device__ __forceinline__ void ct_stage_t(uint32_t (&v)[64], const TW tw, uint32_t q,
                                           uint32_t two_q, uint32_t zero) {
    constexpr int kBlocks = 32 >> S;
    constexpr int kSlot0 = 32 - (kBlocks >= 2 ? kBlocks : 1);
    constexpr int kStride = 1 << S;
#pragma unroll
    for (int b = 0; b < kBlocks; b += 2) {
        uint4 t = tw.slot(kSlot0 + b / 2);
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            ct_bfly<REDUCE_X>(v[i0], v[i0 + kStride], t.x, t.y, q, two_q, zero);
        }
        if (kBlocks >= 2) {
#pragma unroll
            for (int e = 0; e < kStride; e++) {
                int i0 = (b + 1) * 2 * kStride + e;
                ct_bfly<REDUCE_X>(v[i0], v[i0 + kStride], t.z, t.w, q, two_q, zero);
            }
        }
    }
}

// 4q-lazy forms (q < 2^29; fused_common.cuh gs_bfly_l4 / ct_bfly_l4)
template <int S, int BIN0, class TW>
__device__ __forceinline__ void gs_stage_l4(uint32_t (&v)[64], const TW tw, uint32_t q, uint32_t two_q,
                                            uint32_t four_q, uint32_t zero) {
    constexpr int kBlocks = 32 >> S;
    constexpr int kSlot0 = 32 - (kBlocks >= 2 ? kBlocks : 1);
    constexpr int kStride = 1 << S;
#pragma unroll
    for (int b = 0; b < kBlocks; b += 2) {
        uint4 t = tw.slot(kSlot0 + b / 2);
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            gs_bfly_l4(l4_bound(S, e, BIN0), v[i0], v[i0 + kStride], t.x, t.y, q, two_q, four_q, zero);
        }
        if (kBlocks >= 2) {
#pragma unroll
            for (int e = 0; e < kStride; e++) {
                int i0 = (b + 1) * 2 * kStride + e;
                gs_bfly_l4(l4_bound(S, e, BIN0), v[i0], v[i0 + kStride], t.z, t.w, q, two_q, four_q, zero);
            }
        }
    }
}
template <int S, int BIN, class TW>
__device__ __forceinline__ void ct_stage_l4(uint32_t (&v)[64], const TW tw, uint32_t q, uint32_t two_q,
                                            uint32_t four_q, uint32_t zero) {
    constexpr int kBlocks = 32 >> S;
    constexpr int kSlot0 = 32 - (kBlocks >= 2 ? kBlocks : 1);
    constexpr int kStride = 1 << S;
#pragma unroll
    for (int b = 0; b < kBlocks; b += 2) {
        uint4 t = tw.slot(kSlot0 + b / 2);
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            ct_bfly_l4(BIN, v[i0], v[i0 + kStride], t.x, t.y, q, two_q, four_q, zero);
        }
        if (kBlocks >= 2) {
#pragma unroll
            for (int e = 0; e < kStride; e++) {
                int i0 = (b + 1) * 2 * kStride + e;
                ct_bfly_l4(BIN, v[i0], v[i0 + kStride], t.z, t.w, q, two_q, four_q, zero);
            }
        }
    }
}
template <int BIN0, class TW>
__device__ __forceinline__ void gs_round_l4(uint32_t (&v)[64], const TW tw, uint32_t q, uint32_t two_q,
                                            uint32_t four_q, uint32_t zero) {
    gs_stage_l4<0, BIN0>(v, tw, q, two_q, four_q, zero);
    gs_stage_l4<1, BIN0>(v, tw, q, two_q, four_q, zero);
    gs_stage_l4<2, BIN0>(v, tw, q, two_q, four_q, zero);
    gs_stage_l4<3, BIN0>(v, tw, q, two_q, four_q, zero);
    gs_stage_l4<4, BIN0>(v, tw, q, two_q, four_q, zero);
    gs_stage_l4<5, BIN0>(v, tw, q, two_q, four_q, zero);
}
// inputs below BIN0 * q, outputs below ct_l4_out_n(BIN0, 6) * q (LAST: below 4q)
template <int BIN0, bool LAST = false, class TW>
__device__ __forceinline__ void ct_round_l4(uint32_t (&v)[64], const TW tw, uint32_t q, uint32_t two_q,
                                            uint32_t four_q, uint32_t zero) {
    constexpr int B5 = BIN0, B4 = ct_l4_out(B5), B3 = ct_l4_out(B4), B2 = ct_l4_out(B3),
                  B1 = ct_l4_out(B2), B0 = ct_l4_out(B1);
    ct_stage_l4<5, B5>(v, tw, q, two_q, four_q, zero);
    ct_stage_l4<4, B4>(v, tw, q, two_q, four_q, zero);
    ct_stage_l4<3, B3>(v, tw, q, two_q, four_q, zero);
    ct_stage_l4<2, B2>(v, tw, q, two_q, four_q, zero);
    ct_stage_l4<1, B1>(v, tw, q, two_q, four_q, zero);
    ct_stage_l4<0, (LAST ? -B0 : B0)>(v, tw, q, two_q, four_q, zero);
}
template <int K, int BIN>
__device__ __forceinline__ void ct_stage_uniform_l4(uint32_t (&v)[64], const UniformTw &u, uint32_t q,
                                                    uint32_t two_q, uint32_t four_q, uint32_t zero) {
    constexpr int kStride = 1 << K;
#pragma unroll
    for (int b = 0; b < (32 >> K); b++) {
        const uint32_t w = u.w[(32 >> K) + b], wp = u.wp[(32 >> K) + b];
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            ct_bfly_l4(BIN, v[i0], v[i0 + kStride], w, wp, q, two_q, four_q, zero);
        }
    }
}
template <int BIN0>
__device__ __forceinline__ void ct_round_uniform_l4(uint32_t (&v)[64], const UniformTw &u, uint32_t q,
                                                    uint32_t two_q, uint32_t four_q, uint32_t zero) {
    constexpr int B5 = BIN0, B4 = ct_l4_out(B5), B3 = ct_l4_out(B4), B2 = ct_l4_out(B3),
                  B1 = ct_l4_out(B2), B0 = ct_l4_out(B1);
    ct_stage_uniform_l4<5, B5>(v, u, q, two_q, four_q, zero);
    ct_stage_uniform_l4<4, B4>(v, u, q, two_q, four_q, zero);
    ct_stage_uniform_l4<3, B3>(v, u, q, two_q, four_q, zero);
    ct_stage_uniform_l4<2, B2>(v, u, q, two_q, four_q, zero);
    ct_stage_uniform_l4<1, B1>(v, u, q, two_q, four_q, zero);
    ct_stage_uniform_l4<0, B0>(v, u, q, two_q, four_q, zero);
}

// CT stage S < 5 restricted to the registers [32 H, 32 H + 32): after stage 5 the two halves
// of a 64-coefficient row are independent, which lets a kernel finish and ship one half while
// the other is still being computed (tile_ct_h_kernel).  BIN < 0: classic butterfly with
// REDUCE_X = true; BIN > 0: 4q-lazy with input bound BIN.
template <int S, int H, int BIN, class TW>
__device__ __forceinline__ void ct_half_stage(uint32_t (&v)[64], const TW tw, uint32_t q, uint32_t two_q,
                                              uint32_t four_q, uint32_t zero) {
    static_assert(S < 5, "stage 5 pairs the halves");
    constexpr int kBlocks = 32 >> S;                 // blocks per row; half H owns kBlocks/2 of them
    constexpr int kSlot0 = 32 - kBlocks;
    constexpr int kStride = 1 << S;
#pragma unroll
    for (int b = H * (kBlocks / 2); b < (H + 1) * (kBlocks / 2); b++) {
        const uint4 t = tw.slot(kSlot0 + b / 2);     // (w, w') of blocks b & ~1 and b | 1
        const uint32_t w = (b & 1) ? t.z : t.x, wp = (b & 1) ? t.w : t.y;
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            const int i0 = b * 2 * kStride + e;
            if (BIN > 0) {
                ct_bfly_l4(BIN, v[i0], v[i0 + kStride], w, wp, q, two_q, four_q, zero);
            } else {
                ct_bfly<true>(v[i0], v[i0 + kStride], w, wp, q, two_q, zero);
            }
        }
    }
}

template <bool REDUCE0, class TW>
__device__ __forceinline__ void gs_round(uint32_t (&v)[64], const TW tw, uint32_t q, uint32_t two_q,
                                         uint32_t zero) {
    gs_stage_t<0, REDUCE0>(v, tw, q, two_q, zero);
    gs_stage_t<1, true>(v, tw, q, two_q, zero);
    gs_stage_t<2, true>(v, tw, q, two_q, zero);
    gs_stage_t<3, true>(v, tw, q, two_q, zero);
    gs_stage_t<4, true>(v, tw, q, two_q, zero);
    gs_stage_t<5, true>(v, tw, q, two_q, zero);
}
template <bool REDUCE_FIRST, class TW>
__device__ __forceinline__ void ct_round(uint32_t (&v)[64], const TW tw, uint32_t q, uint32_t two_q,
                                         uint32_t zero) {
    ct_stage_t<5, REDUCE_FIRST>(v, tw, q, two_q, zero);
    ct_stage_t<4, true>(v, tw, q, two_q, zero);
    ct_stage_t<3, true>(v, tw, q, two_q, zero);
    ct_stage_t<2, true>(v, tw, q, two_q, zero);
    ct_stage_t<1, true>(v, tw, q, two_q, zero);
    ct_stage_t<0, true>(v, tw, q, two_q, zero);
}

// CT stage K on registers that pair rows i and i + 2^K of one column, twiddles that do not
// depend on the thread (table[(32 >> K) + block]) straight from the constant bank
template <int K, bool REDUCE_X>
__device__ __forceinline__ void ct_stage_uniform(uint32_t (&v)[64], const UniformTw &u, uint32_t q,
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

constexpr int kM_SmemBytesTw = kM_SmemBytes + kM_TwTile * 16;  // + one shared twiddle table

struct TileParams {
    uint32_t *out;
    const uint4 *tw_tile;  // [chunks][32][65]
    uint32_t batch;
    uint32_t chunks;       // tiles per polynomial
    uint32_t q;
    uint32_t zero;
    uint32_t qinv;         // q^-1 mod 2^32 (DUAL: Montgomery product of the two inputs)
    uint32_t scale;        // DUAL: every output is multiplied by this constant (Shoup pair)
    uint32_t scale_shoup;
    uint32_t four_q;       // 4q as an opaque value for the 4q-lazy kernels (q < 2^29), else unused
};


}  // namespace nttb200
