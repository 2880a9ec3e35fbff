// kernels_poly.cu -- N = 2^13 .. 2^15 in ONE pass with every private twiddle in tensor memory.
//
// The G = N/4096 tiles of a polynomial are taken by G teams of one CTA at the same time, two
// register rounds per tile (stages 0-11) and a third round through the tile buffers for the
// log2 G cross-tile stages -- one HBM read + one write per coefficient.  The successor of the
// reference's tile-local stages followed by cross-tile ntt_1stage calls
// (src/aie_core.cc:161-361, src/aie2.py:178-295).
//
// Why tensor memory: a first version fetched a tile position's 4032 private (w, w') pairs with
// LDG.128 on the critical path (G x 33 KiB per CTA does not fit L1 next to 132 KiB of shared
// memory: 41 % hit rate, long-scoreboard stalls, issue slots 51 % busy --
// profiles/r1_secondary_kernels_ncu.txt).  Here each position's table sits in TENSOR MEMORY:
// 128 columns per table, lanes = threads; positions of equal parity share a lane half, so
// G = 8 fills exactly the 512 columns.  Round-2 pairs (63 per position) are staged in shared
// memory, the G-1 cross-tile pairs travel as kernel parameters (constant bank).  After the
// prologue the kernel touches global memory for data only.
#include <cuda.h>

#include "tile_common.cuh"

namespace nttb200 {

// forward kernel: + one 8 KiB output staging slot per team (half a tile, see polyt_ct_kernel)
constexpr int kY_StageBase = kM_Teams * kF_PolyBytes + 128 + 8 * 512;
constexpr int kY_SmemBytesCt = ((kY_StageBase + 1023) / 1024) * 1024 + kM_Teams * (kF_PolyBytes / 2) + 1024;

struct Tw16 {               // round-2 pairs of one position in shared memory: 32 uint4 slots
    uint32_t addr;
    __device__ __forceinline__ uint4 slot(int s) const { return lds128(addr + s * 16); }
};

// prologue shared by both kernels: TMEM allocation, mbarriers, round-2 tables to shared
// memory, private tables to tensor memory.  Returns this thread's lane base address.
template <int G>
__device__ __forceinline__ uint32_t poly_prologue(const uint4 *tw_tile, uint32_t bar_base, int tid,
                                                  int warp, int j, uint32_t &tmem_base) {
    const uint32_t tmem_slot = bar_base + 64, r2base = bar_base + 128;
    if (warp == 0) tmem_alloc_512(tmem_slot);
    if (tid < kM_Teams) mbar_init(bar_base + tid * 8, 1);
    for (int i = tid; i < G * 32; i += kM_Threads) {
        const uint4 x = __ldg(tw_tile + (size_t) (i >> 5) * kM_TwTile + (i & 31) * kM_TwRow + 64);
        sts128(r2base + i * 16, x.x, x.y, x.z, x.w);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    tmem_base = lds32(tmem_slot);
    const uint32_t lane_base = tmem_base + ((uint32_t) (warp & 3) << 21);
    {   // lane half h (= quadrant / 2) holds the positions of parity h, 128 columns each
        const int h = (warp & 3) >> 1;
#pragma unroll 1
        for (int pos = h; pos < G; pos += 2) {
            tmem_fill_table(lane_base + (uint32_t) (pos >> 1) * 128u,
                            tw_tile + (size_t) pos * kM_TwTile + j, kM_TwRow, warp);
        }
        tmem_wait_st();
    }
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    return lane_base;
}

template <int LOGG, bool DUAL, bool L4>
__global__ void __launch_bounds__(kM_Threads, 1)
polyt_gs_kernel(const __grid_constant__ CUtensorMap map_lo, const __grid_constant__ CUtensorMap map_hi,
                const __grid_constant__ CUtensorMap map_b_lo,
                const __grid_constant__ CUtensorMap map_b_hi, const TileParams prm,
                const __grid_constant__ CrossTw cross) {
    constexpr int G = 1 << LOGG;           // tiles = teams per polynomial
    constexpr int kGroups = kM_Teams / G;  // polynomials in flight per CTA
    constexpr int kSlice = 64 / G;         // register rows a thread keeps in round 3
    extern __shared__ uint8_t smem_raw[];
    const uint32_t data_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = data_base + kM_Teams * kF_PolyBytes;
    const uint32_t park_base = (data_base + kY_StageBase + 1023u) & ~1023u;   // G = 2: 8 KiB per team
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int team = warp >> 1;
    const int j = tid & 63;
    const int grp = team >> LOGG, t = team & (G - 1);
    const uint32_t q = prm.q, two_q = 2u * prm.q, four_q = prm.four_q, zero = prm.zero;

    uint32_t tmem_base;
    const uint32_t lane_base = poly_prologue<G>(prm.tw_tile, bar_base, tid, warp, j, tmem_base);
    const uint32_t tw1 = lane_base + (uint32_t) (t >> 1) * 128u;   // team parity == position parity
    const Tw16 tw2{bar_base + 128 + (uint32_t) t * 512u};

    const uint32_t buf = data_base + team * kF_PolyBytes;
    const uint32_t gbuf = data_base + (grp << LOGG) * kF_PolyBytes;
    const uint32_t bar = bar_base + team * 8;
    const uint32_t stride = gridDim.x * kGroups;
    uint32_t poly = blockIdx.x * kGroups + grp;
    uint32_t parity = 0;
    if (j == 0 && poly < prm.batch) {
        mbar_expect_tx(bar, kF_PolyBytes);
        tma_load_3d(buf, &map_lo, bar, 0, 0, (int) (poly * G + t));
        tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) (poly * G + t));
    }
    const uint32_t r1_row = buf + j * 128;
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t r2_col = buf + (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;
    auto group_sync = [&]() {
        asm volatile("bar.sync %0, %1;" ::"r"(9 + grp), "n"(G * 64) : "memory");
    };

    for (; poly < prm.batch; poly += stride) {
        uint32_t v[64];
        const int tile = (int) (poly * G + t);
        mbar_wait(bar, parity);
        parity ^= 1;
#pragma unroll
        for (int c = 0; c < 16; c++) {
            uint4 x = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
            v[4 * c + 0] = x.x;
            v[4 * c + 1] = x.y;
            v[4 * c + 2] = x.z;
            v[4 * c + 3] = x.w;
        }
        if (DUAL) {
            // second operand through the same buffer, then v = a*b*2^-32 mod q in (0, 2q)
            team_sync(team);
            if (j == 0) {
                mbar_expect_tx(bar, kF_PolyBytes);
                tma_load_3d(buf, &map_b_lo, bar, 0, 0, tile);
                tma_load_3d(buf + kF_PolyBytes / 2, &map_b_hi, bar, 0, 0, tile);
            }
            mbar_wait(bar, parity);
            parity ^= 1;
#pragma unroll
            for (int c = 0; c < 16; c++) {
                uint4 x = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
                const uint32_t bb[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    uint64_t prod = (uint64_t) v[4 * c + e] * bb[e];
                    uint32_t m = (uint32_t) prod * prm.qinv;
                    v[4 * c + e] = (uint32_t) (prod >> 32) - __umulhi(m, q) + q;
                }
            }
        }
        // ---- round 1: stages 0..5, private pairs from tensor memory
        if (L4) {
            gs_round_tmem_l4<(DUAL ? 2 : 1)>(v, tw1, q, two_q, four_q, zero);
        } else {
            gs_round_tmem<DUAL>(v, tw1, q, two_q, zero);
        }
#pragma unroll
        for (int c = 0; c < 16; c++) {
            sts128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor), v[4 * c],
                   v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
        }
        team_sync(team);
#pragma unroll
        for (int i = 0; i < 64; i++) {
            v[i] = lds32(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4)));
        }
        const uint32_t next = poly + stride;
        if constexpr (LOGG == 1) {
            // G = 2 exchanges its third round through separate parking slots (below), so the tile
            // buffer is free here and takes the next tile while rounds 2 and 3 run -- as in the
            // N = 4096 kernel
            fence_proxy_async();
            team_sync(team);
            if (j == 0 && next < prm.batch) {
                mbar_expect_tx(bar, kF_PolyBytes);
                tma_load_3d(buf, &map_lo, bar, 0, 0, (int) (next * G + t));
                tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) (next * G + t));
            }
        } else {
            team_sync(team);
        }
        // ---- round 2: stages 6..11, the position's 63 pairs from shared memory
        if (L4) {
            gs_round_l4<4>(v, tw2, q, two_q, four_q, zero);
        } else {
            gs_round<true>(v, tw2, q, two_q, zero);
        }

        if constexpr (LOGG == 1) {
            // ---- round 3, two tiles: stage 12 pairs a[j + 64 i] of tile 0 with the same element of
            // tile 1.  Team t keeps rows 32 t .. 32 t + 31 of its own tile and receives the same
            // rows of the other tile: half the exchange of the general scheme, through an 8 KiB
            // slot per team (slot[ii][j]), and the tile buffer stays out of it.
            const uint32_t my_slot = park_base + (uint32_t) team * (kF_PolyBytes / 2) + j * 4;
            const uint32_t his_slot = park_base + (uint32_t) (team ^ 1) * (kF_PolyBytes / 2) + j * 4;
            uint32_t u[32];
            const uint32_t cw = cross.w[1], cwp = cross.wp[1];
            uint32_t *dst = prm.out + ((size_t) poly << 13) + j;
            auto finish = [&](uint32_t x, uint32_t y, int row) {   // x: tile 0 (a sum), y: tile 1 (a product)
                if (DUAL) {
                    x = shoup_mul_lazy(x, prm.scale, prm.scale_shoup, q);   // any word in, [0, 2q) out
                    y = shoup_mul_lazy(y, prm.scale, prm.scale_shoup, q);
                } else if (L4) {
                    x = min(x - two_q, x);   // sums of the last stage are below 4q
                }
                dst[row * 64] = min(x - q, x);
                dst[4096 + row * 64] = min(y - q, y);
            };
            if (t == 0) {
#pragma unroll
                for (int ii = 0; ii < 32; ii++) {
                    asm volatile("st.shared.u32 [%0], %1;" ::"r"(my_slot + ii * 256), "r"(v[32 + ii]) : "memory");
                }
            } else {
#pragma unroll
                for (int ii = 0; ii < 32; ii++) {
                    asm volatile("st.shared.u32 [%0], %1;" ::"r"(my_slot + ii * 256), "r"(v[ii]) : "memory");
                }
            }
            group_sync();
#pragma unroll
            for (int ii = 0; ii < 32; ii++) u[ii] = lds32(his_slot + ii * 256);
            group_sync();   // the other team may refill its slot only after this
            if (t == 0) {
#pragma unroll
                for (int ii = 0; ii < 32; ii++) {
                    if (L4) {
                        gs_bfly_l4(4, v[ii], u[ii], cw, cwp, q, two_q, four_q, zero);
                    } else {
                        gs_bfly<true>(v[ii], u[ii], cw, cwp, q, two_q, zero);
                    }
                    finish(v[ii], u[ii], ii);
                }
            } else {
#pragma unroll
                for (int ii = 0; ii < 32; ii++) {
                    if (L4) {
                        gs_bfly_l4(4, u[ii], v[32 + ii], cw, cwp, q, two_q, four_q, zero);
                    } else {
                        gs_bfly<true>(u[ii], v[32 + ii], cw, cwp, q, two_q, zero);
                    }
                    finish(u[ii], v[32 + ii], 32 + ii);
                }
            }
        } else {
        // ---- round 3: register i is a[t*4096 + j + 64 i].  Park it at [i][j] of this
        // team's buffer, then collect rows t*kSlice .. +kSlice-1 of ALL G tiles.
#pragma unroll
        for (int i = 0; i < 64; i++) {
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(buf + (i * 64 + j) * 4), "r"(v[i]) : "memory");
        }
        group_sync();
        uint32_t w[64];
#pragma unroll
        for (int tt = 0; tt < G; tt++) {
#pragma unroll
            for (int ii = 0; ii < kSlice; ii++) {
                w[tt * kSlice + ii] =
                    lds32(gbuf + tt * kF_PolyBytes + (((t * kSlice + ii) * 64 + j) << 2));
            }
        }
        fence_proxy_async();
        group_sync();
        // ---- every buffer of the group is free: prefetch this team's next tile
        if (j == 0 && next < prm.batch) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) (next * G + t));
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) (next * G + t));
        }
        // ---- stages 12 .. 12+LOGG-1 pair tiles tt and tt + 2^m; twiddle
        //      table[(G >> (m+1)) + (tt >> (m+1))], the same for every thread: constant bank
#pragma unroll
        for (int m = 0; m < LOGG; m++) {
#pragma unroll
            for (int b2 = 0; b2 < (G >> (m + 1)); b2++) {
                const uint32_t cw = cross.w[(G >> (m + 1)) + b2], cwp = cross.wp[(G >> (m + 1)) + b2];
#pragma unroll
                for (int e = 0; e < (1 << m); e++) {
                    const int t0 = (b2 << (m + 1)) + e;
#pragma unroll
                    for (int ii = 0; ii < kSlice; ii++) {
                        if (L4) {
                            gs_bfly_l4(l4_bound(m, e, 4), w[t0 * kSlice + ii], w[(t0 + (1 << m)) * kSlice + ii],
                                       cw, cwp, q, two_q, four_q, zero);
                        } else {
                            gs_bfly<true>(w[t0 * kSlice + ii], w[(t0 + (1 << m)) * kSlice + ii], cw, cwp, q,
                                          two_q, zero);
                        }
                    }
                }
            }
        }
        uint32_t *dst = prm.out + ((size_t) poly << (12 + LOGG)) + j + 64 * (t * kSlice);
#pragma unroll
        for (int tt = 0; tt < G; tt++) {
#pragma unroll
            for (int ii = 0; ii < kSlice; ii++) {
                uint32_t r = w[tt * kSlice + ii];
                if (DUAL) {
                    r = shoup_mul_lazy(r, prm.scale, prm.scale_shoup, q);   // any word in, [0, 2q) out
                } else if (L4 && !((tt >> (LOGG - 1)) & 1)) {
                    r = min(r - two_q, r);   // a sum of the last stage: below 4q
                }
                dst[tt * 4096 + ii * 64] = min(r - q, r);
            }
        }
        }   // LOGG > 1
    }
    tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc_512(tmem_base);
}

// Forward partner: the cross-tile stages come FIRST in the CT order (largest strides),
// then every team finishes its own tile (columns, exchange, rows) and the rows leave
// through a TMA store -- in two halves through an 8 KiB staging slot, like tile_ct_h_kernel
// (kernels_multi.cu): once the rows are in registers the tile buffer takes the prefetch of
// the polynomial after this one; after row stage 5 the two halves of a row are independent,
// so the left half is finished and handed to the TMA store while the right half's five
// stages run.  (The first version staged the output in the tile buffer and could only load
// the next polynomial after the store had drained -- the whole load latency was exposed:
// 0.55 / 0.45 / 0.39 of the HBM roofline at N = 2^13 / 2^14 / 2^15 against 0.61 / 0.56 / 0.51.)
template <int LOGG, bool L4>
__global__ void __launch_bounds__(kM_Threads, 1)
polyt_ct_kernel(const __grid_constant__ CUtensorMap map_lo, const __grid_constant__ CUtensorMap map_hi,
                const __grid_constant__ CUtensorMap out_lo, const __grid_constant__ CUtensorMap out_hi,
                const TileParams prm, const __grid_constant__ CrossTw cross) {
    constexpr int G = 1 << LOGG;
    constexpr int kGroups = kM_Teams / G;
    constexpr int kSlice = 64 / G;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t data_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = data_base + kM_Teams * kF_PolyBytes;
    const uint32_t stage_base = (data_base + kY_StageBase + 1023u) & ~1023u;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int team = warp >> 1;
    const int j = tid & 63;
    const int grp = team >> LOGG, t = team & (G - 1);
    const uint32_t q = prm.q, two_q = 2u * prm.q, four_q = prm.four_q, zero = prm.zero;

    uint32_t tmem_base;
    const uint32_t lane_base = poly_prologue<G>(prm.tw_tile, bar_base, tid, warp, j, tmem_base);
    const uint32_t tw1 = lane_base + (uint32_t) (t >> 1) * 128u;
    const Tw16 tw2{bar_base + 128 + (uint32_t) t * 512u};

    const uint32_t buf = data_base + team * kF_PolyBytes;
    const uint32_t stg = stage_base + team * (kF_PolyBytes / 2);
    const uint32_t gbuf = data_base + (grp << LOGG) * kF_PolyBytes;
    const uint32_t bar = bar_base + team * 8;
    const uint32_t stride = gridDim.x * kGroups;
    uint32_t poly = blockIdx.x * kGroups + grp;
    uint32_t parity = 0;
    if (j == 0 && poly < prm.batch) {
        mbar_expect_tx(bar, kF_PolyBytes);
        tma_load_3d(buf, &map_lo, bar, 0, 0, (int) (poly * G + t));
        tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) (poly * G + t));
    }
    const uint32_t r1_row = buf + j * 128;
    const uint32_t st_row = stg + j * 128;
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t col_off = (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;  // column j of a tile buffer
    const uint32_t r2_col = buf + col_off;
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;
    auto group_sync = [&]() {
        asm volatile("bar.sync %0, %1;" ::"r"(9 + grp), "n"(G * 64) : "memory");
    };
    // 4q-lazy bounds: after the cross-tile stages, after the columns, at row stage 4, at the end
    constexpr int kB1 = ct_l4_out_n(1, LOGG), kB2 = ct_l4_out_n(kB1, 6), kB4 = ct_l4_out(kB2),
                  kB3 = ct_l4_out_n(kB4, 5);

    for (; poly < prm.batch; poly += stride) {
        uint32_t v[64];
        const int tile = (int) (poly * G + t);
        mbar_wait(bar, parity);
        parity ^= 1;
        group_sync();  // all G tiles of the polynomial are in shared memory
        // ---- cross-tile stages logn-1 .. 12 on rows t*kSlice .. +kSlice-1 of every tile
#pragma unroll
        for (int tt = 0; tt < G; tt++) {
#pragma unroll
            for (int ii = 0; ii < kSlice; ii++) {
                const int i = t * kSlice + ii;  // not a compile-time constant: t is per team
                v[tt * kSlice + ii] = lds32(gbuf + tt * kF_PolyBytes + col_off + i * 128 +
                                            (r2_chunk ^ ((i & 7) << 4)));
            }
        }
#pragma unroll
        for (int mm = 0; mm < LOGG; mm++) {
            const int m = LOGG - 1 - mm;
#pragma unroll
            for (int b2 = 0; b2 < (G >> (m + 1)); b2++) {
                const uint32_t cw = cross.w[(G >> (m + 1)) + b2], cwp = cross.wp[(G >> (m + 1)) + b2];
#pragma unroll
                for (int e = 0; e < (1 << m); e++) {
                    const int t0 = (b2 << (m + 1)) + e;
#pragma unroll
                    for (int ii = 0; ii < kSlice; ii++) {
                        if (L4) {
                            ct_bfly_l4(ct_l4_out_n(1, mm), v[t0 * kSlice + ii], v[(t0 + (1 << m)) * kSlice + ii],
                                       cw, cwp, q, two_q, four_q, zero);
                        } else if (mm == 0) {
                            ct_bfly<false>(v[t0 * kSlice + ii], v[(t0 + (1 << m)) * kSlice + ii], cw, cwp,
                                           q, two_q, zero);
                        } else {
                            ct_bfly<true>(v[t0 * kSlice + ii], v[(t0 + (1 << m)) * kSlice + ii], cw, cwp,
                                          q, two_q, zero);
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int tt = 0; tt < G; tt++) {
#pragma unroll
            for (int ii = 0; ii < kSlice; ii++) {
                const int i = t * kSlice + ii;
                asm volatile("st.shared.u32 [%0], %1;" ::"r"(gbuf + tt * kF_PolyBytes + col_off + i * 128 +
                                                             (r2_chunk ^ ((i & 7) << 4))),
                             "r"(v[tt * kSlice + ii])
                             : "memory");
            }
        }
        group_sync();
        // ---- this team's tile: columns (stages 11..6), exchange, rows (stages 5..0)
#pragma unroll
        for (int i = 0; i < 64; i++) {
            v[i] = lds32(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4)));
        }
        if (L4) {
            ct_round_l4<kB1>(v, tw2, q, two_q, four_q, zero);
        } else {
            ct_round<true>(v, tw2, q, two_q, zero);
        }
#pragma unroll
        for (int i = 0; i < 64; i++) {
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4))),
                         "r"(v[i])
                         : "memory");
        }
        team_sync(team);
#pragma unroll
        for (int c = 0; c < 16; c++) {
            uint4 x = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
            v[4 * c + 0] = x.x;
            v[4 * c + 1] = x.y;
            v[4 * c + 2] = x.z;
            v[4 * c + 3] = x.w;
        }
        // ---- the tile buffer is free (nobody else reads it after the group barrier above):
        // prefetch this team's tile of the next polynomial; the staging slot is free once the
        // previous tile's right half has been read by its store
        fence_proxy_async();
        if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        team_sync(team);
        const uint32_t next = poly + stride;
        if (j == 0 && next < prm.batch) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) (next * G + t));
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) (next * G + t));
        }
        // ---- rows: stage 5 pairs the halves, stages 4..0 per half, private pairs from tensor memory
        uint32_t ts345[16], ts2[16];
        tmem_ld16(tw1 + 112, ts345);
        tmem_wait_ld16(ts345);
        tmem_ld16(tw1 + 96, ts2);
        ct_blocks_sel<5, 0, 1, kB2, L4>(v, ts345 + 12, q, two_q, four_q, zero);
        tmem_wait_ld16(ts2);
#pragma unroll
        for (int h = 0; h < 2; h++) {
            if (h == 0) {
                ct_half_tmem<0, kB4, L4>(v, tw1, ts2, ts345, q, two_q, four_q, zero);
            } else {
                ct_half_tmem<1, kB4, L4>(v, tw1, ts2, ts345, q, two_q, four_q, zero);
                // the left half's store has read the slot while these stages ran
                if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                team_sync(team);
            }
#pragma unroll
            for (int c = 0; c < 8; c++) {
                uint32_t o[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    uint32_t r = v[32 * h + 4 * c + e];
                    if (L4) {
                        o[e] = canon_l4(kB3, r, q, two_q, four_q);
                    } else {
                        r = min(r - two_q, r);
                        o[e] = min(r - q, r);
                    }
                }
                sts128(st_row + ((c << 4) ^ r1_xor), o[0], o[1], o[2], o[3]);
            }
            fence_proxy_async();
            team_sync(team);
            if (j == 0) {
                tma_store_3d(h == 0 ? &out_lo : &out_hi, stg, 0, 0, tile);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
    }
    if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc_512(tmem_base);
}

// --------------------------------------------------------------------- host side
int tile_maps(CUtensorMap *lo, CUtensorMap *hi, const int32_t *base, size_t tiles);  // kernels_fused.cu

template <int LOGG>
static int polyt_attrs() {
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    NTTB200_CUDA(cudaFuncSetAttribute(polyt_gs_kernel<LOGG, false, false>, attr, kY_SmemBytesCt));
    NTTB200_CUDA(cudaFuncSetAttribute(polyt_gs_kernel<LOGG, true, false>, attr, kY_SmemBytesCt));
    NTTB200_CUDA(cudaFuncSetAttribute(polyt_gs_kernel<LOGG, false, true>, attr, kY_SmemBytesCt));
    NTTB200_CUDA(cudaFuncSetAttribute(polyt_gs_kernel<LOGG, true, true>, attr, kY_SmemBytesCt));
    NTTB200_CUDA(cudaFuncSetAttribute(polyt_ct_kernel<LOGG, false>, attr, kY_SmemBytesCt));
    NTTB200_CUDA(cudaFuncSetAttribute(polyt_ct_kernel<LOGG, true>, attr, kY_SmemBytesCt));
    return NTTB200_OK;
}

int polyt_prepare() {
    int rc = polyt_attrs<1>();
    if (rc == NTTB200_OK) rc = polyt_attrs<2>();
    if (rc == NTTB200_OK) rc = polyt_attrs<3>();
    return rc;
}

template <int LOGG, bool DUAL>
static void polyt_gs_launch(int grid, cudaStream_t st, const CUtensorMap &a_lo, const CUtensorMap &a_hi,
                            const CUtensorMap &b_lo, const CUtensorMap &b_hi, const TileParams &tp,
                            const CrossTw &cross, bool l4) {
    if (l4) {
        polyt_gs_kernel<LOGG, DUAL, true><<<grid, kM_Threads, kY_SmemBytesCt, st>>>(a_lo, a_hi, b_lo, b_hi,
                                                                                  tp, cross);
    } else {
        polyt_gs_kernel<LOGG, DUAL, false><<<grid, kM_Threads, kY_SmemBytesCt, st>>>(a_lo, a_hi, b_lo, b_hi,
                                                                                   tp, cross);
    }
}
template <int LOGG>
static void polyt_ct_launch(int grid, cudaStream_t st, const CUtensorMap &i_lo, const CUtensorMap &i_hi,
                            const CUtensorMap &o_lo, const CUtensorMap &o_hi, const TileParams &tp,
                            const CrossTw &cross, bool l4) {
    if (l4) {
        polyt_ct_kernel<LOGG, true><<<grid, kM_Threads, kY_SmemBytesCt, st>>>(i_lo, i_hi, o_lo, o_hi, tp, cross);
    } else {
        polyt_ct_kernel<LOGG, false><<<grid, kM_Threads, kY_SmemBytesCt, st>>>(i_lo, i_hi, o_lo, o_hi, tp, cross);
    }
}

// N = 2^13..2^15 golden network in one pass.  d_b != nullptr: input = d_in (*) d_b (Montgomery
// product), output scaled by N^-1 * 2^32 -- the tail of a negacyclic multiplication.
int launch_polyt_gs(nttb200_plan *p, const int32_t *d_in, const int32_t *d_b, int32_t *d_out,
                    size_t batch, cudaStream_t st) {
    const int logg = (int) p->logn - 12;
    if (logg < 1 || logg > 3 || !p->d_tw_tile) return NTTB200_ERR_UNSUPPORTED;
    const uint64_t tiles = (uint64_t) batch << logg;
    if (tiles > 0x7fffffffull) return NTTB200_ERR_UNSUPPORTED;
    CUtensorMap a_lo, a_hi, b_lo, b_hi;
    if (tile_maps(&a_lo, &a_hi, d_in, (size_t) tiles) != NTTB200_OK) return NTTB200_ERR_UNSUPPORTED;
    TileParams tp;
    tp.out = reinterpret_cast<uint32_t *>(d_out);
    tp.tw_tile = p->d_tw_tile;
    tp.batch = (uint32_t) batch;
    tp.chunks = p->n >> 12;
    tp.q = p->q;
    tp.zero = 0;
    tp.qinv = tp.scale = tp.scale_shoup = 0;
    tp.four_q = 4u * p->q;
    if (d_b) {
        if (tile_maps(&b_lo, &b_hi, d_b, (size_t) tiles) != NTTB200_OK) return NTTB200_ERR_UNSUPPORTED;
        tp.qinv = inv_mod_2_32(p->q);
        const uint64_t sc = ((uint64_t) p->n_inv << 32) % p->q;
        tp.scale = (uint32_t) sc;
        tp.scale_shoup = (uint32_t) ((sc << 32) / p->q);
    } else {
        b_lo = a_lo;
        b_hi = a_hi;
    }
    const uint64_t groups = kM_Teams >> logg;
    const uint64_t ctas = (batch + groups - 1) / groups;
    const int grid = (int) (ctas < (uint64_t) p->sm_count ? ctas : (uint64_t) p->sm_count);
    const bool dual = d_b != nullptr, l4 = use_l4(p);
    switch (logg * 2 + (dual ? 1 : 0)) {
        case 2: polyt_gs_launch<1, false>(grid, st, a_lo, a_hi, b_lo, b_hi, tp, p->cross_tw, l4); break;
        case 3: polyt_gs_launch<1, true>(grid, st, a_lo, a_hi, b_lo, b_hi, tp, p->cross_tw, l4); break;
        case 4: polyt_gs_launch<2, false>(grid, st, a_lo, a_hi, b_lo, b_hi, tp, p->cross_tw, l4); break;
        case 5: polyt_gs_launch<2, true>(grid, st, a_lo, a_hi, b_lo, b_hi, tp, p->cross_tw, l4); break;
        case 6: polyt_gs_launch<3, false>(grid, st, a_lo, a_hi, b_lo, b_hi, tp, p->cross_tw, l4); break;
        default: polyt_gs_launch<3, true>(grid, st, a_lo, a_hi, b_lo, b_hi, tp, p->cross_tw, l4); break;
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    p->last_path = dual ? "poly_tmem_3round_dual" : "poly_tmem_3round";
    return NTTB200_OK;
}

int launch_polyt_ct(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    cudaStream_t st) {
    const int logg = (int) p->logn - 12;
    if (logg < 1 || logg > 3 || !p->d_tw_tile) return NTTB200_ERR_UNSUPPORTED;
    const uint64_t tiles = (uint64_t) batch << logg;
    if (tiles > 0x7fffffffull) return NTTB200_ERR_UNSUPPORTED;
    CUtensorMap i_lo, i_hi, o_lo, o_hi;
    if (tile_maps(&i_lo, &i_hi, d_in, (size_t) tiles) != NTTB200_OK ||
        tile_maps(&o_lo, &o_hi, d_out, (size_t) tiles) != NTTB200_OK) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    TileParams tp;
    tp.out = reinterpret_cast<uint32_t *>(d_out);
    tp.tw_tile = p->d_tw_tile;
    tp.batch = (uint32_t) batch;
    tp.chunks = p->n >> 12;
    tp.q = p->q;
    tp.zero = 0;
    tp.qinv = tp.scale = tp.scale_shoup = 0;
    tp.four_q = 4u * p->q;
    const uint64_t groups = kM_Teams >> logg;
    const uint64_t ctas = (batch + groups - 1) / groups;
    const int grid = (int) (ctas < (uint64_t) p->sm_count ? ctas : (uint64_t) p->sm_count);
    const bool l4 = use_l4(p);
    if (logg == 1) {
        polyt_ct_launch<1>(grid, st, i_lo, i_hi, o_lo, o_hi, tp, p->cross_tw, l4);
    } else if (logg == 2) {
        polyt_ct_launch<2>(grid, st, i_lo, i_hi, o_lo, o_hi, tp, p->cross_tw, l4);
    } else {
        polyt_ct_launch<3>(grid, st, i_lo, i_hi, o_lo, o_hi, tp, p->cross_tw, l4);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    p->last_path = "poly_tmem_3round_ct";
    return NTTB200_OK;
}

}  // namespace nttb200
