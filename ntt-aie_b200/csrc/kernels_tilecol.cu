// kernels_tilecol.cu -- N = 2^16 as ONE persistent kernel whose teams are never in
// lock step: tile items and column items, ordered by counters, intermediate kept in L2.
//
// The reference runs a transform as tile-local stages followed by cross-tile stages, with
// lock-protected fifos between them (src/aie2.py:128-154,178-295; src/aie_core.cc:161-361).
// The first two GPU designs for N > 4096 were (a) two launches -- tile pass, column pass --
// which costs a second HBM round trip (N = 2^16: 0.40 of the HBM roofline), and (b) all
// tiles of a polynomial on the teams of one CTA with a third exchange round, which couples
// up to 16 warps at CTA-wide barriers (N = 2^15: 0.42; ncu: barrier stalls 1.2 cycles per
// issue).  Here every team of 64 threads works alone on
//     T-items  one 4096-coefficient tile: stages 0..11 exactly like the N = 4096 kernel
//              (TMA in, two register rounds, canonical store), private twiddles of the
//              tile's position in TENSOR MEMORY;
//     C-items  the same 1/G slice of all G tiles of one polynomial: 16 x 128-bit loads
//              (L2 hits: the tiles were written a moment ago), the log2 G cross-tile stages
//              in registers with constant-bank twiddles, 16 x 128-bit stores;
// a C-item of polynomial p starts when the G T-items of p have published their stores
// (per-polynomial counter, release/acquire at GPU scope), and each team defers its C-items
// by `lag` polynomials so that the wait is practically never taken.  Teams drift freely --
// no CTA-wide barrier after the prologue -- and every coefficient crosses HBM once in each
// direction; the intermediate lives in the 126 MB L2 for the few microseconds between the
// two items.  All CTAs are co-resident (grid <= #SMs, one CTA per SM), which is what makes
// waiting on another CTA's counter legal.
//
// Forward (Cooley-Tukey) partner: the same two item kinds in the opposite order (C-items
// read the input, T-items finish the tiles: columns, exchange, rows, TMA store).
#include <cuda.h>

#include "tile_common.cuh"

namespace nttb200 {

constexpr int kTC_SmemBytes = kM_Teams * kF_PolyBytes + 128 + 8 * 512 + 1024;
constexpr uint32_t kTC_SpinLimit = 1u << 26;   // polls (>= 64 ns each) before a waiter gives up

struct Tw16c {  // round-2 pairs of one position in shared memory: 32 uint4 slots
    uint32_t addr;
    __device__ __forceinline__ uint4 slot(int s) const { return lds128(addr + s * 16); }
};

struct TileColParams {
    uint32_t *out;
    const uint4 *tw_tile;  // [G][32][65]
    uint32_t *done;        // one counter per polynomial, zero at launch
    uint32_t *error;       // set if a waiter gave up (never in a healthy run)
    uint32_t batch;
    uint32_t lag;          // C-items trail the T-items by this many polynomials
    uint32_t q;
    uint32_t zero;
    uint32_t qinv;
    uint32_t scale;
    uint32_t scale_shoup;
    uint32_t four_q;       // opaque 4q for the 4q-lazy butterflies (q < 2^29)
};

// Counter reads are RELAXED (LDG.STRONG.GPU): ld.acquire costs an L1 invalidation
// (CCTL.IVALL) and a CTA fence per read.  The reads of the published data that follow are
// control-dependent on the value and bypass L1 (ld.global.cg), and the publisher's
// fence.acq_rel.gpu has pushed its stores to L2 before the increment became visible.
__device__ __forceinline__ uint32_t ld_counter(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint4 ldcg128(const uint32_t *p) {
    uint4 v;
    asm volatile("ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p)
                 : "memory");
    return v;
}

// wait until `*ctr >= target` (thread 0 of the team polls; the team barrier that follows
// orders everybody else behind it)
__device__ __forceinline__ void wait_counter(const uint32_t *ctr, uint32_t target, uint32_t *error) {
    uint32_t spins = 0;
    while (ld_counter(ctr) < target) {
        __nanosleep(64);
        if (++spins > kTC_SpinLimit) {
            atomicExch(error, 1u);
            break;
        }
    }
}

// ------------------------------------------------------------------ GS (golden network)
// L4 (q < 2^29): 4q-lazy butterflies; the intermediate between the two item kinds is then
// left LAZY as well (values below 4q), so a T-item stores its registers as they are and the
// C-item's first stage does the one conditional subtraction its sums need.
template <bool DUAL, bool L4>
__global__ void __launch_bounds__(kM_Threads, 1)
tilecol_gs_kernel(const __grid_constant__ CUtensorMap map_lo, const __grid_constant__ CUtensorMap map_hi,
                  const __grid_constant__ CUtensorMap map_b_lo,
                  const __grid_constant__ CUtensorMap map_b_hi, const TileColParams prm,
                  const __grid_constant__ CrossTw cross) {
    constexpr int LOGG = 4;                // N = 2^16
    constexpr int G = 1 << LOGG;
    constexpr int H = G > 8 ? 2 : 1;       // CTA classes: 8 position tables fit one CTA's TMEM
    constexpr int K = G / (2 * H);         // positions per (CTA class, team parity)
    constexpr int U = 16 / G;              // 128-bit column groups per tile and thread (C-items)
    extern __shared__ uint8_t smem_raw[];
    const uint32_t data_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = data_base + kM_Teams * kF_PolyBytes;
    const uint32_t tmem_slot = bar_base + 64, r2base = bar_base + 128;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int team = warp >> 1;
    const int j = tid & 63;
    const uint32_t q = prm.q, two_q = 2u * prm.q, four_q = prm.four_q, zero = prm.zero;
    const uint32_t cta_half = blockIdx.x & (H - 1);
    const uint32_t parity_h = team & 1;

    // ---- prologue: TMEM, mbarriers, this CTA's position tables
    if (warp == 0) tmem_alloc_512(tmem_slot);
    if (tid < kM_Teams) mbar_init(bar_base + tid * 8, 1);
    for (int i = tid; i < (G / H) * 32; i += kM_Threads) {   // round-2 pairs: [local position][slot]
        const uint32_t pos = cta_half * 8 + (i >> 5);
        const uint4 x = __ldg(prm.tw_tile + (size_t) pos * kM_TwTile + (i & 31) * kM_TwRow + 64);
        sts128(r2base + i * 16, x.x, x.y, x.z, x.w);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    const uint32_t tmem_base = lds32(tmem_slot);
    const uint32_t lane_base = tmem_base + ((uint32_t) (warp & 3) << 21);
    {   // lane half h holds the positions of parity h: columns k*128
        const uint32_t h = (uint32_t) (warp & 3) >> 1;
#pragma unroll 1
        for (int k = 0; k < K; k++) {
            const uint32_t pos = cta_half * 8 + 2 * k + h;
            tmem_fill_table(lane_base + (uint32_t) k * 128u, prm.tw_tile + (size_t) pos * kM_TwTile + j,
                            kM_TwRow, warp);
        }
        tmem_wait_st();
    }
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();

    // ---- this team's two work queues
    const uint32_t class_teams = (gridDim.x / H) * (kM_Teams / 2);
    const uint32_t t_total = prm.batch * K;                       // T-items of this class
    uint32_t tq = (blockIdx.x / H) * (kM_Teams / 2) + (team >> 1);
    const uint32_t num_teams = gridDim.x * kM_Teams;
    const uint32_t c_total = prm.batch * G;
    uint32_t cq = blockIdx.x * kM_Teams + team;

    const uint32_t buf = data_base + team * kF_PolyBytes;
    const uint32_t bar = bar_base + team * 8;
    uint32_t parity = 0;
    const uint32_t r1_row = buf + j * 128;
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t r2_col = buf + (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;

    auto tile_index = [&](uint32_t i) -> uint32_t {   // T-item i of this class -> tile in memory
        const uint32_t p = i / K, k = i - p * K;
        return p * G + cta_half * 8 + 2 * k + parity_h;
    };
    if (tq < t_total && j == 0) {
        const int tile = (int) tile_index(tq);
        mbar_expect_tx(bar, kF_PolyBytes);
        tma_load_3d(buf, &map_lo, bar, 0, 0, tile);
        tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, tile);
    }
    // A team publishes a finished tile: its stores, then one release increment (a polynomial is
    // complete at G).  Deferred to the middle
    // of the team's next T-item, when those stores have long left the SM and the fence is cheap.
    uint32_t pending = 0xffffffffu;
    auto publish = [&]() {
        if (pending != 0xffffffffu) {
            // ONE release per team: the team barrier orders the second warp's stores before the
            // first warp's fence, whose cumulativity carries them along (half the MEMBAR.GPU
            // round trips of a fence per warp; `pending` is team-uniform, so is this branch)
            team_sync(team);
            if ((tid & 63) == 0) {
                asm volatile("fence.acq_rel.gpu;" ::: "memory");
                asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(prm.done + pending) : "memory");
            }
            pending = 0xffffffffu;
        }
    };
    // The counter of the team's next C-item is read early (every thread for itself, one
    // broadcast transaction per warp), so the check at the start of the item costs nothing
    // when the polynomial is complete -- which the lag makes the normal case.
    uint32_t ctr_val = 0;
    auto prefetch_counter = [&]() {
        if (cq < c_total) ctr_val = ld_counter(prm.done + cq / G);
    };
    prefetch_counter();

    while (tq < t_total || cq < c_total) {
        // ---- C-items whose polynomial trails this team's next T-item by at least `lag`
        // (lag > one queue step, so the wait targets a polynomial below every unpublished
        // tile of the slowest team: no cycle), or any C-item once the T-items are exhausted
        // (then nothing of this team is pending while it waits)
        const bool t_left = tq < t_total;
        const uint32_t t_poly = t_left ? tq / K : 0;
        while (cq < c_total && (!t_left || cq / G + prm.lag <= t_poly)) {
            const uint32_t p = cq / G, k = cq - p * G;
            if (!t_left) publish();
            if (ctr_val < G) {
                uint32_t spins = 0;
                while ((ctr_val = ld_counter(prm.done + p)) < G) {
                    __nanosleep(64);
                    if (++spins > kTC_SpinLimit) {
                        {
                            *reinterpret_cast<volatile uint32_t *>(prm.error) = 1u;   // mapped host word
                            __threadfence_system();
                        }
                        break;
                    }
                }
            }
            uint32_t *base = prm.out + ((size_t) p << (12 + LOGG)) + k * (4096 / G) + 4 * j;
            uint32_t w[64];
#pragma unroll
            for (int tt = 0; tt < G; tt++) {
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const uint4 x = ldcg128(base + tt * 4096 + u * 256);
                    w[(tt * U + u) * 4 + 0] = x.x;
                    w[(tt * U + u) * 4 + 1] = x.y;
                    w[(tt * U + u) * 4 + 2] = x.z;
                    w[(tt * U + u) * 4 + 3] = x.w;
                }
            }
            cq += num_teams;
            prefetch_counter();
            // stages 12 .. 12+LOGG-1 pair tiles tt and tt + 2^m, twiddle table[(G >> (m+1)) + block]
#pragma unroll
            for (int m = 0; m < LOGG; m++) {
#pragma unroll
                for (int b2 = 0; b2 < (G >> (m + 1)); b2++) {
                    const uint32_t cw = cross.w[(G >> (m + 1)) + b2], cwp = cross.wp[(G >> (m + 1)) + b2];
#pragma unroll
                    for (int e = 0; e < (1 << m); e++) {
                        const int t0 = (b2 << (m + 1)) + e;
#pragma unroll
                        for (int x = 0; x < U * 4; x++) {
                            if (L4) {
                                gs_bfly_l4(l4_bound(m, e, 4), w[t0 * U * 4 + x], w[(t0 + (1 << m)) * U * 4 + x],
                                           cw, cwp, q, two_q, four_q, zero);
                            } else if (m == 0) {
                                gs_bfly<false>(w[t0 * U * 4 + x], w[(t0 + 1) * U * 4 + x], cw, cwp, q, two_q,
                                               zero);
                            } else {
                                gs_bfly<true>(w[t0 * U * 4 + x], w[(t0 + (1 << m)) * U * 4 + x], cw, cwp, q,
                                              two_q, zero);
                            }
                        }
                    }
                }
            }
#pragma unroll
            for (int tt = 0; tt < G; tt++) {
#pragma unroll
                for (int u = 0; u < U; u++) {
                    uint32_t o[4];
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        uint32_t r = w[(tt * U + u) * 4 + e];
                        if (DUAL) {
                            r = shoup_mul_lazy(r, prm.scale, prm.scale_shoup, q);   // any word in
                        } else if (L4 && !((tt >> (LOGG - 1)) & 1)) {
                            r = min(r - two_q, r);   // a sum of the last stage: below 4q
                        }
                        o[e] = min(r - q, r);   // now in [0, 2q)
                    }
                    *reinterpret_cast<uint4 *>(base + tt * 4096 + u * 256) = make_uint4(o[0], o[1], o[2], o[3]);
                }
            }
        }
        if (!t_left) continue;

        // ---- T-item: stages 0..11 of one tile
        const uint32_t p = tq / K, k = tq - p * K;
        const uint32_t tile_cur = tile_index(tq);
        const uint32_t tw1 = lane_base + k * 128u;
        const Tw16c tw2{r2base + (2 * k + parity_h) * 512u};
        uint32_t v[64];
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
            fence_proxy_async();
            team_sync(team);
            if (j == 0) {
                mbar_expect_tx(bar, kF_PolyBytes);
                tma_load_3d(buf, &map_b_lo, bar, 0, 0, (int) tile_cur);
                tma_load_3d(buf + kF_PolyBytes / 2, &map_b_hi, bar, 0, 0, (int) tile_cur);
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
        fence_proxy_async();
        team_sync(team);
        // ---- the buffer is free: prefetch this team's next tile; publish the previous one
        tq += class_teams;
        if (tq < t_total && j == 0) {
            const int tile = (int) tile_index(tq);
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, tile);
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, tile);
        }
        publish();
        if (ctr_val < G) prefetch_counter();   // the next C-item's polynomial was incomplete
        if (L4) {
            gs_round_l4<4>(v, tw2, q, two_q, four_q, zero);
        } else {
            gs_round<true>(v, tw2, q, two_q, zero);
        }
        uint32_t *dst = prm.out + (size_t) tile_cur * 4096 + j;
#pragma unroll
        for (int i = 0; i < 64; i++) {
            dst[i * 64] = L4 ? v[i] : min(v[i] - q, v[i]);
        }
        pending = p;
    }
    publish();
    tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc_512(tmem_base);
}

// ------------------------------------------------------------ CT (forward partner)
// The same two item kinds in the opposite order: C-items first (the 1/16 slice of all 16
// tiles of a polynomial straight from the input: 16 x 128-bit loads, the four cross-tile
// stages 15..12, 16 x 128-bit stores of the LAZY intermediate into `out`), T-items trail by
// `lag` polynomials (the tile comes back from L2 by TMA once all 16 C-items of its polynomial
// have published; columns, exchange, rows, output in two halves through the staging slot as
// in tile_ct_h_kernel).  The TMA load reads what other SMs wrote with ordinary stores: the
// writers' fence.acq_rel.gpu puts the data in L2 before the counter moves, the reader orders
// its async-proxy load behind the counter read with fence.proxy.async.
constexpr int kTC_StageBase = kM_Teams * kF_PolyBytes + 128 + 8 * 512;
constexpr int kTC_SmemBytesCt = ((kTC_StageBase + 1023) / 1024) * 1024 + kM_Teams * (kF_PolyBytes / 2) + 1024;

template <bool L4>
__global__ void __launch_bounds__(kM_Threads, 1)
tilecol_ct_kernel(const uint32_t *__restrict__ in, const __grid_constant__ CUtensorMap mid_lo,
                  const __grid_constant__ CUtensorMap mid_hi, const __grid_constant__ CUtensorMap out_lo,
                  const __grid_constant__ CUtensorMap out_hi, const TileColParams prm,
                  const __grid_constant__ CrossTw cross) {
    constexpr int LOGG = 4, G = 16, H = 2, K = G / (2 * H);
    extern __shared__ uint8_t smem_raw[];
    const uint32_t data_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = data_base + kM_Teams * kF_PolyBytes;
    const uint32_t tmem_slot = bar_base + 64, r2base = bar_base + 128;
    const uint32_t stage_base = (data_base + kTC_StageBase + 1023u) & ~1023u;
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int team = warp >> 1;
    const int j = tid & 63;
    const uint32_t q = prm.q, two_q = 2u * prm.q, four_q = prm.four_q, zero = prm.zero;
    const uint32_t cta_half = blockIdx.x & (H - 1);
    const uint32_t parity_h = team & 1;

    // ---- prologue: TMEM, mbarriers, this CTA's position tables (as in the GS kernel)
    if (warp == 0) tmem_alloc_512(tmem_slot);
    if (tid < kM_Teams) mbar_init(bar_base + tid * 8, 1);
    for (int i = tid; i < (G / H) * 32; i += kM_Threads) {
        const uint32_t pos = cta_half * 8 + (i >> 5);
        const uint4 x = __ldg(prm.tw_tile + (size_t) pos * kM_TwTile + (i & 31) * kM_TwRow + 64);
        sts128(r2base + i * 16, x.x, x.y, x.z, x.w);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    const uint32_t tmem_base = lds32(tmem_slot);
    const uint32_t lane_base = tmem_base + ((uint32_t) (warp & 3) << 21);
    {
        const uint32_t h = (uint32_t) (warp & 3) >> 1;
#pragma unroll 1
        for (int k = 0; k < K; k++) {
            const uint32_t pos = cta_half * 8 + 2 * k + h;
            tmem_fill_table(lane_base + (uint32_t) k * 128u, prm.tw_tile + (size_t) pos * kM_TwTile + j,
                            kM_TwRow, warp);
        }
        tmem_wait_st();
    }
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();

    // ---- this team's two work queues
    const uint32_t class_teams = (gridDim.x / H) * (kM_Teams / 2);
    const uint32_t t_total = prm.batch * K;
    uint32_t tq = (blockIdx.x / H) * (kM_Teams / 2) + (team >> 1);
    const uint32_t num_teams = gridDim.x * kM_Teams;
    const uint32_t c_total = prm.batch * G;
    uint32_t cq = blockIdx.x * kM_Teams + team;

    const uint32_t buf = data_base + team * kF_PolyBytes;
    const uint32_t stg = stage_base + team * (kF_PolyBytes / 2);
    const uint32_t bar = bar_base + team * 8;
    uint32_t parity = 0;
    const uint32_t r1_row = buf + j * 128;
    const uint32_t st_row = stg + j * 128;
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t r2_col = buf + (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;

    auto tile_index = [&](uint32_t i) -> uint32_t {
        const uint32_t p = i / K, k = i - p * K;
        return p * G + cta_half * 8 + 2 * k + parity_h;
    };
    // thread j == 0 of the team: load T-item i's tile if its polynomial is complete
    bool loaded = false;     // meaningful in thread j == 0 only
    auto try_load = [&](uint32_t i, bool must) {
        if (j != 0 || loaded || i >= t_total) return;
        const uint32_t p = i / K;
        uint32_t spins = 0;
        while (ld_counter(prm.done + p) < G) {
            if (!must) return;
            __nanosleep(64);
            if (++spins > kTC_SpinLimit) {
                {
                            *reinterpret_cast<volatile uint32_t *>(prm.error) = 1u;   // mapped host word
                            __threadfence_system();
                        }
                break;
            }
        }
        asm volatile("fence.proxy.async;" ::: "memory");
        const int tile = (int) tile_index(i);
        mbar_expect_tx(bar, kF_PolyBytes);
        tma_load_3d(buf, &mid_lo, bar, 0, 0, tile);
        tma_load_3d(buf + kF_PolyBytes / 2, &mid_hi, bar, 0, 0, tile);
        loaded = true;
    };
    uint32_t pending = 0xffffffffu;
    auto publish = [&]() {
        if (pending != 0xffffffffu) {
            // ONE release per team: the team barrier orders the second warp's stores before the
            // first warp's fence, whose cumulativity carries them along (half the MEMBAR.GPU
            // round trips of a fence per warp; `pending` is team-uniform, so is this branch)
            team_sync(team);
            if ((tid & 63) == 0) {
                asm volatile("fence.acq_rel.gpu;" ::: "memory");
                asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(prm.done + pending) : "memory");
            }
            pending = 0xffffffffu;
        }
    };
    // 4q-lazy bounds: after the cross-tile stages, after the columns, at row stage 4, at the end
    constexpr int kB1 = ct_l4_out_n(1, LOGG), kB2 = ct_l4_out_n(kB1, 6), kB4 = ct_l4_out(kB2),
                  kB3 = ct_l4_out_n(kB4, 5);

    while (cq < c_total || tq < t_total) {
        const bool c_left = cq < c_total;
        const uint32_t c_poly = c_left ? cq / G : 0;
        // ---- T-items whose polynomial trails this team's next C-item by at least `lag`, or any
        // T-item once the C-items are exhausted
        while (tq < t_total && (!c_left || tq / K + prm.lag <= c_poly)) {
            if (!c_left) publish();          // nothing of this team may stay unpublished while it waits
            const uint32_t k = tq - (tq / K) * K;
            const uint32_t tile_cur = tile_index(tq);
            const uint32_t tw1 = lane_base + k * 128u;
            const Tw16c tw2{r2base + (2 * k + parity_h) * 512u};
            try_load(tq, true);
            uint32_t v[64];
            mbar_wait(bar, parity);
            parity ^= 1;
            loaded = false;
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
            // the tile buffer is free: the next T-item's tile if its polynomial is already complete
            fence_proxy_async();
            if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            team_sync(team);
            tq += class_teams;
            try_load(tq, false);
            publish();
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
                    tma_store_3d(h == 0 ? &out_lo : &out_hi, stg, 0, 0, (int) tile_cur);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
        }
        if (!c_left) continue;

        // ---- C-item: the cross-tile stages of one slice of polynomial p
        publish();
        const uint32_t p = cq / G, k = cq - p * G;
        const size_t off = ((size_t) p << (12 + LOGG)) + k * (4096 / G) + 4 * j;
        uint32_t w[64];
#pragma unroll
        for (int tt = 0; tt < G; tt++) {
            uint4 x;
            asm volatile("ld.global.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(x.x), "=r"(x.y), "=r"(x.z), "=r"(x.w)
                         : "l"(in + off + tt * 4096));
            w[tt * 4 + 0] = x.x;
            w[tt * 4 + 1] = x.y;
            w[tt * 4 + 2] = x.z;
            w[tt * 4 + 3] = x.w;
        }
        // the team's next C-item starts its way from HBM to L2 now (16 chunks of 1 KiB)
        if (j < G && cq + num_teams < c_total) {
            const uint32_t cn = cq + num_teams, pn = cn / G, kn = cn - pn * G;
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], 1024;" ::"l"(
                             in + ((size_t) pn << (12 + LOGG)) + kn * (4096 / G) + (size_t) j * 4096)
                         : "memory");
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
                    for (int x = 0; x < 4; x++) {
                        if (L4) {
                            ct_bfly_l4(ct_l4_out_n(1, mm), w[t0 * 4 + x], w[(t0 + (1 << m)) * 4 + x], cw, cwp, q,
                                       two_q, four_q, zero);
                        } else if (mm == 0) {
                            ct_bfly<false>(w[t0 * 4 + x], w[(t0 + (1 << m)) * 4 + x], cw, cwp, q, two_q, zero);
                        } else {
                            ct_bfly<true>(w[t0 * 4 + x], w[(t0 + (1 << m)) * 4 + x], cw, cwp, q, two_q, zero);
                        }
                    }
                }
            }
        }
        // the intermediate stays lazy: below 4q (classic) / kB1 * q (4q-lazy)
#pragma unroll
        for (int tt = 0; tt < G; tt++) {
            *reinterpret_cast<uint4 *>(prm.out + off + tt * 4096) =
                make_uint4(w[tt * 4], w[tt * 4 + 1], w[tt * 4 + 2], w[tt * 4 + 3]);
        }
        pending = p;
        cq += num_teams;
    }
    publish();
    if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    tmem_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc_512(tmem_base);
}

// --------------------------------------------------------------------- host side
int tile_maps(CUtensorMap *lo, CUtensorMap *hi, const int32_t *base, size_t tiles);  // kernels_fused.cu

int tilecol_prepare() {
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    NTTB200_CUDA(cudaFuncSetAttribute(tilecol_ct_kernel<false>, attr, kTC_SmemBytesCt));
    NTTB200_CUDA(cudaFuncSetAttribute(tilecol_ct_kernel<true>, attr, kTC_SmemBytesCt));
    NTTB200_CUDA(cudaFuncSetAttribute(tilecol_gs_kernel<false, false>, attr, kTC_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tilecol_gs_kernel<true, false>, attr, kTC_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tilecol_gs_kernel<false, true>, attr, kTC_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tilecol_gs_kernel<true, true>, attr, kTC_SmemBytes));
    return NTTB200_OK;
}

// Only N = 2^16 takes these kernels -- measured at 2^28 coefficients: 0.439 of the HBM roofline
// against 0.403 for the two passes; for N = 2^13..2^15 the one-CTA-per-polynomial kernels of
// kernels_poly.cu are faster (0.50/0.49/0.42 against 0.42/0.41/0.38).
// Below ~14 tiles per team the prologue, the lag and the drain phase cost more than the saved
// HBM pass (measured at N = 2^16: 512 polynomials 0.199 ms against 0.12 ms for the two passes,
// 1024 polynomials 0.214 against 0.227, 4096 polynomials 0.748 against 0.814).
constexpr uint64_t kTC_MinTilesPerTeam = 12;
// in flight at any time: one tile per team; the items that wait on a counter trail by this
// share of that, in percent
constexpr uint64_t kTC_LagPct = 150;

// The error word of the plan: mapped host memory, so the host can read it without a
// synchronisation.  Checked (and cleared) at the start of the next persistent launch.
static int tilecol_error_word(nttb200_plan *p) {
    std::lock_guard<std::mutex> lock(p->tc_mu);   // plans may be driven from several host threads
    if (!p->tc_err_host) {
        NTTB200_CUDA(cudaHostAlloc((void **) &p->tc_err_host, sizeof(uint32_t), cudaHostAllocMapped));
        *p->tc_err_host = 0;
        NTTB200_CUDA(cudaHostGetDevicePointer((void **) &p->tc_err_dev, p->tc_err_host, 0));
    }
    if (*reinterpret_cast<volatile uint32_t *>(p->tc_err_host)) {
        *p->tc_err_host = 0;
        return fail_msg(NTTB200_ERR_CUDA,
                        "an earlier persistent tile/column launch on this plan gave up waiting for a "
                        "polynomial counter: its output is incomplete");
    }
    return NTTB200_OK;
}

void tilecol_release(nttb200_plan *p) {
    if (p->tc_err_host) cudaFreeHost(p->tc_err_host);
    p->tc_err_host = p->tc_err_dev = nullptr;
}

int launch_tilecol_gs(nttb200_plan *p, const int32_t *d_in, const int32_t *d_b, int32_t *d_out,
                      size_t batch, cudaStream_t st) {
    if (p->logn != 16 || !p->d_tw_tile) return NTTB200_ERR_UNSUPPORTED;
    const uint64_t tiles = (uint64_t) batch << 4;
    if (tiles > 0x7fffffffull || ((uintptr_t) d_out & 15u)) return NTTB200_ERR_UNSUPPORTED;
    if (tiles < (uint64_t) p->sm_count * kM_Teams * kTC_MinTilesPerTeam) return NTTB200_ERR_UNSUPPORTED;
    CUtensorMap a_lo, a_hi, b_lo, b_hi;
    if (tile_maps(&a_lo, &a_hi, d_in, (size_t) tiles) != NTTB200_OK) return NTTB200_ERR_UNSUPPORTED;
    TileColParams tp;
    tp.out = reinterpret_cast<uint32_t *>(d_out);
    tp.tw_tile = p->d_tw_tile;
    tp.batch = (uint32_t) batch;
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
    // one CTA per SM, all co-resident; an even grid: the positions are split over two CTA classes
    uint64_t ctas = (tiles + kM_Teams - 1) / kM_Teams;
    int grid = (int) (ctas < (uint64_t) p->sm_count ? ctas : (uint64_t) p->sm_count);
    grid = grid < 2 ? 2 : (grid & ~1);
    const uint64_t lag_tiles = (uint64_t) grid * kM_Teams * kTC_LagPct / 100;
    tp.lag = (uint32_t) ((lag_tiles >> 4) + 2);   // > one queue step (grid * 8 / G polynomials)
    // counters: one per polynomial + the error word, stream-ordered scratch
    {
        int rce = tilecol_error_word(p);
        if (rce != NTTB200_OK) return rce;
    }
    uint32_t *ctr = nullptr;
    {
        int rca = scratch_alloc_async((void **) &ctr, sizeof(uint32_t) * (batch + 1), st);
        if (rca != NTTB200_OK) return rca;
    }
    NTTB200_CUDA(cudaMemsetAsync(ctr, 0, sizeof(uint32_t) * (batch + 1), st));
    tp.done = ctr;
    tp.error = p->tc_err_dev;
    const bool dual = d_b != nullptr;
    if (dual && use_l4(p)) {
        tilecol_gs_kernel<true, true><<<grid, kM_Threads, kTC_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi, tp,
                                                                               p->cross_tw);
    } else if (dual) {
        tilecol_gs_kernel<true, false><<<grid, kM_Threads, kTC_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi, tp,
                                                                                p->cross_tw);
    } else if (use_l4(p)) {
        tilecol_gs_kernel<false, true><<<grid, kM_Threads, kTC_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi, tp,
                                                                                p->cross_tw);
    } else {
        tilecol_gs_kernel<false, false><<<grid, kM_Threads, kTC_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi, tp,
                                                                                 p->cross_tw);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    cudaError_t e2 = cudaFreeAsync(ctr, st);
    if (e != cudaSuccess) return cuda_fail(e, "tilecol_gs_kernel");
    if (e2 != cudaSuccess) return cuda_fail(e2, "cudaFreeAsync");
    p->last_path = dual ? "tilecol_persistent_dual" : "tilecol_persistent";
    return NTTB200_OK;
}

// N = 2^16 forward transform in one persistent kernel: 4096 polynomials 0.811 ms against 0.901 ms
// for column passes + tile pass (0.405 against 0.365 of the HBM roofline).
int launch_tilecol_ct(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch, cudaStream_t st) {
    if (p->logn != 16 || !p->d_tw_tile) return NTTB200_ERR_UNSUPPORTED;
    const uint64_t tiles = (uint64_t) batch << 4;
    if (tiles > 0x7fffffffull || ((uintptr_t) d_out & 15u) || ((uintptr_t) d_in & 15u)) return NTTB200_ERR_UNSUPPORTED;
    if (tiles < (uint64_t) p->sm_count * kM_Teams * kTC_MinTilesPerTeam) return NTTB200_ERR_UNSUPPORTED;
    CUtensorMap m_lo, m_hi;
    if (tile_maps(&m_lo, &m_hi, d_out, (size_t) tiles) != NTTB200_OK) return NTTB200_ERR_UNSUPPORTED;
    TileColParams tp;
    tp.out = reinterpret_cast<uint32_t *>(d_out);
    tp.tw_tile = p->d_tw_tile;
    tp.batch = (uint32_t) batch;
    tp.q = p->q;
    tp.zero = 0;
    tp.qinv = tp.scale = tp.scale_shoup = 0;
    tp.four_q = 4u * p->q;
    uint64_t ctas = (tiles + kM_Teams - 1) / kM_Teams;
    int grid = (int) (ctas < (uint64_t) p->sm_count ? ctas : (uint64_t) p->sm_count);
    grid = grid < 2 ? 2 : (grid & ~1);
    const uint64_t lag_tiles = (uint64_t) grid * kM_Teams * kTC_LagPct / 100;
    tp.lag = (uint32_t) ((lag_tiles >> 4) + 2);
    {
        int rce = tilecol_error_word(p);
        if (rce != NTTB200_OK) return rce;
    }
    uint32_t *ctr = nullptr;
    {
        int rca = scratch_alloc_async((void **) &ctr, sizeof(uint32_t) * (batch + 1), st);
        if (rca != NTTB200_OK) return rca;
    }
    NTTB200_CUDA(cudaMemsetAsync(ctr, 0, sizeof(uint32_t) * (batch + 1), st));
    tp.done = ctr;
    tp.error = p->tc_err_dev;
    if (use_l4(p)) {
        tilecol_ct_kernel<true><<<grid, kM_Threads, kTC_SmemBytesCt, st>>>(
            reinterpret_cast<const uint32_t *>(d_in), m_lo, m_hi, m_lo, m_hi, tp, p->cross_tw);
    } else {
        tilecol_ct_kernel<false><<<grid, kM_Threads, kTC_SmemBytesCt, st>>>(
            reinterpret_cast<const uint32_t *>(d_in), m_lo, m_hi, m_lo, m_hi, tp, p->cross_tw);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    cudaError_t e2 = cudaFreeAsync(ctr, st);
    if (e != cudaSuccess) return cuda_fail(e, "tilecol_ct_kernel");
    if (e2 != cudaSuccess) return cuda_fail(e2, "cudaFreeAsync");
    p->last_path = "tilecol_persistent_ct";
    return NTTB200_OK;
}

}  // namespace nttb200
