// kernels_multi.cu -- register-radix passes for transforms longer than one 4096 tile.
//
// A length-2^logn golden transform (reference src/test.cpp:34-60) is run as
//   pass 1  "tile pass": stages 0..11 on every contiguous 4096-coefficient tile, the
//           same 64 x 64 TMA-staged team kernel as kernels_fused.cu, except that a
//           tile's twiddles depend on its position c inside the polynomial
//           (table[(N >> (s+1)) + c*(2048 >> s) + ...]) so they are read from a
//           per-position table in global memory laid out [c][slot][65] uint4:
//           coalesced LDG.128 for the thread-private round-1 pairs, one broadcast
//           LDG.128 for the round-2 pairs (L1-resident across a batch);
//   pass 2+ "column pass": the remaining stages s0..s0+K-1 (K <= 6) pair
//           coefficients 2^s apart.  Each thread owns all 2^K partners of VC
//           adjacent columns in registers: 2^K coalesced 32..128-bit loads, K
//           stages, 2^K stores; the twiddle of a butterfly depends only on the row
//           block and the tile's high index bits -- a broadcast load.
// Each pass costs one HBM read + one HBM write (8 bytes per coefficient).  This is
// the GPU analogue of the reference's tile-local stages followed by cross-tile
// stages (src/aie2.py:178-295, src/aie_core.cc:161-187).
//
// Also in this file (all built from the same team/tile machinery):
//   tile_ct_kernel / tile_ct_h_kernel the forward (Cooley-Tukey) tile pass, output through
//                                     a TMA store
//   tile_gs_kernel<DUAL>              pointwise product at load + N^-1 at the store
//   template mode RNS                 tile position -> residue channel with its own modulus
//                                     (column_kernel<.., RNS>: polynomial -> channel)
//   column_kernel<.., SCATTER>        the multi-GPU exchange as NVLink peer stores
#include <vector>

#include "tile_common.cuh"

namespace nttb200 {

// RNS: residue channel l has its own modulus:
// pos[l] = (q_l, q_l^-1 mod 2^32, scale_l, scale_l's Shoup companion).  Passed as a kernel
// parameter so that the (warp-uniform) lookup is a uniform constant-bank load and the
// modulus stays in uniform registers, as in the single-modulus kernels.
// A tile kernel's RNS template mode says which channel tile position c belongs to:
//   kRnsTile: c itself (N = 4096, one tile per channel);
//   kRnsSpan: c >> log_g (N = 4096 * 2^log_g, the G tiles of a channel are adjacent positions).
// The two are separate instantiations so that the N = 4096 kernels carry no shift.
constexpr int kM_MaxChannels = 32;
constexpr int kRnsOff = 0, kRnsTile = 1, kRnsSpan = 2;
struct RnsConsts {
    uint4 pos[kM_MaxChannels];
    uint32_t log_g;   // kRnsSpan: log2 of the tiles per channel
    uint32_t limbs;   // column pass: polynomial P = b*L + l is channel P mod L
};

template <int RNS>
__device__ __forceinline__ uint4 rns_channel(const RnsConsts &rns, uint32_t c) {
    return rns.pos[RNS == kRnsSpan ? c >> rns.log_g : c];
}

// DUAL = false: plain golden stages 0..11 of every tile.
// DUAL = true : the tile's input is the pointwise product of two buffers (second pair
//   of tensor maps), taken as a Montgomery product a*b*2^-32, and every output is
//   multiplied by `scale` (= N^-1 * 2^32 mod q for the inverse transform of a
//   negacyclic product).  The network is linear, so scaling here instead of after the
//   last column pass gives the same residues.
// TWMODE: where the twiddles come from.  0 = global memory (LDG; any workload),
// 2 = shared-memory table per SEGMENT: the CTA's range of position-major tiles is cut
//     at position changes, the table of the segment's position is staged between two
//     __syncthreads (batched large-N and RNS workloads, where a segment is long).
// L4: 4q-lazy butterflies (q < 2^29, single modulus); the tile's output is canonical either way.
// SCALED: plain GS load, every output multiplied by `scale` (Shoup, as DUAL's store) -- with
//   scale = N^-1 mod q the inverse NTT of a psi^-bitrev table in the same passes.
template <bool DUAL, int RNS, int TWMODE = 0, bool L4 = false, bool SCALED = false>
__global__ void __launch_bounds__(kM_Threads, 1)
tile_gs_kernel(const __grid_constant__ CUtensorMap map_lo, const __grid_constant__ CUtensorMap map_hi,
               const __grid_constant__ CUtensorMap map_b_lo,
               const __grid_constant__ CUtensorMap map_b_hi, const TileParams prm,
               const __grid_constant__ RnsConsts rns) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t data_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = data_base + kM_Teams * kF_PolyBytes;
    const int tid = threadIdx.x;
    // broadcast from lane 0 so the compiler knows the team index (and the whole
    // per-team loop) is warp-uniform: q, 2q and the opaque zero then live in uniform
    // registers instead of taking a third vector-register read port in every IADD3
    const int team = __shfl_sync(0xffffffffu, tid >> 6, 0);
    const int j = tid & 63;
    uint32_t q = prm.q, two_q = 2u * prm.q;
    uint32_t qinv = prm.qinv, scale = prm.scale, scale_shoup = prm.scale_shoup;
    const uint32_t zero = prm.zero, four_q = prm.four_q;
    static_assert(!L4 || !RNS, "an RNS channel may be any modulus in [2, 2^30]: classic butterflies only");
    static_assert(!(DUAL && SCALED) && !(L4 && SCALED), "SCALED is the plain-load form of DUAL's store");

    const uint32_t tws = bar_base + 64;
    if (tid < kM_Teams) mbar_init(bar_base + tid * 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    // Work: tiles in position-major order u = c * batch + poly, so that one CTA stays
    // on (at most two) tile positions and their twiddles stay in L1.  CTA b owns the
    // contiguous range [b*T/G, (b+1)*T/G); its teams stride through it.
    // (the host guarantees batch * chunks < 2^31, so tile arithmetic stays 32-bit)
    const uint64_t total = (uint64_t) prm.batch * prm.chunks;
    const uint32_t u_begin = (uint32_t) (total * blockIdx.x / gridDim.x);
    const uint32_t u_end = (uint32_t) (total * (blockIdx.x + 1) / gridDim.x);
    const uint32_t buf = data_base + team * kF_PolyBytes;
    const uint32_t bar = bar_base + team * 8;
    uint32_t parity = 0;

    auto tile_of = [&](uint32_t uu, uint32_t &c) -> uint32_t {
        c = uu / prm.batch;
        uint32_t poly = uu - c * prm.batch;
        return poly * prm.chunks + c;  // tile index in memory
    };

    const uint32_t r1_row = buf + j * 128;
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t r2_col = buf + (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;

    // segments of constant tile position (TWMODE 2); otherwise the whole range at once
    const uint32_t c_first = TWMODE == 2 ? u_begin / prm.batch : 0;
    const uint32_t c_last = (TWMODE == 2 && u_end > u_begin) ? (u_end - 1) / prm.batch : c_first;
    for (uint32_t cs = c_first; cs <= c_last && u_begin < u_end; cs++) {
    uint32_t seg_begin = u_begin, seg_end = u_end;
    if (TWMODE == 2) {
        const uint32_t lo = cs * prm.batch, hi = lo + prm.batch;
        seg_begin = u_begin > lo ? u_begin : lo;
        seg_end = u_end < hi ? u_end : hi;
        __syncthreads();  // every team is done with the previous position's table
        const uint4 *src = prm.tw_tile + (size_t) cs * kM_TwTile;
        for (int i = tid; i < kM_TwTile; i += kM_Threads) {
            uint4 x = __ldg(src + i);
            sts128(tws + i * 16, x.x, x.y, x.z, x.w);
        }
        __syncthreads();
    }
    uint32_t u = seg_begin + team;
    uint32_t c_cur = 0, tile_cur = 0;
    if (u < seg_end) {
        tile_cur = tile_of(u, c_cur);
        if (j == 0) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) tile_cur);
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) tile_cur);
        }
    }

    for (; u < seg_end; u += kM_Teams) {
        uint32_t v[64];
        const uint4 *tw = prm.tw_tile + (size_t) c_cur * kM_TwTile;
        if (RNS) {
            const uint4 pc = rns_channel<RNS>(rns, c_cur);
            q = pc.x;
            two_q = 2u * pc.x;
            qinv = pc.y;
            scale = pc.z;
            scale_shoup = pc.w;
        }
        mbar_wait(bar, parity);
        parity ^= 1;
#pragma unroll
        for (int c = 0; c < 16; c++) {
            uint4 t = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
            v[4 * c + 0] = t.x;
            v[4 * c + 1] = t.y;
            v[4 * c + 2] = t.z;
            v[4 * c + 3] = t.w;
        }
        if (DUAL) {
            // second operand through the same buffer, then v = a*b*2^-32 mod q in (0, 2q)
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
                uint4 t = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
                const uint32_t bb[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    uint64_t prod = (uint64_t) v[4 * c + e] * bb[e];
                    uint32_t m = (uint32_t) prod * qinv;
                    v[4 * c + e] = (uint32_t) (prod >> 32) - __umulhi(m, q) + q;
                }
            }
        }
        if (L4 && TWMODE != 0) {
            gs_round_l4<(DUAL ? 2 : 1)>(v, TwShared{tws + j * 16}, q, two_q, four_q, zero);
        } else if (L4) {
            gs_round_l4<(DUAL ? 2 : 1)>(v, TwGlobal{tw + j}, q, two_q, four_q, zero);
        } else if (TWMODE != 0) {
            gs_round<DUAL>(v, TwShared{tws + j * 16}, q, two_q, zero);
        } else {
            gs_round<DUAL>(v, TwGlobal{tw + j}, q, two_q, zero);
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

        const uint32_t tile_store = tile_cur;
        const uint32_t next = u + kM_Teams;
        if (next < seg_end) {
            tile_cur = tile_of(next, c_cur);
            if (j == 0) {
                mbar_expect_tx(bar, kF_PolyBytes);
                tma_load_3d(buf, &map_lo, bar, 0, 0, (int) tile_cur);
                tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) tile_cur);
            }
        }
        if (L4 && TWMODE != 0) {
            gs_round_l4<4>(v, TwShared{tws + 64 * 16}, q, two_q, four_q, zero);
        } else if (L4) {
            gs_round_l4<4>(v, TwGlobal{tw + 64}, q, two_q, four_q, zero);
        } else if (TWMODE != 0) {
            gs_round<true>(v, TwShared{tws + 64 * 16}, q, two_q, zero);
        } else {
            gs_round<true>(v, TwGlobal{tw + 64}, q, two_q, zero);
        }

        uint32_t *dst = prm.out + (size_t) tile_store * 4096 + j;
#pragma unroll
        for (int i = 0; i < 64; i++) {
            uint32_t r = v[i];
            if (DUAL || SCALED) {
                r = shoup_mul_lazy(r, scale, scale_shoup, q);   // any word in, [0, 2q) out
            } else if (L4 && !(i & 32)) {
                r = min(r - two_q, r);                          // a sum of the last stage: below 4q
            }
            dst[i * 64] = min(r - q, r);
        }
    }
    }  // segments
}

// Forward partner: CT stages 11..0 of every tile (stride 2048 -> 1).  Columns first
// (uniform twiddles), exchange, rows (thread-private twiddles); the rows go back to the
// team's buffer and leave through a TMA store.
// An 8 KiB staging slot per team takes the output in two halves (see tile_ct_h_kernel below),
// so the tile buffer receives the prefetch of the team's next tile as soon as the rows are in
// registers instead of after the store has drained.
template <int RNS, bool L4 = false>
__global__ void __launch_bounds__(kM_Threads, 1)
tile_ct_kernel(const __grid_constant__ CUtensorMap map_lo, const __grid_constant__ CUtensorMap map_hi,
               const __grid_constant__ CUtensorMap out_lo, const __grid_constant__ CUtensorMap out_hi,
               const TileParams prm, const __grid_constant__ RnsConsts rns) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t data_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = data_base + kM_Teams * kF_PolyBytes;
    const int tid = threadIdx.x;
    // broadcast from lane 0 so the compiler knows the team index (and the whole
    // per-team loop) is warp-uniform: q, 2q and the opaque zero then live in uniform
    // registers instead of taking a third vector-register read port in every IADD3
    const int team = __shfl_sync(0xffffffffu, tid >> 6, 0);
    const int j = tid & 63;
    uint32_t q = prm.q, two_q = 2u * prm.q;
    const uint32_t zero = prm.zero;

    static_assert(!L4 || !RNS, "4q-lazy only in the single-modulus form");
    const uint32_t four_q = prm.four_q;
    constexpr int kBCol = ct_l4_out_n(1, 6), kB4 = ct_l4_out(kBCol), kB3 = ct_l4_out(kB4), kB2 = ct_l4_out(kB3),
                  kB1 = ct_l4_out(kB2), kB0 = ct_l4_out(kB1), kBRow = ct_l4_out(kB0);
    const uint32_t stg = ((bar_base + 64 + 1023u) & ~1023u) + team * (kF_PolyBytes / 2);
    const uint32_t st_row = stg + j * 128;
    if (tid < kM_Teams) mbar_init(bar_base + tid * 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    // (the host guarantees batch * chunks < 2^31, so tile arithmetic stays 32-bit)
    const uint64_t total = (uint64_t) prm.batch * prm.chunks;
    const uint32_t u_begin = (uint32_t) (total * blockIdx.x / gridDim.x);
    const uint32_t u_end = (uint32_t) (total * (blockIdx.x + 1) / gridDim.x);
    const uint32_t buf = data_base + team * kF_PolyBytes;
    const uint32_t bar = bar_base + team * 8;
    uint32_t parity = 0;
    uint32_t u = u_begin + team;
    auto tile_of = [&](uint32_t uu, uint32_t &c) -> uint32_t {
        c = uu / prm.batch;
        uint32_t poly = uu - c * prm.batch;
        return poly * prm.chunks + c;
    };
    uint32_t c_cur = 0, tile_cur = 0;
    if (u < u_end) {
        tile_cur = tile_of(u, c_cur);
        if (j == 0) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) tile_cur);
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) tile_cur);
        }
    }
    const uint32_t r1_row = buf + j * 128;
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t r2_col = buf + (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;

    for (; u < u_end; u += kM_Teams) {
        uint32_t v[64];
        const uint4 *tw = prm.tw_tile + (size_t) c_cur * kM_TwTile;
        if (RNS) {
            const uint4 pc = rns_channel<RNS>(rns, c_cur);
            q = pc.x;
            two_q = 2u * pc.x;
        }
        mbar_wait(bar, parity);
        parity ^= 1;
        // ---- columns: register i = a[j + 64 i]; stages 11..6
#pragma unroll
        for (int i = 0; i < 64; i++) {
            v[i] = lds32(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4)));
        }
        if (L4) {
            ct_round_l4<1>(v, TwGlobal{tw + 64}, q, two_q, four_q, zero);
        } else {
            ct_round<false>(v, TwGlobal{tw + 64}, q, two_q, zero);
        }
        // ---- exchange: column write, row read (thread j owns a[64j .. 64j+63])
#pragma unroll
        for (int i = 0; i < 64; i++) {
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4))),
                         "r"(v[i])
                         : "memory");
        }
        team_sync(team);
#pragma unroll
        for (int c = 0; c < 16; c++) {
            uint4 t = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
            v[4 * c + 0] = t.x;
            v[4 * c + 1] = t.y;
            v[4 * c + 2] = t.z;
            v[4 * c + 3] = t.w;
        }
        // ---- the tile buffer is free: prefetch the team's next tile; the staging slot is free
        // once the previous tile's right half has been read by its store
        fence_proxy_async();
        if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        team_sync(team);
        const uint32_t next = u + kM_Teams;
        uint32_t tile_next = 0;
        if (next < u_end) tile_next = tile_of(next, c_cur);
        if (j == 0 && next < u_end) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) tile_next);
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) tile_next);
        }
        // ---- rows: stage 5 pairs the halves, stages 4..0 run per half
        const TwGlobal twr{tw + j};
        if (L4) {
            ct_stage_l4<5, kBCol>(v, twr, q, two_q, four_q, zero);
        } else {
            ct_stage_t<5, true>(v, twr, q, two_q, zero);
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            if (h == 0) {
                ct_half_stage<4, 0, (L4 ? kB4 : -1)>(v, twr, q, two_q, four_q, zero);
                ct_half_stage<3, 0, (L4 ? kB3 : -1)>(v, twr, q, two_q, four_q, zero);
                ct_half_stage<2, 0, (L4 ? kB2 : -1)>(v, twr, q, two_q, four_q, zero);
                ct_half_stage<1, 0, (L4 ? kB1 : -1)>(v, twr, q, two_q, four_q, zero);
                ct_half_stage<0, 0, (L4 ? kB0 : -1)>(v, twr, q, two_q, four_q, zero);
            } else {
                ct_half_stage<4, 1, (L4 ? kB4 : -1)>(v, twr, q, two_q, four_q, zero);
                ct_half_stage<3, 1, (L4 ? kB3 : -1)>(v, twr, q, two_q, four_q, zero);
                ct_half_stage<2, 1, (L4 ? kB2 : -1)>(v, twr, q, two_q, four_q, zero);
                ct_half_stage<1, 1, (L4 ? kB1 : -1)>(v, twr, q, two_q, four_q, zero);
                ct_half_stage<0, 1, (L4 ? kB0 : -1)>(v, twr, q, two_q, four_q, zero);
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
                        o[e] = canon_l4(kBRow, r, q, two_q, four_q);
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
        tile_cur = tile_next;
    }
    // the last tile's halves may still be read out of the staging slot by their stores: no
    // CTA leaves before that; the writes themselves complete before the grid does
    if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}


// N = 4096 forward transform with EIGHT teams: 16 KiB input buffer + 8 KiB output staging per
// team.  The input arrives by TMA and the next tile is prefetched into the input buffer as soon
// as the rows are in registers (like fused_gs4096_kernel); the output leaves by TMA in two
// halves through the staging slot: after stage 5 the two 32-word halves of a row are
// independent, so the left half is finished, staged and handed to the TMA store first, and the
// store reads the slot while the right half's five stages run -- the slot is free again when
// the right half wants it.  No second tile buffer, no exposed wait.  (Measured and dropped: the
// columns loaded straight into registers with coalesced LDG.32 and an L2 prefetch of the next
// tile, one buffer per team: 0.547 ms classic / 0.496 ms 4q-lazy -- the load latency stays
// exposed to the team.)
constexpr int kH_Stage = kF_PolyBytes / 2;
constexpr int kH_TeamBytes = kF_PolyBytes + kH_Stage;   // 24 KiB
constexpr int kH_SmemBytes = kM_Teams * kH_TeamBytes + kM_TwTile * 16 + 128 + 1024;

template <bool L4>
__global__ void __launch_bounds__(kM_Threads, 1)
tile_ct_h_kernel(const __grid_constant__ CUtensorMap map_lo, const __grid_constant__ CUtensorMap map_hi,
                 const __grid_constant__ CUtensorMap out_lo, const __grid_constant__ CUtensorMap out_hi,
                 const __grid_constant__ UniformTw uni, const TileParams prm) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t data_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bar_base = data_base + kM_Teams * kH_TeamBytes;
    const uint32_t tws = bar_base + 128;
    const int tid = threadIdx.x;
    const int team = __shfl_sync(0xffffffffu, tid >> 6, 0);
    const int j = tid & 63;
    const uint32_t q = prm.q, two_q = 2u * prm.q, four_q = prm.four_q, zero = prm.zero;

    const uint32_t total = prm.batch;  // chunks == 1
    const uint32_t stride = gridDim.x * kM_Teams;
    uint32_t tile = team * gridDim.x + blockIdx.x;
    const uint32_t buf = data_base + team * kH_TeamBytes;   // 1024-byte aligned: 24 KiB = 24 * 1024
    const uint32_t stg = buf + kF_PolyBytes;
    const uint32_t bar = bar_base + team * 8;
    uint32_t parity = 0;
    if (j == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (tile < total) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) tile);
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) tile);
        }
    }
    for (int i = tid; i < kM_TwTile; i += kM_Threads) {
        uint4 x = __ldg(prm.tw_tile + i);
        sts128(tws + i * 16, x.x, x.y, x.z, x.w);
    }
    __syncthreads();

    const uint32_t r1_row = buf + j * 128;
    const uint32_t st_row = stg + j * 128;
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t r2_col = buf + (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;
    const TwShared twp{tws + j * 16};
    constexpr int kBCol = ct_l4_out_n(1, 6);                                   // L4 bounds: after the columns,
    constexpr int kB4 = ct_l4_out(kBCol), kB3 = ct_l4_out(kB4), kB2 = ct_l4_out(kB3),
                  kB1 = ct_l4_out(kB2), kB0 = ct_l4_out(kB1), kBRow = ct_l4_out(kB0);  // ... per row stage

    for (; tile < total; tile += stride) {
        uint32_t v[64];
        mbar_wait(bar, parity);
        parity ^= 1;
#pragma unroll
        for (int i = 0; i < 64; i++) {
            v[i] = lds32(r2_col + i * 128 + (r2_chunk ^ ((i & 7) << 4)));
        }
        // stages 11..6: twiddles table[1..63] from the constant bank
        if (L4) {
            ct_round_uniform_l4<1>(v, uni, q, two_q, four_q, zero);
        } else {
            ct_stage_uniform<5, false>(v, uni, q, two_q, zero);
            ct_stage_uniform<4, true>(v, uni, q, two_q, zero);
            ct_stage_uniform<3, true>(v, uni, q, two_q, zero);
            ct_stage_uniform<2, true>(v, uni, q, two_q, zero);
            ct_stage_uniform<1, true>(v, uni, q, two_q, zero);
            ct_stage_uniform<0, true>(v, uni, q, two_q, zero);
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
            uint4 t = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
            v[4 * c + 0] = t.x;
            v[4 * c + 1] = t.y;
            v[4 * c + 2] = t.z;
            v[4 * c + 3] = t.w;
        }
        // ---- the input buffer is free: prefetch the next tile; the staging slot is free once the
        // previous tile's right half has been read by its store
        fence_proxy_async();
        if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        team_sync(team);
        const uint32_t next = tile + stride;
        if (j == 0 && next < total) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) next);
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) next);
        }
        // ---- rows: stage 5 pairs the halves, stages 4..0 run per half
        if (L4) {
            ct_stage_l4<5, kBCol>(v, twp, q, two_q, four_q, zero);
        } else {
            ct_stage_t<5, true>(v, twp, q, two_q, zero);
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
            if (h == 0) {
                ct_half_stage<4, 0, (L4 ? kB4 : -1)>(v, twp, q, two_q, four_q, zero);
                ct_half_stage<3, 0, (L4 ? kB3 : -1)>(v, twp, q, two_q, four_q, zero);
                ct_half_stage<2, 0, (L4 ? kB2 : -1)>(v, twp, q, two_q, four_q, zero);
                ct_half_stage<1, 0, (L4 ? kB1 : -1)>(v, twp, q, two_q, four_q, zero);
                ct_half_stage<0, 0, (L4 ? kB0 : -1)>(v, twp, q, two_q, four_q, zero);
            } else {
                ct_half_stage<4, 1, (L4 ? kB4 : -1)>(v, twp, q, two_q, four_q, zero);
                ct_half_stage<3, 1, (L4 ? kB3 : -1)>(v, twp, q, two_q, four_q, zero);
                ct_half_stage<2, 1, (L4 ? kB2 : -1)>(v, twp, q, two_q, four_q, zero);
                ct_half_stage<1, 1, (L4 ? kB1 : -1)>(v, twp, q, two_q, four_q, zero);
                ct_half_stage<0, 1, (L4 ? kB0 : -1)>(v, twp, q, two_q, four_q, zero);
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
                        o[e] = canon_l4(kBRow, r, q, two_q, four_q);
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
                tma_store_3d(h == 0 ? &out_lo : &out_hi, stg, 0, 0, (int) tile);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
    }
    if (j == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// ------------------------------------------------------------------ column pass
struct ColParams {
    uint32_t logn;
    uint32_t s0;      // first stage of the pass (stride 2^s0)
    uint32_t q;
    uint32_t zero;
    uint64_t threads; // total logical threads = batch * N / (2^K * VC)
};

// Scatter store of the exchange step of the multi-GPU split (one transform, batch 1):
// instead of writing its result in place, the pass writes element idx of this rank's
// length-2^logn vector straight into the peer that owns it after the transpose,
//     rank' = idx >> (logn - log_g),  offset' = rank * 2^(logn-log_g) + (idx & (2^(logn-log_g) - 1)),
// through NVLink peer pointers -- the all-to-all fused into the last local pass
// (the GPU analogue of the reference's neighbour-memory butterflies,
// src/aie2.py:184-187, which also write into another tile's memory).
struct ScatterParams {
    uint32_t *peer[16];
    uint32_t log_g;
    uint32_t rank;
};

template <int VC> struct VecT;
template <> struct VecT<1> { using type = uint32_t; };
template <> struct VecT<2> { using type = uint2; };
template <> struct VecT<4> { using type = uint4; };

// RNS: polynomial P of the pass is b*L + l of a [batch][L][N] layout, so it runs modulo
// q_l = rns.pos[P mod L].x with twiddles tw + l*N ([L][N] tables).  The channel is
// warp-uniform as long as a warp stays inside one polynomial (s0 = 12: 1024 threads each).
template <int K, int VC, bool CT, bool SCATTER, bool RNS = false>
__global__ void __launch_bounds__(256)
column_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out,
              const uint2 *__restrict__ tw, const ColParams p, const ScatterParams sp,
              const __grid_constant__ RnsConsts rns) {
    constexpr int R = 1 << K;
    using V = typename VecT<VC>::type;
    static_assert(!(RNS && SCATTER), "the scatter serves one single-modulus vector");
    uint32_t q = p.q, two_q = 2u * p.q;
    const uint32_t zero = p.zero;
    const uint32_t n = 1u << p.logn;
    const uint32_t cg_bits = p.s0 - (VC == 4 ? 2 : VC == 2 ? 1 : 0);   // column groups per row
    const uint32_t high_bits = p.logn - p.s0 - K;
    for (uint64_t t = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; t < p.threads;
         t += (uint64_t) gridDim.x * blockDim.x) {
        const uint32_t cg = (uint32_t) (t & ((1ull << cg_bits) - 1));
        const uint64_t rest = t >> cg_bits;
        const uint32_t high = (uint32_t) (rest & ((1ull << high_bits) - 1));
        const uint64_t poly = rest >> high_bits;
        const size_t base = poly * n + ((size_t) high << (p.s0 + K)) + (size_t) cg * VC;
        const uint2 *twp = tw;
        if (RNS) {   // the host keeps batch * L below 2^31
            const uint32_t l = (uint32_t) poly % rns.limbs;
            q = rns.pos[l].x;
            two_q = 2u * q;
            twp = tw + ((size_t) l << p.logn);
        }
        uint32_t v[R][VC];
#pragma unroll
        for (int r = 0; r < R; r++) {
            V x = *reinterpret_cast<const V *>(in + base + ((size_t) r << p.s0));
            const uint32_t *xs = reinterpret_cast<const uint32_t *>(&x);
#pragma unroll
            for (int c = 0; c < VC; c++) v[r][c] = xs[c];
        }
#pragma unroll
        for (int mm = 0; mm < K; mm++) {
            const int m = CT ? K - 1 - mm : mm;  // CT: largest stride first
            const uint32_t s = p.s0 + m;
            const uint2 *tws = twp + (n >> (s + 1)) + ((size_t) high << (K - m - 1));
#pragma unroll
            for (int b = 0; b < (R >> (m + 1)); b++) {
                const uint2 w = __ldg(tws + b);
#pragma unroll
                for (int e = 0; e < (1 << m); e++) {
                    const int r0 = (b << (m + 1)) + e;
#pragma unroll
                    for (int c = 0; c < VC; c++) {
                        if (CT) {
                            if (mm == 0) {
                                ct_bfly<false>(v[r0][c], v[r0 + (1 << m)][c], w.x, w.y, q, two_q, zero);
                            } else {
                                ct_bfly<true>(v[r0][c], v[r0 + (1 << m)][c], w.x, w.y, q, two_q, zero);
                            }
                        } else if (mm == 0) {
                            gs_bfly<false>(v[r0][c], v[r0 + (1 << m)][c], w.x, w.y, q, two_q, zero);
                        } else {
                            gs_bfly<true>(v[r0][c], v[r0 + (1 << m)][c], w.x, w.y, q, two_q, zero);
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            V x;
            uint32_t *xs = reinterpret_cast<uint32_t *>(&x);
#pragma unroll
            for (int c = 0; c < VC; c++) {
                uint32_t x1 = CT ? min(v[r][c] - two_q, v[r][c]) : v[r][c];
                xs[c] = min(x1 - q, x1);
            }
            if (SCATTER) {
                const uint32_t idx = (uint32_t) (base + ((size_t) r << p.s0));  // batch is 1
                const uint32_t slice_bits = p.logn - sp.log_g;
                uint32_t *dst = sp.peer[idx >> slice_bits] + ((size_t) sp.rank << slice_bits) +
                                (idx & ((1u << slice_bits) - 1u));
                *reinterpret_cast<V *>(dst) = x;
            } else {
                *reinterpret_cast<V *>(out + base + ((size_t) r << p.s0)) = x;
            }
        }
    }
}

// --------------------------------------------------------------------- host side
int tile_maps(CUtensorMap *lo, CUtensorMap *hi, const int32_t *base, size_t tiles);  // kernels_fused.cu

static const RnsConsts kNoRns{};
constexpr int kM_SmemBytesStaged = kM_SmemBytes + kM_Teams * (kF_PolyBytes / 2) + 1024;

int multi_set_attrs() {
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, false>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<true, false>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, kRnsTile>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_ct_kernel<kRnsOff>, attr, kM_SmemBytesStaged));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_ct_kernel<kRnsTile>, attr, kM_SmemBytesStaged));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_ct_kernel<kRnsOff, true>, attr, kM_SmemBytesStaged));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, false, 2>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<true, false, 2>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, kRnsTile, 2>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, kRnsSpan>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<true, kRnsSpan>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, kRnsSpan, 2>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<true, kRnsSpan, 2>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, kRnsTile, 0, false, true>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, kRnsSpan, 0, false, true>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, kRnsTile, 2, false, true>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, kRnsSpan, 2, false, true>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_ct_kernel<kRnsSpan>, attr, kM_SmemBytesStaged));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, false, 0, true>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<true, false, 0, true>, attr, kM_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<false, false, 2, true>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_gs_kernel<true, false, 2, true>, attr, kM_SmemBytesTw));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_ct_h_kernel<false>, attr, kH_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(tile_ct_h_kernel<true>, attr, kH_SmemBytes));
    return NTTB200_OK;
}

int multi_prepare(nttb200_plan *p) {
    if (p->logn < 12 || p->logn > NTTB200_MAX_LOGN) return NTTB200_ERR_UNSUPPORTED;
    // [N/4096][32][65] uint4, gathered from d_tw by a kernel (tables.cu): at N = 2^26 this
    // layout is 545 MB -- nothing of it is built on or shipped from the host
    const size_t count = (size_t) (p->n >> 12) * kM_TwTile;
    cudaError_t e = cudaMalloc(&p->d_tw_tile, sizeof(uint4) * count);
    if (e != cudaSuccess) {
        p->d_tw_tile = nullptr;
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? NTTB200_ERR_ALLOC : cuda_fail(e, "cudaMalloc(tile table)");
    }
    int rc = build_tile_table(p);
    if (rc != NTTB200_OK) return rc;
    NTTB200_CUDA(cudaDeviceSynchronize());
    if (p->logn >= 13) {
        uint2 head[16];
        NTTB200_CUDA(cudaMemcpy(head, p->d_tw, sizeof(head), cudaMemcpyDeviceToHost));
        for (int i = 0; i < 16; i++) {
            p->cross_tw.w[i] = head[i].x;
            p->cross_tw.wp[i] = head[i].y;
        }
    }
    rc = polyt_prepare();
    if (rc == NTTB200_OK) rc = tilecol_prepare();
    if (rc != NTTB200_OK) return rc;
    return multi_set_attrs();
}

void multi_release(nttb200_plan *p) {
    if (p->d_tw_tile) cudaFree(p->d_tw_tile);
    p->d_tw_tile = nullptr;
}

// rns != nullptr: batch counts the polynomials of all channels (b*L + l), tw is [L][N]
template <int K, int VC, bool CT>
static int launch_column(uint32_t logn, uint32_t q, const uint2 *tw, int sm_count, const int32_t *in,
                         int32_t *out, size_t batch, int s0, cudaStream_t st,
                         const ScatterParams *scatter = nullptr, const RnsConsts *rns = nullptr) {
    ColParams cp;
    cp.logn = logn;
    cp.s0 = (uint32_t) s0;
    cp.q = q;
    cp.zero = 0;
    cp.threads = ((uint64_t) batch << logn) >> (K + (VC == 4 ? 2 : VC == 2 ? 1 : 0));
    if (cp.threads == 0) return NTTB200_OK;
    uint64_t blocks = (cp.threads + 255) / 256;
    uint64_t cap = (uint64_t) sm_count * 64;
    int grid = (int) (blocks < cap ? blocks : cap);
    const uint32_t *src = reinterpret_cast<const uint32_t *>(in);
    uint32_t *dst = reinterpret_cast<uint32_t *>(out);
    ScatterParams none{};
    if (rns) {
        column_kernel<K, VC, CT, false, true><<<grid, 256, 0, st>>>(src, dst, tw, cp, none, *rns);
    } else if (scatter) {
        column_kernel<K, VC, CT, true><<<grid, 256, 0, st>>>(src, dst, tw, cp, *scatter, kNoRns);
    } else {
        column_kernel<K, VC, CT, false><<<grid, 256, 0, st>>>(src, dst, tw, cp, none, kNoRns);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

// stages [s0, s0+k) as one column pass; needs s0 >= 2 (128-bit columns) and aligned buffers
template <bool CT>
static int column_pass_t(nttb200_plan *p, const int32_t *in, int32_t *out, size_t batch, int s0,
                         int k, cudaStream_t st, const ScatterParams *sc = nullptr) {
    if (s0 < 2 || k < 1 || k > 6 || s0 + k > (int) p->logn) return NTTB200_ERR_UNSUPPORTED;
    if (((uintptr_t) in & 15u) || ((uintptr_t) out & 15u)) return NTTB200_ERR_UNSUPPORTED;
    const uint32_t ln = p->logn, q = p->q;
    const uint2 *tw = p->d_tw;
    const int sm = p->sm_count;
    switch (k) {
        case 1: return launch_column<1, 4, CT>(ln, q, tw, sm, in, out, batch, s0, st, sc);
        case 2: return launch_column<2, 4, CT>(ln, q, tw, sm, in, out, batch, s0, st, sc);
        case 3: return launch_column<3, 4, CT>(ln, q, tw, sm, in, out, batch, s0, st, sc);
        case 4: return launch_column<4, 4, CT>(ln, q, tw, sm, in, out, batch, s0, st, sc);
        case 5: return launch_column<5, 2, CT>(ln, q, tw, sm, in, out, batch, s0, st, sc);
        default: return launch_column<6, 1, CT>(ln, q, tw, sm, in, out, batch, s0, st, sc);
    }
}

// RNS, N = 2^13..2^16: the cross-tile stages 12..logn-1 of every channel of `polys`
// = batch * L polynomials as one column pass of K = logn - 12 stages
template <bool CT>
static int rns_column_pass(const nttb200_rns_plan *rp, const RnsConsts &rc, const int32_t *in,
                           int32_t *out, size_t polys, cudaStream_t st) {
    const uint32_t ln = rp->logn;
    const uint2 *tw = rp->d_tw;
    const int sm = rp->sm_count;
    switch (ln - 12) {
        case 1: return launch_column<1, 4, CT>(ln, 0, tw, sm, in, out, polys, 12, st, nullptr, &rc);
        case 2: return launch_column<2, 4, CT>(ln, 0, tw, sm, in, out, polys, 12, st, nullptr, &rc);
        case 3: return launch_column<3, 4, CT>(ln, 0, tw, sm, in, out, polys, 12, st, nullptr, &rc);
        case 4: return launch_column<4, 4, CT>(ln, 0, tw, sm, in, out, polys, 12, st, nullptr, &rc);
        default: return NTTB200_ERR_UNSUPPORTED;
    }
}

int launch_column_pass(nttb200_plan *p, const int32_t *in, int32_t *out, size_t batch, int s0, int k,
                       cudaStream_t st) {
    return column_pass_t<false>(p, in, out, batch, s0, k, st);
}

static TileParams tile_params(nttb200_plan *p, int32_t *d_out, size_t batch) {
    TileParams tp;
    tp.out = reinterpret_cast<uint32_t *>(d_out);
    tp.tw_tile = p->d_tw_tile;
    tp.batch = (uint32_t) batch;
    tp.chunks = p->n >> 12;
    tp.q = p->q;
    tp.zero = 0;
    tp.qinv = 0;
    tp.scale = 0;
    tp.scale_shoup = 0;
    tp.four_q = 4u * p->q;
    return tp;
}

static int tile_grid(nttb200_plan *p, uint64_t tiles) {
    uint64_t ctas = (tiles + kM_Teams - 1) / kM_Teams;
    return (int) (ctas < (uint64_t) p->sm_count ? ctas : (uint64_t) p->sm_count);
}

// from this batch on, the runs of one tile position are long enough to stage the position's
// table in shared memory (TWMODE 2)
constexpr size_t kM_SegTablesMinBatch = 64;

// Tile pass + column passes.  d_b == nullptr: plain transform of d_in.  Otherwise the input
// is d_in (*) d_b and the output is scaled by N^-1 (inverse transform of a negacyclic product).
static int launch_tile_column_gs(nttb200_plan *p, const int32_t *d_in, const int32_t *d_b,
                                 int32_t *d_out, size_t batch, cudaStream_t st) {
    const uint64_t tiles = (uint64_t) batch * (p->n >> 12);
    CUtensorMap map_lo, map_hi, b_lo, b_hi;
    if (tile_maps(&map_lo, &map_hi, d_in, (size_t) tiles) != NTTB200_OK) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    TileParams tp = tile_params(p, d_out, batch);
    int grid = tile_grid(p, tiles);
    const bool l4 = use_l4(p) && tp.chunks > 1;
    const bool seg = batch >= kM_SegTablesMinBatch;
    if (d_b) {
        if (tile_maps(&b_lo, &b_hi, d_b, (size_t) tiles) != NTTB200_OK) return NTTB200_ERR_UNSUPPORTED;
        tp.qinv = inv_mod_2_32(p->q);
        // the Montgomery product carries 2^-32: scale by N^-1 * 2^32 mod q
        uint64_t sc = ((uint64_t) p->n_inv << 32) % p->q;
        tp.scale = (uint32_t) sc;
        tp.scale_shoup = (uint32_t) ((sc << 32) / p->q);
        if (seg && l4) {
            tile_gs_kernel<true, false, 2, true><<<grid, kM_Threads, kM_SmemBytesTw, st>>>(
                map_lo, map_hi, b_lo, b_hi, tp, kNoRns);
        } else if (seg) {
            tile_gs_kernel<true, false, 2><<<grid, kM_Threads, kM_SmemBytesTw, st>>>(
                map_lo, map_hi, b_lo, b_hi, tp, kNoRns);
        } else if (l4) {
            tile_gs_kernel<true, false, 0, true><<<grid, kM_Threads, kM_SmemBytes, st>>>(map_lo, map_hi, b_lo,
                                                                                         b_hi, tp, kNoRns);
        } else {
            tile_gs_kernel<true, false><<<grid, kM_Threads, kM_SmemBytes, st>>>(map_lo, map_hi, b_lo,
                                                                                b_hi, tp, kNoRns);
        }
    } else if (seg && l4) {
        tile_gs_kernel<false, false, 2, true><<<grid, kM_Threads, kM_SmemBytesTw, st>>>(
            map_lo, map_hi, map_lo, map_hi, tp, kNoRns);
    } else if (seg) {
        tile_gs_kernel<false, false, 2><<<grid, kM_Threads, kM_SmemBytesTw, st>>>(
            map_lo, map_hi, map_lo, map_hi, tp, kNoRns);
    } else if (l4) {
        tile_gs_kernel<false, false, 0, true><<<grid, kM_Threads, kM_SmemBytes, st>>>(map_lo, map_hi, map_lo,
                                                                                      map_hi, tp, kNoRns);
    } else {
        tile_gs_kernel<false, false><<<grid, kM_Threads, kM_SmemBytes, st>>>(map_lo, map_hi, map_lo,
                                                                             map_hi, tp, kNoRns);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    // remaining stages 12..logn-1 in column passes of <= 6 stages, evenly split
    int rest = (int) p->logn - 12;
    int passes = (rest + 5) / 6;
    int s0 = 12;
    for (int k = 0; k < passes; k++) {
        int take = (rest + (passes - k) - 1) / (passes - k);
        int rc = launch_column_pass(p, d_out, d_out, batch, s0, take, st);
        if (rc != NTTB200_OK) return rc;
        s0 += take;
        rest -= take;
    }
    return NTTB200_OK;
}

int launch_multi_gs(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    cudaStream_t st) {
    if (!p->d_tw_tile) return NTTB200_ERR_UNSUPPORTED;
    if (batch == 0) return NTTB200_OK;
    const uint64_t tiles = (uint64_t) batch * (p->n >> 12);
    if (tiles > 0x7fffffffull || batch > 0xffffffffull || ((uintptr_t) d_in & 15u) ||
        ((uintptr_t) d_out & 15u)) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    int rc = launch_tilecol_gs(p, d_in, nullptr, d_out, batch, st);
    if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    rc = launch_polyt_gs(p, d_in, nullptr, d_out, batch, st);
    if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    rc = launch_tile_column_gs(p, d_in, nullptr, d_out, batch, st);
    if (rc == NTTB200_OK) p->last_path = "tile_tma + column_passes";
    return rc;
}

// Stages [sb, se) of ONE length-N vector (batch 1) with the result scattered to the
// peers that own it after the transpose (see ScatterParams).  The first stages run
// as the usual passes in place on d_buf; the last column pass stores remotely.
// Needs se == logn, a last pass at least log_g stages deep, and slices of >= 4 words.
int launch_gs_range_scatter(nttb200_plan *p, int32_t *d_buf, int sb, int se, void *const *peers,
                            int world, int rank, cudaStream_t st) {
    int log_g = 0;
    while ((1 << log_g) < world) log_g++;
    if ((1 << log_g) != world || world > 16 || world < 2 || rank < 0 || rank >= world) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if (se != (int) p->logn || sb < 0 || sb >= se || (int) p->logn - log_g < 2) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    if (((uintptr_t) d_buf & 15u) || (p->flags & NTTB200_FORCE_GENERIC)) return NTTB200_ERR_UNSUPPORTED;
    for (int k = 0; k < world; k++) {
        if (!peers[k] || ((uintptr_t) peers[k] & 15u)) return NTTB200_ERR_INVALID_ARG;
    }
    int s0 = sb;
    if (sb == 0) {
        if (!p->d_tw_tile || p->logn < 13) return NTTB200_ERR_UNSUPPORTED;
        const uint64_t tiles = p->n >> 12;
        CUtensorMap map_lo, map_hi;
        if (tile_maps(&map_lo, &map_hi, d_buf, (size_t) tiles) != NTTB200_OK) {
            return NTTB200_ERR_UNSUPPORTED;
        }
        TileParams tp = tile_params(p, d_buf, 1);
        tile_gs_kernel<false, false><<<tile_grid(p, tiles), kM_Threads, kM_SmemBytes, st>>>(
            map_lo, map_hi, map_lo, map_hi, tp, kNoRns);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        NTTB200_CUDA(cudaGetLastError());
        s0 = 12;
    } else if (sb < 2) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    int rest = se - s0;
    int passes = (rest + 5) / 6;
    if (passes < 1) return NTTB200_ERR_UNSUPPORTED;
    ScatterParams sc{};
    for (int k = 0; k < world; k++) sc.peer[k] = reinterpret_cast<uint32_t *>(peers[k]);
    sc.log_g = (uint32_t) log_g;
    sc.rank = (uint32_t) rank;
    for (int k = 0; k < passes; k++) {
        int take = (rest + (passes - k) - 1) / (passes - k);
        const bool last = k == passes - 1;
        // the destination peer is chosen per element from idx >> slice_bits, independent of
        // how many stages the last pass runs
        int rc = column_pass_t<false>(p, d_buf, d_buf, 1, s0, take, st, last ? &sc : nullptr);
        if (rc != NTTB200_OK) return rc;
        s0 += take;
        rest -= take;
    }
    p->last_path = "passes + peer scatter";
    return NTTB200_OK;
}

static bool multi_args_ok(nttb200_plan *p, const void *a, const void *b, size_t batch) {
    const uint64_t tiles = (uint64_t) batch * (p->n >> 12);
    return p->d_tw_tile && tiles <= 0x7fffffffull && batch <= 0xffffffffull &&
           !((uintptr_t) a & 15u) && !((uintptr_t) b & 15u);
}

// inverse transform of the pointwise product of two transformed operands, scaled by
// N^-1: the tail of a negacyclic multiplication (pointwise product and scaling fused
// into the tile pass)
int launch_multi_gs_dual(nttb200_plan *p, const int32_t *d_a, const int32_t *d_b, int32_t *d_out,
                         size_t batch, cudaStream_t st) {
    if (!multi_args_ok(p, d_a, d_out, batch) || ((uintptr_t) d_b & 15u) || !(p->q & 1u)) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    if (batch == 0) return NTTB200_OK;
    int rc = launch_tilecol_gs(p, d_a, d_b, d_out, batch, st);
    if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    rc = launch_polyt_gs(p, d_a, d_b, d_out, batch, st);
    if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    rc = launch_tile_column_gs(p, d_a, d_b, d_out, batch, st);
    if (rc == NTTB200_OK) p->last_path = "tile_tma_dual + column_passes";
    return rc;
}

// forward (CT) transform: column passes from the largest stride down to 2^12, then the
// CT tile pass
int launch_multi_ct(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    cudaStream_t st) {
    // N = 4096 reads table[1..63] from uni_gs, which fused_prepare fills with d_tw_r1
    if (!multi_args_ok(p, d_in, d_out, batch) || (p->logn == 12 && !p->d_tw_r1)) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    if (batch == 0) return NTTB200_OK;
    // (measured and kept out: an 8-team forward kernel that stores each thread's 64
    // consecutive results as 16 x STG.128 -- 32 lines per warp store -- ran 0.588 ms per
    // 65,536 tiles against 0.516 ms for a double-buffered TMA-store kernel)
    int rc = launch_polyt_ct(p, d_in, d_out, batch, st);
    if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    rc = launch_tilecol_ct(p, d_in, d_out, batch, st);
    if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    const int32_t *src = d_in;
    int rest = (int) p->logn - 12;
    int passes = (rest + 5) / 6;
    int top = (int) p->logn;
    for (int k = 0; k < passes; k++) {
        int take = (rest + (passes - k) - 1) / (passes - k);
        rc = column_pass_t<true>(p, src, d_out, batch, top - take, take, st);
        if (rc != NTTB200_OK) return rc;
        src = d_out;
        top -= take;
        rest -= take;
    }
    const uint64_t tiles = (uint64_t) batch * (p->n >> 12);
    CUtensorMap in_lo, in_hi, out_lo, out_hi;
    if (tile_maps(&in_lo, &in_hi, src, (size_t) tiles) != NTTB200_OK ||
        tile_maps(&out_lo, &out_hi, d_out, (size_t) tiles) != NTTB200_OK) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    TileParams tp = tile_params(p, d_out, batch);
    const bool l4 = use_l4(p);
    if (tp.chunks == 1) {
        // per 65,536 tiles: 0.515 ms (two buffers, six teams), 0.504 (tile_ct_h_kernel, classic
        // butterflies), 0.487 (4q-lazy)
        const int grid = (int) (tiles < (uint64_t) p->sm_count ? tiles : (uint64_t) p->sm_count);
        if (l4) {
            tile_ct_h_kernel<true><<<grid, kM_Threads, kH_SmemBytes, st>>>(in_lo, in_hi, out_lo, out_hi,
                                                                           p->uni_gs, tp);
        } else {
            tile_ct_h_kernel<false><<<grid, kM_Threads, kH_SmemBytes, st>>>(in_lo, in_hi, out_lo, out_hi,
                                                                            p->uni_gs, tp);
        }
    } else if (l4) {
        tile_ct_kernel<kRnsOff, true><<<tile_grid(p, tiles), kM_Threads, kM_SmemBytesStaged, st>>>(
            in_lo, in_hi, out_lo, out_hi, tp, kNoRns);
    } else {
        tile_ct_kernel<kRnsOff><<<tile_grid(p, tiles), kM_Threads, kM_SmemBytesStaged, st>>>(
            in_lo, in_hi, out_lo, out_hi, tp, kNoRns);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    p->last_path = p->logn == 12 ? "tile_tma_ct" : "column_passes_ct + tile_tma_ct";
    return NTTB200_OK;
}

// ------------------------------------------------------------------------- RNS
// L residue channels: coefficients [batch][L][N]; channel l is transformed modulo q_l with
// its own table.  The tile kernels already pick their twiddles by tile position; with
// G = N/4096 tiles per channel, position c of the position-major order is tile c mod G of
// channel c >> log2 G, and the concatenated [L][G][32][65] table is indexed by c as for one
// modulus.  N > 4096 adds the cross-tile stages as one RNS column pass.
template <int RNS>
static void rns_tile_launch(int kind, int grid, bool seg, const CUtensorMap &a_lo, const CUtensorMap &a_hi,
                            const CUtensorMap &b_lo, const CUtensorMap &b_hi, const TileParams &tp,
                            const RnsConsts &rc, cudaStream_t st) {
    if (kind == 0) {         // GS
        if (seg) {
            tile_gs_kernel<false, RNS, 2><<<grid, kM_Threads, kM_SmemBytesTw, st>>>(a_lo, a_hi, a_lo,
                                                                                   a_hi, tp, rc);
        } else {
            tile_gs_kernel<false, RNS><<<grid, kM_Threads, kM_SmemBytes, st>>>(a_lo, a_hi, a_lo, a_hi,
                                                                               tp, rc);
        }
    } else if (kind == 1) {  // CT (b_lo / b_hi: output tensor maps)
        tile_ct_kernel<RNS><<<grid, kM_Threads, kM_SmemBytesStaged, st>>>(a_lo, a_hi, b_lo, b_hi, tp, rc);
    } else if (kind == 3) {  // GS, every output times N^-1
        if (seg) {
            tile_gs_kernel<false, RNS, 2, false, true><<<grid, kM_Threads, kM_SmemBytesTw, st>>>(
                a_lo, a_hi, a_lo, a_hi, tp, rc);
        } else {
            tile_gs_kernel<false, RNS, 0, false, true><<<grid, kM_Threads, kM_SmemBytes, st>>>(
                a_lo, a_hi, a_lo, a_hi, tp, rc);
        }
    } else if constexpr (RNS == kRnsSpan) {  // kind 2: GS of the pointwise product, scaled
        if (seg) {
            tile_gs_kernel<true, RNS, 2><<<grid, kM_Threads, kM_SmemBytesTw, st>>>(a_lo, a_hi, b_lo,
                                                                                  b_hi, tp, rc);
        } else {
            tile_gs_kernel<true, RNS><<<grid, kM_Threads, kM_SmemBytes, st>>>(a_lo, a_hi, b_lo, b_hi,
                                                                              tp, rc);
        }
    }
}

// kind 0: GS, 1: CT, 2: GS of the pointwise product d_a (*) d_b, scaled by N^-1 (N > 4096:
// the N = 4096 product runs as one kernel, kernels_polymul.cu), 3: GS scaled by N^-1
int rns_launch(const nttb200_rns_plan *rp, int kind, const int32_t *d_a, const int32_t *d_b,
               int32_t *d_out, size_t batch, cudaStream_t st) {
    const uint32_t limbs = rp->limbs, log_g = rp->logn - 12;
    const uint64_t tiles = ((uint64_t) batch * limbs) << log_g;
    if (tiles == 0) return NTTB200_OK;
    if (limbs > (uint32_t) kM_MaxChannels || (kind == 2 && log_g == 0)) return NTTB200_ERR_UNSUPPORTED;
    if (tiles > 0x7fffffffull || batch > 0xffffffffull || ((uintptr_t) d_a & 15u) ||
        ((uintptr_t) d_out & 15u) || (d_b && ((uintptr_t) d_b & 15u))) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    RnsConsts rc{};
    for (uint32_t l = 0; l < limbs; l++) rc.pos[l] = kind == 3 ? rp->pos_scaled[l] : rp->pos[l];
    rc.log_g = log_g;
    rc.limbs = limbs;
    TileParams tp;
    tp.out = reinterpret_cast<uint32_t *>(d_out);
    tp.tw_tile = rp->d_tw_tile;
    tp.batch = (uint32_t) batch;
    tp.chunks = limbs << log_g;
    tp.q = 0;
    tp.zero = 0;
    tp.qinv = tp.scale = tp.scale_shoup = 0;
    tp.four_q = 0;   // a channel may be any modulus in [2, 2^30]: classic butterflies
    uint64_t ctas = (tiles + kM_Teams - 1) / kM_Teams;
    int grid = (int) (ctas < (uint64_t) rp->sm_count ? ctas : (uint64_t) rp->sm_count);
    const size_t polys = batch * limbs;
    // CT: the cross-tile stages (largest strides) come first, then the tile pass in place
    const int32_t *src = d_a;
    if (kind == 1 && log_g) {
        int rc1 = rns_column_pass<true>(rp, rc, d_a, d_out, polys, st);
        if (rc1 != NTTB200_OK) return rc1;
        src = d_out;
    }
    CUtensorMap a_lo, a_hi, b_lo, b_hi;
    if (tile_maps(&a_lo, &a_hi, src, (size_t) tiles) != NTTB200_OK) return NTTB200_ERR_CUDA;
    if ((kind == 1 || kind == 2) &&
        tile_maps(&b_lo, &b_hi, kind == 1 ? d_out : d_b, (size_t) tiles) != NTTB200_OK) {
        return NTTB200_ERR_CUDA;
    }
    if (kind == 0 || kind == 3) {
        b_lo = a_lo;
        b_hi = a_hi;
    }
    const bool seg = batch >= kM_SegTablesMinBatch;
    if (log_g == 0) {
        rns_tile_launch<kRnsTile>(kind, grid, seg, a_lo, a_hi, b_lo, b_hi, tp, rc, st);
    } else {
        rns_tile_launch<kRnsSpan>(kind, grid, seg, a_lo, a_hi, b_lo, b_hi, tp, rc, st);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    if (kind != 1 && log_g) return rns_column_pass<false>(rp, rc, d_out, d_out, polys, st);
    return NTTB200_OK;
}


}  // namespace nttb200
