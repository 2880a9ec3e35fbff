// kernels_fused.cu -- the throughput path: whole-transform register-radix kernels.
//
// N = 4096 = 64 x 64.  A polynomial is handled by a TEAM of 64 threads (2 warps);
// every coefficient crosses HBM exactly once in each direction:
//
//   TMA (cp.async.bulk.tensor, 128B swizzle) : HBM -> shared, one 16 KiB polynomial
//   round 1  thread j owns a[64j .. 64j+63] (index bits 0-5): golden stages 0-5
//            entirely in registers; its 63 private twiddles stream from a
//            shared-memory copy of the table laid out for conflict-free LDS.128
//   exchange registers -> the same shared buffer -> registers (64 x 64 transpose,
//            swizzled so both directions are bank-conflict free)
//   round 2  thread j owns a[j + 64 i] (index bits 6-11): golden stages 6-11 in
//            registers; those stages' twiddles depend only on the register index,
//            so they are kernel parameters = constant-bank operands of IMAD
//   store    coalesced 128 B rows straight from registers
//
// The next polynomial's TMA load is issued as soon as round 2 has pulled the
// current one out of shared memory, so HBM latency hides behind round-2 math.
// Eight teams per CTA, one persistent CTA per SM.
//
// Arithmetic: lazy Harvey butterflies in [0, 2q) -- IADD3, IADD3, VIADDMNMX,
// IMAD.HI, IMAD, IMAD per butterfly -- canonicalised in the last stage, so the
// result equals the golden's `%` chain (reference src/test.cpp:46-50) bit for bit.
// This is the successor of ntt_stage0_to_Nminus5 + ntt_1stage + swap_buff +
// write_back (reference src/aie_core.cc:133-361) and of their schedule in
// src/aie2.py:161-317; the twiddle index rule is the golden's table[h+i]
// (src/test.cpp:45).
#include <cuda.h>

#include <vector>

#include "fused_common.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kF_N = 4096;
#ifndef NTTB200_TEAMS
#define NTTB200_TEAMS 8
#endif
constexpr int kF_Teams = NTTB200_TEAMS;   // polynomials in flight per CTA
constexpr int kF_Threads = kF_Team * kF_Teams;
constexpr int kF_TwSlots = 32;            // uint4 slots of round-1 twiddles per thread
constexpr int kF_TwBytes = kF_TwSlots * kF_Team * 16;   // 32 KiB
constexpr int kF_SmemBytes = kF_TwBytes + kF_Teams * kF_PolyBytes + 64 + 1024;

__host__ __device__ constexpr int kBitrev6(int x) {
    return ((x & 1) << 5) | ((x & 2) << 3) | ((x & 4) << 1) | ((x & 8) >> 1) | ((x & 16) >> 3) |
           ((x & 32) >> 5);
}

// last stage: canonical outputs in [0, q)
__device__ __forceinline__ void gs_bfly_final(uint32_t &x, uint32_t &y, uint32_t w, uint32_t wp,
                                              uint32_t q, uint32_t two_q, uint32_t zero) {
    uint32_t s = x + y + zero;
    uint32_t d = x - y + two_q;
    s = min(s - two_q, s);
    uint32_t h = __umulhi(d, wp);
    uint32_t r = d * w - h * q;
    x = min(s - q, s);
    y = min(r - q, r);
}

// last stage, 4q-lazy inputs bounded by bin * q
__device__ __forceinline__ void gs_bfly_final_l4(const int bin, uint32_t &x, uint32_t &y, uint32_t w,
                                                 uint32_t wp, uint32_t q, uint32_t two_q,
                                                 uint32_t four_q, uint32_t zero) {
    uint32_t s = x + y + zero;
    uint32_t d = x - y + (bin == 4 ? four_q : two_q);
    if (bin == 4) s = min(s - four_q, s);
    s = min(s - two_q, s);
    uint32_t h = __umulhi(d, wp);
    uint32_t r = d * w - h * q;
    x = min(s - q, s);
    y = min(r - q, r);
}

// round 1, stage S (stride 2^S inside the thread's 64 contiguous coefficients).
// Twiddle of local block b: table[(2048 >> S) + j*(32 >> S) + b]; the (w, w')
// pairs of one thread sit in shared memory as uint4 slots [slot][thread].
template <int S, bool L4>
__device__ __forceinline__ void round1_stage(uint32_t (&v)[64], uint32_t tw_addr, uint32_t q,
                                             uint32_t two_q, uint32_t four_q, uint32_t zero) {
    constexpr int kBlocks = 32 >> S;                       // distinct twiddles
    constexpr int kSlot0 = 32 - (kBlocks >= 2 ? kBlocks : 1);  // 0,16,24,28,30,31
    constexpr int kStride = 1 << S;
#pragma unroll
    for (int b = 0; b < kBlocks; b += 2) {
        uint4 t = lds128(tw_addr + (kSlot0 + b / 2) * (kF_Team * 16));
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            if (L4) {
                gs_bfly_l4(l4_bound(S, e, 1), v[i0], v[i0 + kStride], t.x, t.y, q, two_q, four_q, zero);
            } else {
                gs_bfly<(S > 0)>(v[i0], v[i0 + kStride], t.x, t.y, q, two_q, zero);
            }
        }
        if (kBlocks >= 2) {
#pragma unroll
            for (int e = 0; e < kStride; e++) {
                int i0 = (b + 1) * 2 * kStride + e;
                if (L4) {
                    gs_bfly_l4(l4_bound(S, e, 1), v[i0], v[i0 + kStride], t.z, t.w, q, two_q, four_q, zero);
                } else {
                    gs_bfly<(S > 0)>(v[i0], v[i0 + kStride], t.z, t.w, q, two_q, zero);
                }
            }
        }
    }
}

// round 2, stage K (pairs registers i and i + 2^K); twiddle table[(32 >> K) + (i >> (K+1))]
template <int K, bool L4>
__device__ __forceinline__ void round2_stage(uint32_t (&v)[64], const UniformTw &u, uint32_t q,
                                             uint32_t two_q, uint32_t four_q, uint32_t zero) {
    constexpr int kStride = 1 << K;
#pragma unroll
    for (int b = 0; b < (32 >> K); b++) {
        const uint32_t w = u.w[(32 >> K) + b], wp = u.wp[(32 >> K) + b];
#pragma unroll
        for (int e = 0; e < kStride; e++) {
            int i0 = b * 2 * kStride + e;
            if (L4) {
                // round 2 starts from whatever round 1 left (at most 4q, thread dependent)
                if (K == 5) {
                    gs_bfly_final_l4(l4_bound(K, e, 4), v[i0], v[i0 + kStride], w, wp, q, two_q, four_q, zero);
                } else {
                    gs_bfly_l4(l4_bound(K, e, 4), v[i0], v[i0 + kStride], w, wp, q, two_q, four_q, zero);
                }
            } else if (K == 5) {
                gs_bfly_final(v[i0], v[i0 + kStride], w, wp, q, two_q, zero);
            } else {
                gs_bfly<true>(v[i0], v[i0 + kStride], w, wp, q, two_q, zero);
            }
        }
    }
}

struct FusedParams {
    uint32_t *out;
    const uint4 *tw_r1;   // [32 slots][64 threads] round-1 twiddle pairs
    uint64_t batch;
    uint32_t q;
    uint32_t zero;        // always 0 (see gs_bfly)
    uint32_t four_q;      // 4q as an opaque value (computed in the kernel it is folded into LEA + VIMNMX)
    uint32_t permute;     // ans_order on store (reference src/test.cpp:69-71,212-219)
};

// IN_BR / OUT_BR: layout adapters fused into the load and the store (SURVEY 8f.2): the input
// is stored in bit-reversed order / the output is wanted in bit-reversed order.  Index
// n = 64 r + c maps to bitrev12(n) = 64 bitrev6(c) + bitrev6(r), so "row j of the natural
// polynomial" is column bitrev6(j) of the stored tile, rows taken in bit-reversed order --
// a column read with compile-time register renaming; and the natural coefficient j + 64 i
// lands in row bitrev6(j), column bitrev6(i) -- thread j writes one 256 B row from
// compile-time-permuted registers.  No extra pass over HBM in either case.
// (Measured and kept out of this kernel: round-1 twiddles in tensor memory instead of the
// 32 KiB shared-memory table, 0.471 against 0.462 ms; CTA-wide instead of team barriers,
// 0.516 ms.)
template <bool PERMUTE, bool IN_BR = false, bool OUT_BR = false, bool L4 = false>
__global__ void __launch_bounds__(kF_Threads, 1)
fused_gs4096_kernel(const __grid_constant__ CUtensorMap map_lo,
                    const __grid_constant__ CUtensorMap map_hi,
                    const __grid_constant__ UniformTw uni, const FusedParams prm) {
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment: the 128B swizzle pattern repeats every 8 rows of 128 B
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t tw_base = smem_base;                        // 32 KiB twiddles
    const uint32_t data_base = smem_base + kF_TwBytes;         // 8 x 16 KiB polynomials
    const uint32_t bar_base = data_base + kF_Teams * kF_PolyBytes;

    const int tid = threadIdx.x;
    // broadcast from lane 0 so the compiler knows the team index (and the whole
    // per-team loop) is warp-uniform: q, 2q and the opaque zero then live in uniform
    // registers instead of taking a third vector-register read port in every IADD3
    const int team = __shfl_sync(0xffffffffu, tid >> 6, 0);
    const int j = tid & 63;
    const uint32_t q = prm.q, two_q = 2u * prm.q, four_q = prm.four_q, zero = prm.zero;

    // Polynomial p goes to team (p / gridDim.x) % kF_Teams of CTA p % gridDim.x: consecutive
    // polynomials land on different SMs, so a batch that is not a multiple of gridDim.x * kF_Teams
    // ends with every SM running a few teams instead of a few SMs running all eight.
    const uint32_t buf = data_base + team * kF_PolyBytes;
    const uint32_t bar = bar_base + team * 8;
    const uint64_t stride = (uint64_t) gridDim.x * kF_Teams;
    uint64_t poly = (uint64_t) team * gridDim.x + blockIdx.x;
    uint32_t parity = 0;

    // the team's first load is in flight while the CTA stages the twiddles
    if (j == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (poly < prm.batch) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) poly);
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) poly);
        }
    }
    // stage the round-1 twiddles (kernel-private order, prepared at plan time)
    for (int i = tid; i < kF_TwSlots * kF_Team; i += kF_Threads) {
        uint4 t = __ldg(prm.tw_r1 + i);
        sts128(tw_base + i * 16, t.x, t.y, t.z, t.w);
    }
    __syncthreads();

    // shared-memory addresses.  Buffer layout (as TMA writes it): two halves of
    // [64 rows][32 words], row r / half h holds a[64r + 32h .. +31]; the 16-byte
    // chunk index inside a 128 B row is XORed with (r & 7).
    const uint32_t r1_row = buf + j * 128;            // round 1: thread j owns row j of both halves
    const uint32_t r1_xor = (j & 7) << 4;
    const uint32_t r2_col = buf + (j >> 5) * (kF_PolyBytes / 2) + (j & 3) * 4;  // round 2: column j
    const uint32_t r2_chunk = ((j & 31) >> 2) << 4;
    const uint32_t tw_addr = tw_base + j * 16;
    const uint32_t jr = __brev((uint32_t) j) >> 26;   // bitrev6(j)
    const uint32_t br_col = buf + (jr >> 5) * (kF_PolyBytes / 2) + (jr & 3) * 4;
    const uint32_t br_chunk = ((jr & 31) >> 2) << 4;

    for (; poly < prm.batch; poly += stride) {
        uint32_t v[64];
        mbar_wait(bar, parity);
        parity ^= 1;

        // ---- round 1: rows -> registers, stages 0..5
        if (IN_BR) {
            // natural a[64j + c] = stored[64 bitrev6(c) + bitrev6(j)]: column bitrev6(j)
#pragma unroll
            for (int r = 0; r < 64; r++) {
                v[kBitrev6(r)] = lds32(br_col + r * 128 + (br_chunk ^ ((r & 7) << 4)));
            }
            team_sync(team);  // the row write below overwrites other threads' columns
        } else {
#pragma unroll
            for (int c = 0; c < 16; c++) {
                uint4 t = lds128(r1_row + (c >> 3) * (kF_PolyBytes / 2) + (((c & 7) << 4) ^ r1_xor));
                v[4 * c + 0] = t.x;
                v[4 * c + 1] = t.y;
                v[4 * c + 2] = t.z;
                v[4 * c + 3] = t.w;
            }
        }
        round1_stage<0, L4>(v, tw_addr, q, two_q, four_q, zero);
        round1_stage<1, L4>(v, tw_addr, q, two_q, four_q, zero);
        round1_stage<2, L4>(v, tw_addr, q, two_q, four_q, zero);
        round1_stage<3, L4>(v, tw_addr, q, two_q, four_q, zero);
        round1_stage<4, L4>(v, tw_addr, q, two_q, four_q, zero);
        round1_stage<5, L4>(v, tw_addr, q, two_q, four_q, zero);

        // ---- exchange through the same buffer (row write, column read)
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

        // ---- the buffer is free: prefetch this team's next polynomial
        const uint64_t next = poly + stride;
        if (j == 0 && next < prm.batch) {
            mbar_expect_tx(bar, kF_PolyBytes);
            tma_load_3d(buf, &map_lo, bar, 0, 0, (int) next);
            tma_load_3d(buf + kF_PolyBytes / 2, &map_hi, bar, 0, 0, (int) next);
        }

        // ---- round 2: stages 6..11, uniform twiddles from the constant bank
        round2_stage<0, L4>(v, uni, q, two_q, four_q, zero);
        round2_stage<1, L4>(v, uni, q, two_q, four_q, zero);
        round2_stage<2, L4>(v, uni, q, two_q, four_q, zero);
        round2_stage<3, L4>(v, uni, q, two_q, four_q, zero);
        round2_stage<4, L4>(v, uni, q, two_q, four_q, zero);
        round2_stage<5, L4>(v, uni, q, two_q, four_q, zero);

        // ---- store: register i is coefficient j + 64 i; a warp writes 128 B rows
        if (OUT_BR) {
            // coefficient j + 64 i goes to 64 bitrev6(j) + bitrev6(i): one 256 B row per thread
            uint4 *row = reinterpret_cast<uint4 *>(prm.out + poly * kF_N + jr * 64);
#pragma unroll
            for (int a4 = 0; a4 < 16; a4++) {
                row[a4] = make_uint4(v[kBitrev6(4 * a4)], v[kBitrev6(4 * a4 + 1)],
                                     v[kBitrev6(4 * a4 + 2)], v[kBitrev6(4 * a4 + 3)]);
            }
            continue;
        }
        uint32_t *dst = prm.out + poly * kF_N + j;
#pragma unroll
        for (int i = 0; i < 64; i++) {
            int row = i;
            if (PERMUTE) {
                int blk = i >> 2;  // top four index bits
                blk = ((blk & 0x5) << 1) | ((blk & 0xA) >> 1);
                row = (blk << 2) | (i & 3);
            }
            dst[row * 64] = v[i];
        }
    }
}

// --------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) !=
                cudaSuccess ||
            qres != cudaDriverEntryPointSuccess) {
            return nullptr;
        }
        return (EncodeTiledFn) p;
    }();
    return fn;
}

// view of the batch for TMA: dim0 = 32 words of one half-row, dim1 = 64 rows
// (stride 256 B), dim2 = polynomial (stride 16 KiB); box = one half of one polynomial
// (general form: `rows` rows of 64 words per tile, rows*256 bytes per tile)
// tile_stride_bytes = 0: tiles are contiguous; otherwise the distance between consecutive
// tiles of this view (channel l of an RNS batch: L tiles apart)
int encode_tile_map(CUtensorMap *map, const int32_t *base, uint32_t rows, size_t batch,
                    size_t tile_stride_bytes) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return NTTB200_ERR_CUDA;
    cuuint64_t dims[3] = {32, rows, (cuuint64_t) batch};
    cuuint64_t strides[2] = {256, tile_stride_bytes ? (cuuint64_t) tile_stride_bytes : (cuuint64_t) rows * 256};
    cuuint32_t box[3] = {32, rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_INT32, 3, (void *) base, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? NTTB200_OK : NTTB200_ERR_CUDA;
}

static int make_half_map(CUtensorMap *map, const int32_t *base, size_t batch, size_t tile_stride_bytes = 0) {
    return encode_tile_map(map, base, 64, batch, tile_stride_bytes);
}

// both half-tile maps of a buffer of `tiles` contiguous 4096-word tiles
int tile_maps(CUtensorMap *lo, CUtensorMap *hi, const int32_t *base, size_t tiles) {
    int rc = make_half_map(lo, base, tiles);
    if (rc == NTTB200_OK) rc = make_half_map(hi, base + 32, tiles);
    return rc;
}
// every tile_mul-th tile starting at base: `tiles` tiles, tile_mul * 16 KiB apart
int tile_maps_strided(CUtensorMap *lo, CUtensorMap *hi, const int32_t *base, size_t tiles,
                      uint32_t tile_mul) {
    const size_t stride = (size_t) tile_mul * kF_PolyBytes;
    int rc = make_half_map(lo, base, tiles, stride);
    if (rc == NTTB200_OK) rc = make_half_map(hi, base + 32, tiles, stride);
    return rc;
}

int fused_prepare(nttb200_plan *p) {
    if (p->logn != 12) return NTTB200_ERR_UNSUPPORTED;
    // round-1 twiddles in the kernel's order: slot-major, thread-minor uint4s, two
    // (w, w') pairs per uint4; stage S block b of thread j is table[(2048>>S)+j*(32>>S)+b]
    std::vector<uint2> host(p->n);
    NTTB200_CUDA(cudaMemcpy(host.data(), p->d_tw, sizeof(uint2) * p->n, cudaMemcpyDeviceToHost));
    std::vector<uint4> r1((size_t) kF_TwSlots * kF_Team);
    for (int s = 0; s < 6; s++) {
        int blocks = 32 >> s;
        int slot0 = 32 - (blocks >= 2 ? blocks : 1);
        for (int j = 0; j < kF_Team; j++) {
            for (int b = 0; b < blocks; b += 2) {
                uint2 t0 = host[(2048 >> s) + j * blocks + b];
                uint2 t1 = blocks >= 2 ? host[(2048 >> s) + j * blocks + b + 1] : make_uint2(0, 0);
                r1[(size_t) (slot0 + b / 2) * kF_Team + j] = make_uint4(t0.x, t0.y, t1.x, t1.y);
            }
        }
    }
    NTTB200_CUDA(cudaMalloc(&p->d_tw_r1, sizeof(uint4) * r1.size()));
    NTTB200_CUDA(cudaMemcpy(p->d_tw_r1, r1.data(), sizeof(uint4) * r1.size(),
                            cudaMemcpyHostToDevice));
    for (int i = 0; i < 64; i++) {
        p->uni_gs.w[i] = host[i].x;
        p->uni_gs.wp[i] = host[i].y;
    }
    NTTB200_CUDA(cudaFuncSetAttribute(fused_gs4096_kernel<false>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, kF_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(fused_gs4096_kernel<true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, kF_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(fused_gs4096_kernel<false, false, false, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, kF_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(fused_gs4096_kernel<false, true, false>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, kF_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(fused_gs4096_kernel<false, false, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, kF_SmemBytes));
    NTTB200_CUDA(cudaFuncSetAttribute(fused_gs4096_kernel<false, true, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, kF_SmemBytes));
    return NTTB200_OK;
}

void fused_release(nttb200_plan *p) {
    if (p->d_tw_r1) cudaFree(p->d_tw_r1);
    p->d_tw_r1 = nullptr;
}

static int launch_fused_impl(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                             bool permute_out, cudaStream_t st, bool in_br = false, bool out_br = false);

int launch_fused_gs(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    bool permute_out, cudaStream_t st) {
    return launch_fused_impl(p, d_in, d_out, batch, permute_out, st);
}

// golden network with the bit-reversal adapters fused into the load and/or the store
int launch_fused_gs_bitrev(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                           bool in_br, bool out_br, cudaStream_t st) {
    if (out_br && ((uintptr_t) d_out & 15u)) return NTTB200_ERR_UNSUPPORTED;
    return launch_fused_impl(p, d_in, d_out, batch, false, st, in_br, out_br);
}

static int launch_fused_impl(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                             bool permute_out, cudaStream_t st, bool in_br, bool out_br) {
    if (p->logn != 12 || !p->d_tw_r1) return NTTB200_ERR_UNSUPPORTED;
    if (batch == 0) return NTTB200_OK;
    if (batch > 0x7fffffffull || ((uintptr_t) d_in & 15u) || ((uintptr_t) d_out & 3u)) {
        return NTTB200_ERR_UNSUPPORTED;  // TMA needs 16 B alignment; generic path serves the rest
    }
    CUtensorMap map_lo, map_hi;
    int rc = make_half_map(&map_lo, d_in, batch);
    if (rc == NTTB200_OK) rc = make_half_map(&map_hi, d_in + 32, batch);
    if (rc != NTTB200_OK) return NTTB200_ERR_UNSUPPORTED;
    FusedParams prm;
    prm.out = reinterpret_cast<uint32_t *>(d_out);
    prm.tw_r1 = p->d_tw_r1;
    prm.batch = batch;
    prm.q = p->q;
    prm.zero = 0;
    prm.four_q = 4u * p->q;   // only used when 8q fits a word
    prm.permute = permute_out;
    int grid = (int) (batch < (uint64_t) p->sm_count ? batch : (uint64_t) p->sm_count);
    if (permute_out) {
        fused_gs4096_kernel<true><<<grid, kF_Threads, kF_SmemBytes, st>>>(map_lo, map_hi, p->uni_gs,
                                                                          prm);
    } else if (in_br && out_br) {
        fused_gs4096_kernel<false, true, true><<<grid, kF_Threads, kF_SmemBytes, st>>>(
            map_lo, map_hi, p->uni_gs, prm);
    } else if (in_br) {
        fused_gs4096_kernel<false, true, false><<<grid, kF_Threads, kF_SmemBytes, st>>>(
            map_lo, map_hi, p->uni_gs, prm);
    } else if (out_br) {
        fused_gs4096_kernel<false, false, true><<<grid, kF_Threads, kF_SmemBytes, st>>>(
            map_lo, map_hi, p->uni_gs, prm);
    } else if (use_l4(p)) {
        // 8q fits a word: the 4q-lazy butterflies (fused_common.cuh, gs_bfly_l4)
        fused_gs4096_kernel<false, false, false, true><<<grid, kF_Threads, kF_SmemBytes, st>>>(
            map_lo, map_hi, p->uni_gs, prm);
    } else {
        fused_gs4096_kernel<false><<<grid, kF_Threads, kF_SmemBytes, st>>>(map_lo, map_hi,
                                                                           p->uni_gs, prm);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    p->last_path = (in_br || out_br) ? "fused_gs4096_tma_bitrev" : "fused_gs4096_tma";
    return NTTB200_OK;
}

}  // namespace nttb200
