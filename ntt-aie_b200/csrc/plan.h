// plan.h -- internal plan object and kernel launch interfaces (not installed).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "../../include/nttb200.h"

namespace nttb200 {

constexpr int kHostStreams = 4;  // chunk pipeline depth of nttb200_gs_host

// Uniform twiddles of the strided (second) round of the fused kernels: stage s of
// that round uses 2^(R2-1-k) table entries that depend only on the register index,
// never on the thread or the polynomial, so they travel as kernel parameters
// (constant bank operands of IMAD) -- 63 (w, w') pairs at most.
struct UniformTw {
    uint32_t w[64];
    uint32_t wp[64];
};

// Cross-tile twiddles table[1..15] of the one-pass polynomial kernels (stage 12+m, block b
// uses entry (G >> (m+1)) + b): kernel parameters = constant-bank operands.
struct CrossTw {
    uint32_t w[16];
    uint32_t wp[16];
};

}  // namespace nttb200

struct nttb200_plan {
    int device = 0;
    uint32_t logn = 0;
    uint32_t n = 0;
    uint32_t q = 0;
    uint32_t flags = 0;
    uint64_t mu = 0;         // floor(2^62 / q) for barrett_mul
    uint32_t n_inv = 0;      // N^-1 mod q (0 if it does not exist)
    uint32_t n_inv_shoup = 0;
    uint2 *d_tw = nullptr;   // [N] (w, floor(w*2^32/q)), golden index rule table[h+i]
    // fused-kernel twiddle staging (built lazily per kernel family)
    uint4 *d_tw_r1 = nullptr;        // round-1 per-thread twiddles, kernel-private order
    uint4 *d_tw_tile = nullptr;      // [N/4096][32][65] tile-pass twiddles (logn 12..26)
    nttb200::UniformTw uni_gs{};     // round-2 uniform twiddles, GS network
    nttb200::CrossTw cross_tw{};     // table[1..15] (logn >= 13)
    // persistent kernels (kernels_tilecol.cu): a waiter that gives up sets this word (pinned,
    // mapped host memory, allocated on first use); the next launch on the plan reports it
    uint32_t *tc_err_host = nullptr;
    uint32_t *tc_err_dev = nullptr;
    std::mutex tc_mu;                // guards the lazy allocation above (not host_mu: gs_host holds that one)
    int sm_count = 148;
    // written by every launch, possibly from several host threads driving different streams
    std::atomic<const char *> last_path{"none"};

    // nttb200_gs_host resources (lazily created, guarded by host_mu)
    std::mutex host_mu;
    cudaStream_t hstream[nttb200::kHostStreams] = {};
    int32_t *d_stage[nttb200::kHostStreams] = {};
    size_t stage_polys = 0;  // capacity of each staging buffer in polynomials
    bool host_ready = false;
};

// N = 2^12..2^16, L residue channels with their own moduli and tables (SURVEY 8f.1)
struct nttb200_rns_plan {
    int device = 0;
    uint32_t logn = 12;
    uint32_t limbs = 0;
    int sm_count = 148;
    std::vector<nttb200_plan *> sub;   // one validated single-modulus plan per channel
    uint4 *d_tw_tile = nullptr;        // [limbs][N/4096][32][65]
    uint2 *d_tw = nullptr;             // [limbs][N] (w, w') of the column pass (N > 4096 only)
    std::vector<uint4> pos;            // (q, q^-1 mod 2^32, N^-1*2^32 mod q, its Shoup companion)
    std::vector<uint4> pos_scaled;     // (q, q^-1 mod 2^32, N^-1 mod q, its Shoup companion)
};

namespace nttb200 {

constexpr int kConvMaxChannels = 32;

// Constants of one basis conversion (source moduli b_i, product B; target moduli c_j), passed
// to the kernel as one __grid_constant__ parameter block (6016 bytes).  The fields after wp serve
// the exact operations only; they come last so that the others keep their offsets.
struct RnsConvConsts {
    uint32_t m[kConvMaxChannels][kConvMaxChannels];   // [j][i] = (B / b_i) mod c_j
    uint64_t mu[kConvMaxChannels];     // floor(2^64 / c_j) for reduce64
    uint32_t c[kConvMaxChannels];      // c_j
    uint32_t hc[kConvMaxChannels];     // floor(B/2) mod c_j (0 when not rounding)
    uint32_t binv[kConvMaxChannels];   // B^-1 mod c_j
    uint32_t binvp[kConvMaxChannels];  // its Shoup companion
    uint32_t b[kConvMaxChannels];      // b_i
    uint32_t hb[kConvMaxChannels];     // floor(B/2) mod b_i (0 when not rounding)
    uint32_t w[kConvMaxChannels];      // (B / b_i)^-1 mod b_i
    uint32_t wp[kConvMaxChannels];     // its Shoup companion
    double binvd[kConvMaxChannels];    // 1 / b_i, correctly rounded
    uint32_t nbc[kConvMaxChannels];    // -B mod c_j
    uint32_t tc[kConvMaxChannels];     // t mod c_j (scale-and-round, set per call)
    uint32_t tcp[kConvMaxChannels];    // its Shoup companion
};

// What rns_conv_kernel computes: the fast conversion, the division by B, the exact conversion
// of the centred value, round(t X / B).
enum class ConvMode : int { Fast, Down, Exact, Scale };

}  // namespace nttb200

// Self-contained: copies what it needs from the two plans, which may be destroyed afterwards.
struct nttb200_rns_conv {
    int device = 0;
    uint32_t logn = 12;
    uint32_t src = 0;                  // S
    uint32_t dst = 0;                  // T
    int sm_count = 148;
    nttb200::RnsConvConsts k{};        // hc / hb hold floor(B/2); zeroed per call without rounding
};

namespace nttb200 {

extern std::atomic<uint64_t> g_launches;

// error plumbing (api.cu)
int cuda_fail(cudaError_t e, const char *what);
#define NTTB200_CUDA(call)                                        \
    do {                                                          \
        cudaError_t e__ = (call);                                 \
        if (e__ != cudaSuccess) return ::nttb200::cuda_fail(e__, #call); \
    } while (0)

// 4q-lazy kernels (fused_common.cuh, gs_bfly_l4 / ct_bfly_l4) serve moduli whose 8q fits a word.
inline bool use_l4(const nttb200_plan *p) { return p->q < (1u << 29); }

// Stream-ordered scratch (transform scratch of the multi-kernel products, the counters of the
// persistent kernel) from a library-private memory pool of the CURRENT device that keeps its
// pages across synchronisations (release threshold = max): with the default pool every
// cudaDeviceSynchronize hands the pages back to the driver and the next call pays milliseconds
// to map them again (measured: 8 ms on the first product after a synchronize at N = 2^13).
// Freed with cudaFreeAsync; trimmed when the last plan of the process is destroyed.
int scratch_alloc_async(void **p, size_t bytes, cudaStream_t st);

// device-side table construction and input canonicalisation (tables.cu)
int build_shoup_table(nttb200_plan *p, const int32_t *d_table);
int build_generated_table(nttb200_plan *p, uint32_t kind, uint32_t base, uint32_t gen_logn,
                          uint32_t block_mult);
int build_tile_table(nttb200_plan *p);
int launch_bitrev_permute(nttb200_plan *p, const int32_t *in, int32_t *out, size_t batch,
                          cudaStream_t st);
int launch_transpose(nttb200_plan *p, const int32_t *in, int32_t *out, uint64_t rows, uint64_t cols,
                     cudaStream_t st);
int launch_reduce(nttb200_plan *p, const int32_t *in, int32_t *out, size_t count, cudaStream_t st);

// N = 2^13..2^15 in one pass, private twiddles in tensor memory (kernels_poly.cu)
int polyt_prepare();
int launch_polyt_gs(nttb200_plan *p, const int32_t *d_in, const int32_t *d_b, int32_t *d_out,
                    size_t batch, cudaStream_t st);
int launch_polyt_ct(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    cudaStream_t st);

// N = 2^16 as one persistent kernel of tile items and column items (kernels_tilecol.cu)
int tilecol_prepare();
int launch_tilecol_gs(nttb200_plan *p, const int32_t *d_in, const int32_t *d_b, int32_t *d_out,
                      size_t batch, cudaStream_t st);

int launch_tilecol_ct(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch, cudaStream_t st);
void tilecol_release(nttb200_plan *p);
int fail_msg(int status, const char *msg);   // sets nttb200_last_error, returns status

// one-kernel negacyclic product, N = 4096 (kernels_polymul.cu)
int polymul_prepare();
int launch_polymul4096(nttb200_plan *fwd, nttb200_plan *inv, const int32_t *d_a, const int32_t *d_b,
                       int32_t *d_c, size_t batch, cudaStream_t st);
int launch_polymul4096_strided(nttb200_plan *fwd, nttb200_plan *inv, const int32_t *d_a,
                               const int32_t *d_b, int32_t *d_c, size_t batch, uint32_t tile_mul,
                               uint32_t tile_off, cudaStream_t st);

// generic stage-pass kernels (kernels_generic.cu): stages [sb, se) of the GS
// (ascending stride) or CT (descending stride) network; permute_out applies the
// ans_order block permutation on the last pass's store.
int generic_prepare();
int launch_generic(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch, int sb,
                   int se, bool ct, bool permute_out, cudaStream_t st);
int launch_pointwise(nttb200_plan *p, const int32_t *a, const int32_t *b, int32_t *c, size_t count,
                     cudaStream_t st);
int launch_scale(nttb200_plan *p, const int32_t *a, int32_t *c, size_t count, uint32_t s,
                 uint32_t s_shoup, cudaStream_t st);

// fused register-radix kernels (kernels_fused.cu).  Return NTTB200_ERR_UNSUPPORTED
// when the (logn, options) combination has no fused kernel so the caller can fall
// back to the generic passes (still CUDA -- never a CPU path).
int fused_prepare(nttb200_plan *p);
void fused_release(nttb200_plan *p);
int launch_fused_gs_bitrev(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                           bool in_br, bool out_br, cudaStream_t st);
int launch_fused_gs(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    bool permute_out, cudaStream_t st);

// warp-per-block kernel for N = 2^9..2^11 (kernels_small.cu)
int small_prepare(nttb200_plan *p);
int launch_small(nttb200_plan *p, int kind, const int32_t *d_in, const int32_t *d_b, int32_t *d_out,
                 size_t batch, cudaStream_t st, size_t *done_polys);
int launch_small_gs(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    bool permute_out, cudaStream_t st, size_t *done_polys);

// tile pass + column passes for logn 12..26 (kernels_multi.cu)
int multi_prepare(nttb200_plan *p);
void multi_release(nttb200_plan *p);
int launch_multi_gs(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    cudaStream_t st);
int launch_column_pass(nttb200_plan *p, const int32_t *in, int32_t *out, size_t batch, int s0, int k,
                       cudaStream_t st);
int launch_gs_range_scatter(nttb200_plan *p, int32_t *d_buf, int sb, int se, void *const *peers,
                            int world, int rank, cudaStream_t st);
int rns_launch(const nttb200_rns_plan *rp, int kind, const int32_t *d_a, const int32_t *d_b,
               int32_t *d_out, size_t batch, cudaStream_t st);
// evaluation-domain operators on RNS batches (kernels_rns_eval.cu); the caller has checked the
// arguments, the aliasing and the 16-byte alignment
int launch_rns_stream(const nttb200_rns_plan *rp, uint32_t op, const int32_t *a, const int32_t *b, int32_t *c,
                      size_t batch, bool bcast, const uint32_t *scalars, cudaStream_t st);
int launch_rns_dot(const nttb200_rns_plan *rp, const int32_t *a, const int32_t *w, int32_t *c, uint32_t terms,
                   size_t batch, bool w_shared, bool accumulate, cudaStream_t st);
// basis conversion (kernels_rns_conv.cu).  rns_conv_prepare fills cv->k from the moduli
// (host only; NTTB200_ERR_MODULUS when two of them share a factor).  launch_rns_conv: the
// caller has checked the arguments, the overlap and the 16-byte alignment; src rows (S
// channels) at src + b * src_stride, target input rows (Down and Scale) at tin + b * src_stride,
// output rows (T channels) at out + b * out_stride; round applies to Down, t (>= 1) to Scale.
int rns_conv_prepare(nttb200_rns_conv *cv, const uint32_t *b, const uint32_t *c);
int launch_rns_conv(const nttb200_rns_conv *cv, const int32_t *src, const int32_t *tin, uint64_t src_stride,
                    int32_t *out, uint64_t out_stride, size_t batch, ConvMode mode, bool round, uint32_t t,
                    cudaStream_t st);
// Galois automorphisms (kernels_rns_automorph.cu), one __grid_constant__ parameter block
// (896 bytes).  launch_rns_automorph: the caller has checked the arguments (1 <= count <= 64,
// every g odd in [1, 2N)), the overlap and the 16-byte alignment; eval selects the
// evaluation-domain (rns_ct order) permutation, else the coefficient domain.
constexpr int kAutoMaxElems = 64;
struct RnsAutoConsts {
    uint32_t g[kAutoMaxElems];      // g
    uint32_t ginv[kAutoMaxElems];   // g^-1 mod 2N
    uint32_t off[kAutoMaxElems];    // (g - 1) / 2 mod N, the evaluation-domain offset
    uint32_t q[kConvMaxChannels];   // q_l
};
int launch_rns_automorph(const nttb200_rns_plan *rp, const int32_t *in, int32_t *out, size_t batch,
                         const uint32_t *galois, uint32_t count, bool eval, cudaStream_t st);
// q^-1 mod 2^32 for odd q (Montgomery products): Newton iteration, 3 correct bits doubling per step
inline uint32_t inv_mod_2_32(uint32_t q) {
    uint32_t x = q;
    for (int i = 0; i < 5; i++) x *= 2u - q * x;
    return x;
}
constexpr int kRnsTwTile = 32 * 65;  // uint4s per tile position in d_tw_tile (kernels_multi.cu)
int launch_multi_ct(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                    cudaStream_t st);
int launch_multi_gs_dual(nttb200_plan *p, const int32_t *d_a, const int32_t *d_b, int32_t *d_out,
                         size_t batch, cudaStream_t st);

// CKKS slot encoding and decoding (kernels_ckks.cu).  Channel moduli of the encoder, one
// __grid_constant__ block per encode call.
struct CkksEncConsts {
    uint64_t mu[kConvMaxChannels];   // floor(2^64 / q_l) for reduce64
    uint32_t q[kConvMaxChannels];
};
constexpr int kCkksMaxDecode = 4;
// Exact CRT of the first C <= 4 channels (moduli b_i, product B < 2^120), set per decode call.
struct CkksDecConsts {
    uint64_t m[kCkksMaxDecode][2];   // B / b_i as (low, high) 64-bit limbs
    uint64_t t[kCkksMaxDecode][2];   // (2k + 1) B: S > (k + 1/2) B  <=>  2S > (2k + 1) B
    uint64_t bb[2];                  // B
    uint32_t b[kCkksMaxDecode];      // b_i
    uint32_t w[kCkksMaxDecode];      // (B / b_i)^-1 mod b_i
    uint32_t wp[kCkksMaxDecode];     // its Shoup companion
    double inv_scale;                // 1 / scale, correctly rounded
};

}  // namespace nttb200

// Self-contained: copies N, the device and the moduli from the plan, which may be destroyed.
struct nttb200_ckks_encoder {
    int device = 0;
    uint32_t logn = 12;
    uint32_t limbs = 0;
    int sm_count = 148;
    nttb200::CkksEncConsts k{};
    double2 *d_w = nullptr;        // [n] e^(2 pi i t / n), n = N/2 slots
    double2 *d_zeta = nullptr;     // [n] zeta^k = e^(i pi k / N)
    uint32_t *d_perm = nullptr;    // [n] s_j = (5^j mod 2N - 1) / 4
    uint32_t *d_iperm = nullptr;   // [n] j of s
};

namespace nttb200 {
// builds the device tables of a filled-in encoder (device current); ckks_release frees them
int ckks_prepare(nttb200_ckks_encoder *enc);
void ckks_release(nttb200_ckks_encoder *enc);
// the CRT constants of the first `channels` moduli (NTTB200_ERR_MODULUS when two share a factor)
int ckks_decode_consts(const nttb200_ckks_encoder *enc, uint32_t channels, double scale, CkksDecConsts *k);
// the caller has checked the arguments, the overlap and the 16-byte alignment
int launch_ckks_encode(const nttb200_ckks_encoder *enc, const double2 *slots, double scale, int32_t *out,
                       size_t batch, cudaStream_t st);
int launch_ckks_decode(const nttb200_ckks_encoder *enc, const int32_t *in, uint64_t in_stride, uint32_t channels,
                       const CkksDecConsts &k, double2 *slots, size_t batch, cudaStream_t st);

// Packed integer slots mod t (kernels_packed.cu): the constants of the lift onto the L channels,
// one __grid_constant__ block (656 bytes) built at create time.
struct PackedConsts {
    uint64_t mu[kConvMaxChannels];      // floor(2^64 / q_l) for reduce64
    uint32_t q[kConvMaxChannels];       // q_l
    uint32_t delta[kConvMaxChannels];   // floor(Q / t) mod q_l = -r t^-1 mod q_l
    uint32_t negt[kConvMaxChannels];    // -t mod q_l
    uint64_t mu_t;                      // floor(2^64 / t)
    uint32_t t;
    uint32_t r;                         // Q mod t
};
}  // namespace nttb200

// Self-contained: copies N, the device and the moduli from the plan, which may be destroyed.
struct nttb200_packed_encoder {
    int device = 0;
    uint32_t logn = 12;
    uint32_t limbs = 0;
    int sm_count = 148;
    nttb200::PackedConsts k{};
    nttb200_rns_plan *fwd = nullptr;   // one channel of modulus t, psi^bitrev table (rns_ct)
    nttb200_rns_plan *inv = nullptr;   // psi^-bitrev table (rns_gs_scaled)
    uint32_t *d_slot = nullptr;        // [N] k_i, the rns_ct index of slot i
    uint32_t *d_islot = nullptr;       // [N] i of k
};

namespace nttb200 {
// psi, the plans and the slot tables of a filled-in encoder (k.q, k.t and logn set; device
// current); packed_release frees them
int packed_prepare(nttb200_packed_encoder *enc);
void packed_release(nttb200_packed_encoder *enc);
// the caller has checked the arguments, the overlap, the 16-byte alignment and the size
int launch_packed_encode(const nttb200_packed_encoder *enc, const int32_t *slots, bool centred, int32_t *out,
                         size_t batch, cudaStream_t st);
int launch_packed_decode(const nttb200_packed_encoder *enc, const int32_t *in, bool centred, int32_t *slots,
                         size_t batch, cudaStream_t st);

// Hybrid key switching (kernels_rns_keyswitch.cu): the Galois constants of one call and the
// per-channel moduli of Q P, one __grid_constant__ block (896 bytes).
struct RnsKsConsts {
    uint32_t g[kAutoMaxElems];      // g
    uint32_t off[kAutoMaxElems];    // (g - 1) / 2 mod N, the evaluation-domain offset
    uint64_t mu[kConvMaxChannels];  // floor(2^64 / q_l) for reduce64
    uint32_t q[kConvMaxChannels];   // q_l
};
}  // namespace nttb200

// Self-contained: own transform plans built from the given plans' tables, and own conversion
// constants; the plans given to nttb200_rns_keyswitch_create may be destroyed afterwards.
struct nttb200_rns_keyswitch {
    int device = 0;
    uint32_t logn = 12;
    uint32_t q_limbs = 0;   // L
    uint32_t limbs = 0;     // L + K
    uint32_t alpha = 0;
    uint32_t dnum = 0;      // ceil(L / alpha)
    int sm_count = 148;
    nttb200_rns_plan *q_fwd = nullptr, *q_inv = nullptr;     // the first L channels
    nttb200_rns_plan *qp_fwd = nullptr, *qp_inv = nullptr;   // all L + K channels
    std::vector<nttb200_rns_conv> up_lo;   // [i - 1]: digit i -> Q channels [0, i alpha), i >= 1
    std::vector<nttb200_rns_conv> up_hi;   // [i]: digit i -> channels [min((i + 1) alpha, L), L + K)
    nttb200_rns_conv down;                 // P -> Q
};

namespace nttb200 {
// the plans and conversion constants of a filled-in object (logn, limbs, alpha, dnum set; device
// current; the moduli checked); keyswitch_release frees them
int keyswitch_prepare(nttb200_rns_keyswitch *ks, const nttb200_rns_plan *qp_fwd, const nttb200_rns_plan *qp_inv);
void keyswitch_release(nttb200_rns_keyswitch *ks);
// the caller has checked the arguments, the overlap, the 16-byte alignment and the sizes; paired:
// the input is count * batch polynomials (rows at in + (c * batch + b) * in_stride) and element c
// switches only its own batch of them
int launch_keyswitch(const nttb200_rns_keyswitch *ks, const int32_t *in, uint64_t in_stride, const int32_t *keys,
                     const uint32_t *galois, uint32_t count, int32_t *out, size_t batch, bool coeff_in,
                     bool coeff_out, bool paired, cudaStream_t st);

// Plaintext matrix-vector products (kernels_rns_lintrans.cu): the baby-step giant-step schedule
// of an offset set, babies j = k mod n1 >= 1 and giants i = k / n1 in ascending order.
struct LintransSchedule {
    std::vector<uint32_t> babies;                 // the j >= 1 that occur
    std::vector<uint32_t> giants;                 // every i that occurs, 0 included
    std::vector<uint32_t> offsets;                // a copy of the call's offsets
    std::vector<std::vector<uint32_t>> terms;     // [giant] the indices into the offsets of its terms
};
// INVALID_ARG for a bad logn, n1, count, a null offsets, an offset >= N/2 or a duplicated one
int lintrans_schedule(uint32_t logn, const uint32_t *offsets, uint32_t count, uint32_t n1, LintransSchedule *s);
// the caller has checked everything, the schedule and the key count included
int launch_lintrans(const nttb200_rns_keyswitch *ks, const int32_t *ct, const int32_t *diags,
                    const LintransSchedule &s, uint32_t n1, const int32_t *keys, int32_t *out, size_t batch,
                    cudaStream_t st);
}  // namespace nttb200
