/*
 * nttb200.h -- C ABI of the B200-native NTT engine (libnttb200.so).
 *
 * This is the drop-in boundary for the ONE hot path of hal-lab-u-tokyo/ntt-aie:
 * the butterfly-stage network with 32-bit modular multiplication over a
 * precomputed twiddle table.  Plain pointers and sizes only; no C++ types, no
 * torch types, no exceptions cross this boundary.  Every entry point names the
 * reference interface it replaces (paths relative to the reference tree).
 *
 * Conventions
 *   - element type is int32_t exactly as in the reference (src/test.cpp:34,
 *     src/aie_core.cc:161,189); values are canonical residues in [0, q);
 *   - polynomials are batch-major contiguous: poly b occupies [b*N, (b+1)*N);
 *   - the twiddle table is an INPUT of length N indexed table[h + i]
 *     (src/test.cpp:45): h = number of butterfly blocks of the stage, i = block
 *     index; table[0] is never read.  Any canonical residues are accepted -- the
 *     reference's own natural-power table (src/test.cpp:27-32) reproduces the
 *     reference bit for bit, bit-reversed psi tables make it a real (I)NTT;
 *   - return value 0 = success, non-zero = nttb200_status (the reference's host
 *     returns 0/1 from main, src/test.cpp:162-166,240-247);
 *   - device entry points are asynchronous on the given CUDA stream
 *     (cudaStream_t passed as void*, NULL = default stream); in == out (in place)
 *     is allowed; host entry points are synchronous;
 *   - alignment: every device pointer need only be 4-byte aligned (views such as
 *     t[1:] or one channel of a batch are fine).  16-byte alignment of all of a
 *     call's buffers selects the fast kernels; any other pointer takes the
 *     generic kernels (the stage passes; the word loop of pointwise / scale),
 *     with the same results.  The N = 4096 golden kernel also
 *     runs on an output that is only 4-byte aligned (not with
 *     NTTB200_OUTPUT_BITREV).  Exceptions: the RNS entry points and
 *     nttb200_gs_stage_range_scatter need 16-byte-aligned buffers and return
 *     NTTB200_ERR_UNSUPPORTED otherwise (the scatter returns
 *     NTTB200_ERR_INVALID_ARG for an unaligned peer buffer), except for d_c of
 *     nttb200_rns_polymul_negacyclic at N = 4096, which needs 4-byte alignment only;
 *   - there is NO CPU fallback: every compute entry point fails with
 *     NTTB200_ERR_CUDA / NTTB200_ERR_NO_DEVICE when no B200 is usable.
 */
#ifndef NTTB200_H
#define NTTB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define NTTB200_API __attribute__((visibility("default")))
#else
#define NTTB200_API
#endif

typedef enum nttb200_status {
    NTTB200_OK = 0,
    NTTB200_ERR_INVALID_ARG = 1, /* null pointer, logn out of range, bad flags      */
    NTTB200_ERR_MODULUS = 2,     /* q outside [2, 2^31).  q <= 2^30 is the golden's  */
                                 /* own domain (2q-1 <= INT32_MAX, src/test.cpp:     */
                                 /* 48,50) and takes the fast kernels; 2^30 < q <    */
                                 /* 2^31 is served by the canonical stage-pass       */
                                 /* kernels (wider moduli, outside the reference)    */
    NTTB200_ERR_TABLE = 3,       /* table entry outside [0, q)                      */
    NTTB200_ERR_CUDA = 4,        /* a CUDA call failed; see nttb200_last_error()    */
    NTTB200_ERR_NO_DEVICE = 5,   /* no CUDA device / wrong device ordinal           */
    NTTB200_ERR_ALLOC = 6,       /* host or device allocation failed                */
    NTTB200_ERR_UNSUPPORTED = 7  /* valid request this build cannot serve           */
} nttb200_status;

/* plan flags */
#define NTTB200_ORDER_GOLDEN 0u     /* output in the CPU golden's order (src/test.cpp:34-60)    */
#define NTTB200_ORDER_AIE_DEVICE 1u /* output permuted in 16 blocks of N/16 by ans_order, as the */
                                    /* AIE device leaves it (src/test.cpp:69-71,212-219); N>=16. */
                                    /* Applies to nttb200_gs_batch / gs_host at full depth only: */
                                    /* a partial depth, ct_batch and gs_stage_range return the   */
                                    /* unpermuted (golden) order on such a plan.                 */
#define NTTB200_FORCE_GENERIC 2u    /* debugging: always take the generic stage-pass kernels     */

#define NTTB200_REDUCE_INPUT 4u     /* nttb200_gs_batch / ct_batch accept ANY int32 words and reduce */
                                    /* them mod q first, as the golden's `%` does on first touch     */
                                    /* (src/test.cpp:46-50; e.g. a[i] = i with n > p); costs one     */
                                    /* extra pass.  Without it device inputs must be in [0, q).      */
                                    /* nttb200_gs_host always reduces (the pass hides behind PCIe).  */

#define NTTB200_INPUT_BITREV 8u     /* layout adapters (new; SURVEY 8f.2): the input is stored in    */
#define NTTB200_OUTPUT_BITREV 16u   /* bit-reversed order / the output is delivered in bit-reversed  */
                                    /* order (index i <-> bitrev_logn(i) inside every polynomial).   */
                                    /* Fused into the load / store of the N = 4096 golden kernel     */
                                    /* (no extra pass); one permutation pass elsewhere.  Not         */
                                    /* combinable with NTTB200_ORDER_AIE_DEVICE.                     */

#define NTTB200_MAX_LOGN 27

/* Opaque plan: owns the device copies of the twiddle table (+ Shoup companions
 * floor(w*2^32/q)) for one (N, q, table).  Replaces the compile-time constants
 * the reference bakes into its device image (N, p, Barrett w/u:
 * src/aie2.py:14-19,178) and the root-table buffer object bo_root
 * (src/test.cpp:119-120,137-144,150). */
typedef struct nttb200_plan nttb200_plan;

/* ---- host-side table generation ------------------------------------------ */

/* Replaces make_roots + modPow (src/test.cpp:15-32) exactly as main() uses them
 * (src/test.cpp:137-139): roots[0] = 1, w = g^((p-1)/n) with INTEGER division,
 * roots[i] = roots[i-1]*w mod p.  64-bit intermediates, so it stays correct for
 * every p <= 2^30 (the reference's int32/uint32 products are only valid for
 * p < 46341). */
NTTB200_API int nttb200_make_roots(int32_t n, int32_t *roots, int32_t p, int32_t g);

/* table[k] = base^bitrev_logn(k) mod p (table[0] = 1): with base = psi (a
 * primitive 2n-th root of unity) this is the forward table of nttb200_ct_batch,
 * with base = psi^-1 it turns the golden network (nttb200_gs_batch) into the
 * un-scaled inverse negacyclic NTT.  New operator, no reference counterpart. */
NTTB200_API int nttb200_make_bitrev_table(int32_t n, int32_t *table, int32_t p, int32_t base);

/* b^e mod m with 64-bit intermediates (helper for psi, n^-1 ...). */
NTTB200_API int32_t nttb200_powmod(int32_t b, int64_t e, int32_t m);

/* ---- plan ------------------------------------------------------------------ */

/* Replaces device image load + bo_root fill/sync (src/test.cpp:110-112,137-151).
 * table_host: N = 2^logn int32 words on the host, index rule above.  1 <= logn <=
 * NTTB200_MAX_LOGN, 2 <= q < 2^31 (see NTTB200_ERR_MODULUS). */
NTTB200_API int nttb200_plan_create(nttb200_plan **plan, int device, uint32_t logn, uint32_t q,
                                    const int32_t *table_host, uint32_t flags);
NTTB200_API int nttb200_plan_destroy(nttb200_plan *plan);

/* Same plan, but the table is GENERATED ON THE DEVICE -- the host ships nothing
 * (the reference builds its table on the host and syncs it to the device,
 * src/test.cpp:27-32,137-151; at N = 2^26 that is a 256 MiB upload per plan):
 *     table[h + i] = gen(h * block_mult + i),   h = 1, 2, .., N/2,  i < h,  table[0] = 1
 *     NTTB200_GEN_POWERS: gen(e) = base^e mod q
 *     NTTB200_GEN_BITREV: gen(e) = base^bitrev(e) mod q, bit reversal over gen_logn bits
 * With gen_logn = logn and block_mult = 1 these are make_roots (base = g^((q-1)/N)) and
 * nttb200_make_bitrev_table.  gen_logn > logn with block_mult = G + r gives rank r's local
 * table of a transform of length 2^gen_logn split over G = 2^(gen_logn-logn) devices
 * (the derived table T_r of the four-step split), block_mult = 1 its cross-device table.
 * Needs (N/2) * (block_mult + 1) <= 2^gen_logn and base < q. */
#define NTTB200_GEN_POWERS 0u
#define NTTB200_GEN_BITREV 1u
NTTB200_API int nttb200_plan_create_generated(nttb200_plan **plan, int device, uint32_t logn,
                                              uint32_t q, uint32_t kind, uint32_t base,
                                              uint32_t gen_logn, uint32_t block_mult,
                                              uint32_t flags);

/* Copies the plan's table (N words, the w values; table[0] reported as 1) to the host:
 * what the reference would have had in bo_root (src/test.cpp:119-120). */
NTTB200_API int nttb200_plan_table(const nttb200_plan *plan, int32_t *table_host);

/* ---- the hot path ---------------------------------------------------------- */

/* Replaces the golden `ntt(a, n, roots_rev, p, stage)` (src/test.cpp:34-60) and
 * the device kernels that implement it (ntt_stage0_to_Nminus5 + ntt_1stage +
 * swap_buff + write_back, src/aie_core.cc:133-361, scheduled by src/aie2.py:
 * 161-317): Gentleman-Sande network, stride 1 -> N/2, twiddle table[h+i].
 * stage_limit mirrors the golden's early exit (src/test.cpp:55-58): stages
 * 0..stage_limit are applied; any value outside [0, logn-2] means full depth
 * (the reference passes n-1, src/test.cpp:67).  d_in/d_out: device pointers,
 * batch*N words. */
NTTB200_API int nttb200_gs_batch(nttb200_plan *plan, const int32_t *d_in, int32_t *d_out,
                                 size_t batch, int stage_limit, void *cuda_stream);

/* Forward partner (new operator): Cooley-Tukey network, stride N/2 -> 1, twiddle
 * table[m+i], butterfly V = a[j+t]*S; a[j] = U+V; a[j+t] = U-V.  Same table
 * index rule, same stage_limit meaning. */
NTTB200_API int nttb200_ct_batch(nttb200_plan *plan, const int32_t *d_in, int32_t *d_out,
                                 size_t batch, int stage_limit, void *cuda_stream);

/* A contiguous range of stages [stage_begin, stage_end) of the GS network on
 * batch polynomials: the building block of the multi-GPU split (the reference
 * splits one transform the same way: tile-local stages, then cross-tile stages,
 * src/aie2.py:178-295).  Stage s has stride 2^s. */
NTTB200_API int nttb200_gs_stage_range(nttb200_plan *plan, const int32_t *d_in, int32_t *d_out,
                                       size_t batch, int stage_begin, int stage_end,
                                       void *cuda_stream);

/* The exchange step of the multi-GPU split fused into the last pass: stages
 * [stage_begin, stage_end = logn) of ONE length-N vector d_buf (this rank's shard or
 * its post-transpose rows), whose results are stored straight into the peers that own
 * them after the transpose -- element idx goes to peer idx >> (logn - log2 world) at
 * offset rank*2^(logn-log2 world) + (idx mod 2^(logn-log2 world)).  peer_bufs[k] is a
 * device pointer to rank k's receive buffer mapped into this process (CUDA IPC /
 * symmetric memory; peer_bufs[rank] is the local one).  The successor of the
 * reference's cross-tile butterflies that write into a neighbour tile's memory
 * (src/aie2.py:184-187,226-229).  The caller synchronises the ranks before the
 * receive buffers are read.  world: power of two <= 16. */
NTTB200_API int nttb200_gs_stage_range_scatter(nttb200_plan *plan, int32_t *d_buf, int stage_begin,
                                               int stage_end, void *const *peer_bufs, int world,
                                               int rank, void *cuda_stream);

/* Host-buffer form of the hot path: what the reference host does around one
 * launch -- sync inputs to the device, run, sync the output back
 * (src/test.cpp:148-151,159-168,181-190).  h_in/h_out are HOST pointers
 * (pinned or pageable), batch*N words.  Copies and kernels are pipelined in
 * chunks over internal streams; returns after h_out is complete. */
NTTB200_API int nttb200_gs_host(nttb200_plan *plan, const int32_t *h_in, int32_t *h_out,
                                size_t batch, int stage_limit);

/* Page-locked host buffers for nttb200_gs_host: the successor of the reference's
 * host-only buffer objects `xrt::bo(device, size, XRT_BO_FLAGS_HOST_ONLY, ...)` +
 * `.map<int32_t*>()` (src/test.cpp:115-134).  write_combined != 0 asks for
 * write-combined memory (fast for the device to read, slow for the CPU to read back:
 * use it for inputs only). */
/* out[b][i] = in[b][bitrev_logn(i)] for batch polynomials (in place allowed): the
 * standalone bit-reversal adapter. */
NTTB200_API int nttb200_bitrev_permute(nttb200_plan *plan, const int32_t *d_in, int32_t *d_out,
                                       size_t batch, void *cuda_stream);

/* Layout adapter: batch-major [batch][N] (this library's layout, the reference's flat buffer
 * object per transform) <-> batch-minor [N][batch] (coefficient i of polynomial b at
 * i*batch + b).  to_batch_minor != 0: d_in is [batch][N], d_out becomes [N][batch]; 0: the
 * reverse.  One transposing pass, out of place (d_in != d_out). */
NTTB200_API int nttb200_transpose(nttb200_plan *plan, const int32_t *d_in, int32_t *d_out,
                                  size_t batch, int to_batch_minor, void *cuda_stream);

/* out[i] = in[i] mod q in [0, q) for ANY int32 words (device pointers): the reduction the
 * golden applies with `%` when it first touches an input (src/test.cpp:46-50). */
NTTB200_API int nttb200_reduce(nttb200_plan *plan, const int32_t *d_in, int32_t *d_out,
                               size_t count, void *cuda_stream);

NTTB200_API int nttb200_host_alloc(void **ptr, size_t bytes, int write_combined);
NTTB200_API int nttb200_host_free(void *ptr);

/* ---- operators that make it a polynomial multiplier (new) ------------------- */

/* c[i] = a[i]*b[i] mod q over count words. */
NTTB200_API int nttb200_pointwise(nttb200_plan *plan, const int32_t *d_a, const int32_t *d_b,
                                  int32_t *d_c, size_t count, void *cuda_stream);

/* c[i] = a[i]*scalar mod q over count words (scalar in [0,q)), e.g. N^-1. */
NTTB200_API int nttb200_scale(nttb200_plan *plan, const int32_t *d_a, int32_t *d_c, size_t count,
                              int32_t scalar, void *cuda_stream);

/* c = a (*) b mod (x^N + 1, q) for batch products: CT(fwd) on a and b,
 * pointwise product, GS(inv), scaled by N^-1.  fwd must hold psi^bitrev, inv
 * must hold psi^-bitrev (nttb200_make_bitrev_table); both plans share N and q.
 * d_c may alias d_a or d_b.  d_a/d_b are not modified unless aliased. */
NTTB200_API int nttb200_polymul_negacyclic(nttb200_plan *fwd, nttb200_plan *inv,
                                           const int32_t *d_a, const int32_t *d_b, int32_t *d_c,
                                           size_t batch, void *cuda_stream);

/* ---- RNS batches (new; SURVEY 8f.1) ------------------------------------------- */

/* Polynomials in residue-number-system form: L channels ("limbs") modulo L different
 * primes, N = 2^logn with 12 <= logn <= 16 (N = 4096 .. 65536), coefficients laid out
 * [batch][L][N]: channel l of polynomial b sits at (b*L + l)*N and is transformed modulo
 * q[l] with its own table tables_host[l] (N words, the golden's table[h+i] rule).
 * 1 <= L <= 32, 2 <= q[l] <= 2^30 (wider moduli give NTTB200_ERR_UNSUPPORTED), flags 0.
 * N = 4096: one launch per transform serves all channels (the kernels pick twiddles AND
 * modulus by channel).  N > 4096: two launches per transform serve all channels, a tile
 * pass (stages 0..11) and a column pass (stages 12..logn-1).
 * Argument errors are returned before any device is touched: logn outside [1, 27],
 * limbs outside [1, 32], a null pointer or flags != 0 -> NTTB200_ERR_INVALID_ARG; another
 * logn in [1, 27] -> NTTB200_ERR_UNSUPPORTED; q[l] outside [2, 2^31) -> NTTB200_ERR_MODULUS;
 * tables_host[l][i] outside [0, q[l]) for some i >= 1 -> NTTB200_ERR_TABLE. */
typedef struct nttb200_rns_plan nttb200_rns_plan;
NTTB200_API int nttb200_rns_plan_create_logn(nttb200_rns_plan **plan, int device, uint32_t logn,
                                             uint32_t limbs, const uint32_t *q,
                                             const int32_t *const *tables_host, uint32_t flags);
/* nttb200_rns_plan_create_logn with logn = 12 */
NTTB200_API int nttb200_rns_plan_create(nttb200_rns_plan **plan, int device, uint32_t limbs,
                                        const uint32_t *q, const int32_t *const *tables_host,
                                        uint32_t flags);
/* Same plan with every channel's table GENERATED ON THE DEVICE, as
 * nttb200_plan_create_generated(.., logn, q[l], kind, bases[l], gen_logn = logn,
 * block_mult = 1, ..) builds it: kind = NTTB200_GEN_BITREV with bases[l] = psi_l gives the
 * forward table of the negacyclic product, psi_l^-1 the inverse one.  Same logn, limbs, q
 * and flags rules; kind > NTTB200_GEN_BITREV or bases == NULL -> NTTB200_ERR_INVALID_ARG,
 * bases[l] >= q[l] -> NTTB200_ERR_TABLE. */
NTTB200_API int nttb200_rns_plan_create_generated(nttb200_rns_plan **plan, int device, uint32_t logn,
                                                  uint32_t limbs, const uint32_t *q, uint32_t kind,
                                                  const uint32_t *bases, uint32_t flags);
NTTB200_API int nttb200_rns_plan_destroy(nttb200_rns_plan *plan);
/* golden GS network / CT network on every channel of every polynomial; N from the plan.
 * batch * L * N / 4096 must stay below 2^31 (else NTTB200_ERR_UNSUPPORTED). */
NTTB200_API int nttb200_rns_gs_batch(nttb200_rns_plan *plan, const int32_t *d_in, int32_t *d_out,
                                     size_t batch, void *cuda_stream);
NTTB200_API int nttb200_rns_ct_batch(nttb200_rns_plan *plan, const int32_t *d_in, int32_t *d_out,
                                     size_t batch, void *cuda_stream);
/* c = a (*) b mod (x^N + 1, q[l]) on every channel; fwd holds psi_l^bitrev tables,
 * inv psi_l^-bitrev tables of the same primes and the same N (else NTTB200_ERR_INVALID_ARG).
 * d_c may alias d_a or d_b.  At N = 4096 d_c needs 4-byte alignment only; at N > 4096 it
 * must be 16-byte aligned like the operands (else NTTB200_ERR_UNSUPPORTED, nothing written). */
NTTB200_API int nttb200_rns_polymul_negacyclic(nttb200_rns_plan *fwd, nttb200_rns_plan *inv,
                                               const int32_t *d_a, const int32_t *d_b, int32_t *d_c,
                                               size_t batch, void *cuda_stream);

/* ---- RNS evaluation-domain arithmetic (new) ------------------------------------
 * Operators on polynomials kept in the NTT domain, so that a whole computation runs as
 * nttb200_rns_ct_batch -> (pointwise / scale / dot)* -> nttb200_rns_gs_scaled_batch on one
 * plan, one launch per operation for all channels.  Shared rules:
 *   - data is [batch][L][N] on the plan's L primes and N; inputs canonical (in [0, q[l])),
 *     outputs canonical;
 *   - argument errors are returned before anything is launched: a null plan, a null pointer
 *     with batch > 0 or an option out of range -> NTTB200_ERR_INVALID_ARG; batch == 0 ->
 *     NTTB200_OK with nothing launched;
 *   - a disallowed overlap of the output with an input -> NTTB200_ERR_INVALID_ARG, a buffer that
 *     is not 16-byte aligned -> NTTB200_ERR_UNSUPPORTED; nothing is written in either case;
 *   - indexing is 64-bit: pointwise, scale and dot have no 2^31-word limit. */
#define NTTB200_RNS_ADD 0u
#define NTTB200_RNS_SUB 1u
#define NTTB200_RNS_MUL 2u
/* c[b][l] = a[b][l] op b'[l] mod q[l], elementwise (op: NTTB200_RNS_ADD / SUB / MUL, else
 * INVALID_ARG); b' = d_b[b] if b_batch == batch, d_b[0] (one [L][N] operand broadcast over the
 * batch) if b_batch == 1, another b_batch -> INVALID_ARG.  d_c may equal d_a, or d_b when
 * b_batch == batch; any other overlap -> INVALID_ARG. */
NTTB200_API int nttb200_rns_pointwise(nttb200_rns_plan *plan, uint32_t op, const int32_t *d_a,
                                      const int32_t *d_b, int32_t *d_c, size_t batch, size_t b_batch,
                                      void *cuda_stream);
/* c[b][l] = a[b][l] * scalars[l] mod q[l]; scalars: L words on the HOST, scalars[l] < q[l]
 * (a null scalars or a larger word -> INVALID_ARG, also for batch == 0).  In place (d_c == d_a)
 * allowed; any other overlap -> INVALID_ARG. */
NTTB200_API int nttb200_rns_scale(nttb200_rns_plan *plan, const int32_t *d_a, int32_t *d_c, size_t batch,
                                  const uint32_t *scalars, void *cuda_stream);
/* c[b][l] = (accumulate ? c[b][l] : 0) + sum_{k < terms} a[k][b][l] * w[k][b'][l] mod q[l]:
 * the inner product of key switching.  d_a: [terms][batch][L][N]; d_w: [terms][w_batch][L][N]
 * with w_batch == batch (b' = b) or w_batch == 1 (b' = 0: one key shared by the whole batch),
 * another w_batch -> INVALID_ARG; 1 <= terms <= 64 (else INVALID_ARG).  The products are summed
 * exactly in 64 bits and reduced every 16 terms.  d_c must not overlap d_a or d_w (INVALID_ARG). */
NTTB200_API int nttb200_rns_dot(nttb200_rns_plan *plan, const int32_t *d_a, const int32_t *d_w,
                                int32_t *d_c, uint32_t terms, size_t batch, size_t w_batch,
                                int accumulate, void *cuda_stream);
/* The GS network of nttb200_rns_gs_batch on every channel with every output multiplied by
 * N^-1 mod q[l]: the inverse NTT of a plan holding psi_l^-bitrev tables, in the same passes
 * (the scaling rides on the tile pass's store).  In place allowed.  An even q[l] (no N^-1) ->
 * NTTB200_ERR_MODULUS; batch * L * N / 4096 must stay below 2^31 (else UNSUPPORTED). */
NTTB200_API int nttb200_rns_gs_scaled_batch(nttb200_rns_plan *plan, const int32_t *d_in, int32_t *d_out,
                                            size_t batch, void *cuda_stream);

/* ---- RNS Galois automorphisms (new) --------------------------------------------
 * sigma_g : a(X) -> a(X^g) mod (X^N + 1) for odd g, the permutation under slot rotations
 * (g = 5^r mod 2N rotates CKKS slots by r) and conjugation (g = 2N - 1).
 *   NTTB200_AUTO_COEFF: coefficient domain.  With e = j * g^-1 mod 2N: out[j] = in[e] for
 *     e < N, (q[l] - in[e - N]) mod q[l] otherwise.
 *   NTTB200_AUTO_EVAL: evaluation domain, in the order nttb200_rns_ct_batch produces on a plan
 *     of psi_l^bitrev tables (index k holds a(psi^(2 brev(k) + 1)), brev over logn bits) and
 *     nttb200_rns_gs_scaled_batch consumes on psi_l^-bitrev tables: the permutation
 *     out[k] = in[brev((g * brev(k) + (g - 1) / 2) mod N)], the same for every channel and
 *     every choice of psi_l.  So rns_ct(sigma_coeff(x)) == sigma_eval(rns_ct(x)) bit for bit.
 * Rules of the evaluation-domain operators: inputs canonical, outputs canonical; galois: count
 * words on the HOST, every g odd with 1 <= g < 2N, 1 <= count <= 64; a null plan, a null
 * galois, a bad g or count or an unknown domain -> NTTB200_ERR_INVALID_ARG, also when
 * batch == 0; a null buffer with batch > 0 or an output that overlaps the input (in place
 * included: in the evaluation domain block t is written from another block) -> INVALID_ARG;
 * batch == 0 -> NTTB200_OK with nothing launched; a buffer that is not 16-byte aligned ->
 * NTTB200_ERR_UNSUPPORTED (nothing is written in either case); indexing is 64-bit, with no
 * 2^31-word limit; one launch per call.  Only N, L and the moduli are read from the plan, so
 * either plan of a forward / inverse pair will do. */
#define NTTB200_AUTO_COEFF 0u
#define NTTB200_AUTO_EVAL 1u
/* out[c][b][l] = sigma_{galois[c]}(in[b][l]) for c < count: X -> X^g on every channel of every
 * polynomial, in the coefficient domain or in the evaluation (rns_ct) order.  d_in [batch][L][N],
 * d_out [count][batch][L][N] (count outputs from one read of the input: hoisted rotations). */
NTTB200_API int nttb200_rns_automorphism(nttb200_rns_plan *plan, const int32_t *d_in, int32_t *d_out,
                                         size_t batch, const uint32_t *galois, uint32_t count,
                                         uint32_t domain, void *cuda_stream);

/* ---- RNS basis conversion (new) -------------------------------------------------
 * Moves coefficient-domain values from the primes of one plan to those of another: the step
 * under CKKS rescale, the BGV-style modulus drop and the ModUp / ModDown of hybrid key
 * switching.  A conversion object is built from a source plan `from` (S channels, moduli b_i,
 * product B) and a target plan `to` (T channels, moduli c_j, product C).
 * nttb200_rns_conv_create: both plans on the same device with the same logn, flags 0 (else, or
 * a null pointer, NTTB200_ERR_INVALID_ARG); the S + T moduli pairwise coprime (else
 * NTTB200_ERR_MODULUS; the moduli need not be prime).  These are checked before any device is
 * touched.  The object copies the moduli, N, the device and every constant it needs: the plans
 * may be destroyed after this call.
 * Shared rules of the two operations (those of the evaluation-domain operators): inputs
 * canonical, outputs canonical; a null conv, a null pointer with batch > 0, an unknown flag or
 * a bad stride -> NTTB200_ERR_INVALID_ARG; batch == 0 -> NTTB200_OK with nothing launched; a
 * disallowed overlap of output and input -> NTTB200_ERR_INVALID_ARG; a buffer that is not
 * 16-byte aligned -> NTTB200_ERR_UNSUPPORTED (nothing is written in either case); indexing is
 * 64-bit, with no 2^31-word limit. */
typedef struct nttb200_rns_conv nttb200_rns_conv;
NTTB200_API int nttb200_rns_conv_create(nttb200_rns_conv **conv, const nttb200_rns_plan *from,
                                        const nttb200_rns_plan *to, uint32_t flags);
NTTB200_API int nttb200_rns_conv_destroy(nttb200_rns_conv *conv);

/* Fast (approximate) base conversion, coefficient domain, for ModUp:
 *   out[b][j] = sum_i [in[b][i] * (B/b_i)^-1]_{b_i} * (B/b_i)  mod c_j.
 * Contract: with x in [0, B) the CRT value of the S input residues and y_i the bracket above,
 * sum_i y_i * (B/b_i) = x + alpha*B with 0 <= alpha < S, and out[b][j] is that sum mod c_j
 * (exact, alpha = 0, when S = 1).  in_stride / out_stride: words between consecutive
 * polynomials; 0 means dense (S*N, T*N), otherwise a multiple of N and at least S*N (T*N), else
 * INVALID_ARG.  So a digit (a channel range of a [batch][L][N] ciphertext) can be read, and the
 * result written into the P channels of a [batch][L+K][N] buffer, without copies.  The output
 * must not share a word with any input row (INVALID_ARG): with equal strides the views are
 * compared row by row, so the P channels of the buffer whose Q channels are read may be
 * written; with different strides the whole extents must be disjoint. */
NTTB200_API int nttb200_rns_base_convert(nttb200_rns_conv *conv, const int32_t *d_in, size_t in_stride,
                                         int32_t *d_out, size_t out_stride, size_t batch,
                                         void *cuda_stream);

/* Division by B with the source channels dropped, for rescale / modulus drop and ModDown.
 * d_in: [batch][T+S][N], the T target channels first, then the S source channels;
 * d_out: [batch][T][N]:
 *   out[b][j] = ((x_C,j + h_C,j) - sum_i y'_i * (B/b_i)) * B^-1  mod c_j,
 *   y'_i = (x_B,i + h_B,i) * (B/b_i)^-1  mod b_i,
 * h = floor(B/2) with NTTB200_RNS_ROUND, h = 0 without (other flags -> INVALID_ARG).
 * Contract: with X in [0, C*B) the CRT value of all T + S input channels and X' = (X + h) mod CB,
 * out = (floor(X'/B) - alpha) mod c_j with alpha in [0, S) the overshoot of converting X' mod B.
 * With S = 1, alpha = 0 and the result is exact: floor((X + floor(B/2))/B) = round(X/B) for
 * X < CB - floor(B/2) with ROUND, floor(X/B) without.  from = {q_L-1}, to = {q_0..q_L-2}: the
 * natural [batch][L][N] ciphertext is the input (CKKS rescale); from = P, to = Q: ModDown of a
 * [batch][L+K][N] key-switching result.  The output must not overlap the input (INVALID_ARG;
 * in place is not possible: at batch > 1 output row b lands on input row b-1's source channels). */
#define NTTB200_RNS_ROUND 1u
NTTB200_API int nttb200_rns_mod_down(nttb200_rns_conv *conv, const int32_t *d_in, int32_t *d_out,
                                     size_t batch, uint32_t flags, void *cuda_stream);

/* Exact forms, for BFV multiplication and decryption (Halevi-Polyakov-Shoup): the overshoot
 * of the fast conversion is removed with v = round(sum_i y_i / b_i), computed in FP64 in the
 * same pass.  Exactness: for S <= 32 and moduli <= 2^30 the FP64 sum is within 2^-43 of
 * sum_i y_i / b_i (DESIGN 3.6), so both results are exact unless the fractional part of x / B
 * (of t X / B for scale_round) lies within eps = 2^-40 of 1/2.  In that band either neighbour
 * may be returned: x_c +- B for the conversion, the result +- 1 for scale_round.  Uniform
 * random x meets the band with probability 2^-39; values that must be exact (BFV) stay far from
 * it by the parameter choice. */

/* Exact base conversion of the centred value: out[b][j] = x_c mod c_j, where x_c == x (mod B)
 * and -B/2 < x_c <= B/2.  Arguments, strides and rules as nttb200_rns_base_convert. */
NTTB200_API int nttb200_rns_base_convert_exact(nttb200_rns_conv *conv, const int32_t *d_in,
                                               size_t in_stride, int32_t *d_out, size_t out_stride,
                                               size_t batch, void *cuda_stream);

/* Scale by t / B and round, with the source channels dropped.  d_in [batch][T+S][N], target
 * channels first (the nttb200_rns_mod_down layout); d_out [batch][T][N]:
 *   out[b][j] = round(t * X / B) mod c_j,
 * X the CRT value of all T + S channels.  Valid for every representative of X mod C*B, so a
 * centred X is covered too.  1 <= t < 2^32: t == 0 -> NTTB200_ERR_INVALID_ARG, also when
 * batch == 0.  With t = 1 and S = 1 the result equals nttb200_rns_mod_down(ROUND) bit for bit;
 * with t = 1 and S > 1 it is the exact rounded division by B (rescale by several primes at
 * once).  Layout and no-overlap rule as nttb200_rns_mod_down. */
NTTB200_API int nttb200_rns_scale_round(nttb200_rns_conv *conv, const int32_t *d_in, int32_t *d_out,
                                        size_t batch, uint32_t t, void *cuda_stream);

/* ---- CKKS slot encoding (new) ----------------------------------------------------
 * The canonical embedding of the ring Z[X]/(X^N + 1) into n = N/2 complex slots, computed as an
 * FP64 negacyclic FFT on the device.  With zeta = e^(i pi / N), slot j holds m(zeta^(5^j mod 2N)):
 * for real coefficients x_k (k < N), s_j = (5^j mod 2N - 1) / 4 (a permutation of 0..n-1),
 *   decode: y_k = (x_k + i x_(k+n)) zeta^k (k < n),  Y_s = sum_k y_k e^(+2 pi i s k / n),
 *           z_j = Y_(s_j) / scale;
 *   encode: v_(s_j) = z_j,  y_k = (1/n) sum_s v_s e^(-2 pi i s k / n),
 *           m_k + i m_(k+n) = y_k zeta^-k,  a_k = rint(scale * m_k) (half to even).
 * With this order nttb200_rns_automorphism by galois = 5^r mod 2N takes the slots z to z rotated
 * left by r (slot j receives z_(j+r)), and by 2N - 1 to conj(z), in both domains.
 * An encoder is built from an RNS plan as a conversion object is: it copies N, the device and the
 * moduli, so the plan may be destroyed afterwards.  It owns device tables: the FFT twiddles
 * e^(2 pi i t / n) and zeta^k, each built once in FP64 within 1 ulp, and the permutation s_j.
 * A null pointer or flags != 0 -> NTTB200_ERR_INVALID_ARG.
 * Shared rules of encode and decode: a null encoder, a null pointer with batch > 0 or a scale
 * that is not finite and > 0 -> NTTB200_ERR_INVALID_ARG, also when batch == 0; batch == 0 ->
 * NTTB200_OK with nothing launched; overlapping input and output -> NTTB200_ERR_INVALID_ARG; a
 * buffer that is not 16-byte aligned -> NTTB200_ERR_UNSUPPORTED (nothing is written in either
 * case); argument errors are returned before any device is touched; indexing is 64-bit.  One
 * launch per call for N <= 2^14, two above (the transform is split into a column pass and a
 * row pass through stream-ordered scratch of 16 n bytes per polynomial). */
typedef struct nttb200_ckks_encoder nttb200_ckks_encoder;
NTTB200_API int nttb200_ckks_encoder_create(nttb200_ckks_encoder **enc, const nttb200_rns_plan *plan,
                                            uint32_t flags);
NTTB200_API int nttb200_ckks_encoder_destroy(nttb200_ckks_encoder *enc);

/* d_slots: complex128 [batch][n], interleaved (re, im) doubles; d_out: int32 [batch][L][N], the
 * residues a_k mod q_l of every channel, coefficient domain (nttb200_rns_ct_batch takes them from
 * there).  The residues are exact for every finite scale * m_k, also beyond 2^64 (a = M 2^e with
 * M < 2^53 is reduced as (M mod q)(2^e mod q)).  A value that is not finite gives unspecified
 * residues and no fault.  The FFT error is bounded in DESIGN 3.6. */
NTTB200_API int nttb200_ckks_encode(nttb200_ckks_encoder *enc, const void *d_slots, double scale,
                                    int32_t *d_out, size_t batch, void *cuda_stream);

/* Reads the first `channels` rows (moduli b_0..b_(C-1), product B) of each polynomial at
 * d_in + b * in_stride (0: dense channels * N; else a multiple of N and at least channels * N,
 * the nttb200_rns_base_convert rule) and writes d_slots [batch][n] complex128.  1 <= channels <=
 * min(L, 4), else NTTB200_ERR_INVALID_ARG; the first `channels` moduli not pairwise coprime ->
 * NTTB200_ERR_MODULUS.  The centred value x_c in (-B/2, B/2] is exact (128-bit CRT) and enters
 * the FFT as a double with relative error at most 2^-53.  A message with |x| < B'/2 decodes from
 * any prefix of channels whose product is B': a level-L ciphertext needs no mod_down first. */
NTTB200_API int nttb200_ckks_decode(nttb200_ckks_encoder *enc, const int32_t *d_in, size_t in_stride,
                                    uint32_t channels, double scale, void *d_slots, size_t batch,
                                    void *cuda_stream);

/* ---- Packed integer slots for BFV and BGV (new) -----------------------------------
 * N integer slots mod t, t a prime with t == 1 (mod 2N) and t < 2^30.  psi is the smallest
 * primitive 2N-th root of unity mod t (the least of the N roots psi_0^(2i+1)).  The slots form
 * a 2 x N/2 matrix: slot i = r N/2 + j holds m(psi^e_i) mod t, with e_i = 5^j mod 2N in row
 * r = 0 and e_i = 2N - (5^j mod 2N) in row r = 1.  With this order nttb200_rns_automorphism by
 * galois = 5^s mod 2N rotates both rows left by s (slot j receives slot j + s, as for CKKS), and
 * by 2N - 1 swaps the rows, in both domains.  In the rns_ct order of a one-channel plan of
 * modulus t on psi^bitrev tables, slot i sits at index k_i = brev((e_i - 1) / 2), brev over
 * logn bits.
 * Encode writes the plaintext m (coefficients in [0, t)) on the L channels of the plan, in one
 * of two forms; Q is the product of the channel moduli q_l, r = Q mod t:
 *   NTTB200_PACK_SCALED   round(Q m / t) mod q_l, the BFV message term.  Computed as
 *                         (Delta_l m + rho) mod q_l with Delta_l = floor(Q / t) mod q_l
 *                         = -r t^-1 mod q_l and rho = floor((2 r m + t) / 2t) = round(r m / t)
 *                         (t odd: never a tie); no big integers.
 *   NTTB200_PACK_CENTRED  m_c mod q_l with m_c == m (mod t) in (-t/2, t/2]: the BGV plaintext
 *                         and the BFV plaintext operand of a plaintext x ciphertext product.
 * nttb200_packed_encoder_create: copies N, the device and the moduli of `plan` (which may be
 * destroyed afterwards), finds psi on the host and owns two one-channel RNS plans of modulus t
 * (psi^bitrev and psi^-bitrev tables), the slot table k_i and its inverse.  A null pointer or
 * flags != 0 -> NTTB200_ERR_INVALID_ARG; t not prime, t != 1 (mod 2N), t >= 2^30 or t dividing
 * some q_l -> NTTB200_ERR_MODULUS; both before any device is touched.
 * Shared rules of encode and decode: a null encoder or an unknown mode / flag ->
 * NTTB200_ERR_INVALID_ARG, also when batch == 0; a null buffer with batch > 0 or overlapping
 * input and output -> NTTB200_ERR_INVALID_ARG; batch == 0 -> NTTB200_OK with nothing launched; a
 * buffer that is not 16-byte aligned -> NTTB200_ERR_UNSUPPORTED (nothing is written in either
 * case); indexing is 64-bit, and batch * N / 4096 must stay below 2^31 (the transforms mod t; else
 * NTTB200_ERR_UNSUPPORTED).  The data passes through stream-ordered scratch of 4N bytes per
 * polynomial.  Launches per call: encode 3 at N = 4096 and 4 above (gather, the inverse
 * transform mod t, the lift); decode 2 and 3 (the forward transform mod t, gather). */
#define NTTB200_PACK_SCALED 0u
#define NTTB200_PACK_CENTRED 1u
typedef struct nttb200_packed_encoder nttb200_packed_encoder;
NTTB200_API int nttb200_packed_encoder_create(nttb200_packed_encoder **enc, const nttb200_rns_plan *plan,
                                              uint32_t t, uint32_t flags);
NTTB200_API int nttb200_packed_encoder_destroy(nttb200_packed_encoder *enc);

/* d_slots: int32 [batch][N], each word read as a signed integer and reduced mod t (negative
 * values encode directly); d_out: int32 [batch][L][N], coefficient domain.  mode:
 * NTTB200_PACK_SCALED or NTTB200_PACK_CENTRED. */
NTTB200_API int nttb200_packed_encode(nttb200_packed_encoder *enc, const int32_t *d_slots, uint32_t mode,
                                      int32_t *d_out, size_t batch, void *cuda_stream);

/* d_in: int32 [batch][N], canonical residues mod t in the coefficient domain (what the BFV
 * decryption rns_scale -> convert_exact -> rns_scale on a t plan, or the BGV decryption
 * convert_exact from Q to {t}, produces); d_slots: int32 [batch][N], in [0, t) with flags 0, in
 * (-t/2, t/2] with NTTB200_PACK_CENTRED. */
NTTB200_API int nttb200_packed_decode(nttb200_packed_encoder *enc, const int32_t *d_in, uint32_t flags,
                                      int32_t *d_slots, size_t batch, void *cuda_stream);

/* ---- Hybrid key switching (new) -------------------------------------------------
 * Relinearisation and the second half of a rotation in one call, with the gadget of hybrid key
 * switching (digits of alpha primes, special primes P).
 * nttb200_rns_keyswitch_create: qp_fwd / qp_inv are one forward / inverse pair (psi_l^bitrev and
 * psi_l^-bitrev tables) over L + K channels in the order [Q | P]: Q is the first q_limbs = L
 * channels and P the remaining K >= 1, so the result lands directly in the nttb200_rns_mod_down
 * layout.  Digit i covers the channels [i alpha, min((i + 1) alpha, L)), dnum = ceil(L / alpha)
 * digits (the last one may be shorter); D_i is the product of its primes.  The object copies N,
 * the device, the moduli and the tables (it builds its own forward / inverse plans on Q and on
 * Q P, and the conversion constants of ModUp and ModDown): the plans may be destroyed afterwards.
 * A null pointer, flags != 0, plans with different N or device or channel count, q_limbs == 0,
 * q_limbs >= the channel count (no P channel), alpha == 0 or alpha > L, or channel moduli that
 * differ between the two plans -> NTTB200_ERR_INVALID_ARG; moduli that are not pairwise coprime
 * or an even modulus (no N^-1) -> NTTB200_ERR_MODULUS; all before any device is touched.
 *
 * nttb200_rns_keyswitch_apply: d_in holds x, [batch][L][N] on Q, polynomial b at d_in + b * in_stride
 * (0: dense L * N; else a multiple of N and at least L * N, the nttb200_rns_base_convert rule: the
 * c1 of a [batch][2][L][N] ciphertext batch is d_in = ct + L * N with in_stride 2 L N).
 * d_keys: [count][dnum][2][L + K][N], in the evaluation (rns_ct) order on Q P, caller-owned.
 * Element c, digit i holds (b_i, a_i) with
 *     b_i + a_i s == e_i + P (Q / D_i) [(Q / D_i)^-1]_{D_i} s'   (mod Q P),
 * s' = sigma_g(s) for the rotation key of g = galois[c], s^2 for the relinearisation key (g = 1).
 * For every c < count (1 <= count <= 64; every g odd in [1, 2N); g = 1 allowed):
 *     d_out[c][b] = (u0, u1) = ModDown_P( sum_i sigma_g(ModUp(x)_i) * (b_i, a_i) ),
 * d_out [count][batch][2][L][N], ModDown the rounding division of nttb200_rns_mod_down(ROUND).
 * Then u0 + u1 s ~ sigma_g(x) s' within the usual hybrid key-switching noise: a rotation adds
 * sigma_g(c0) to u0 and keeps u1, relinearisation adds (u0, u1) to (d0, d1).  The result is bit
 * for bit the one of rns_gs_scaled on Q, ModUp of every digit by nttb200_rns_base_convert (own
 * rows copied), rns_ct on Q P, nttb200_rns_automorphism(EVAL), nttb200_rns_dot for b and for a,
 * rns_gs_scaled on Q P, nttb200_rns_mod_down(ROUND), rns_ct on Q.
 * NTTB200_KS_COEFF_IN: d_in holds coefficients (the first transform is skipped);
 * NTTB200_KS_COEFF_OUT: d_out is left in coefficients (the last transform is skipped).
 * Rules of the evaluation-domain operators: a null ks, a null galois, a bad g or count or an
 * unknown flag -> NTTB200_ERR_INVALID_ARG, also when batch == 0; a null buffer with batch > 0, a
 * bad stride, or d_out overlapping d_in or d_keys -> INVALID_ARG; batch == 0 -> NTTB200_OK with
 * nothing launched; a buffer that is not 16-byte aligned -> NTTB200_ERR_UNSUPPORTED (nothing is
 * written in either case); indexing is 64-bit; max(2 count, dnum) * batch * (L + K) * N / 4096
 * must stay below 2^31 (the transforms; else UNSUPPORTED).  Stream-ordered scratch: the digits,
 * dnum * batch * (L + K) * N words, and the products, 2 * count * batch * (L + K) * N words.
 * Launches per call: 2 dnum + 5 at N = 4096 and 2 dnum + 9 above, one (two) fewer for each
 * transform skipped by a flag. */
#define NTTB200_KS_COEFF_IN 1u    /* d_in holds coefficients (else the rns_ct order)        */
#define NTTB200_KS_COEFF_OUT 2u   /* leave the output in coefficients (else the rns_ct order) */
typedef struct nttb200_rns_keyswitch nttb200_rns_keyswitch;
NTTB200_API int nttb200_rns_keyswitch_create(nttb200_rns_keyswitch **ks, const nttb200_rns_plan *qp_fwd,
                                             const nttb200_rns_plan *qp_inv, uint32_t q_limbs, uint32_t alpha,
                                             uint32_t flags);
NTTB200_API int nttb200_rns_keyswitch_destroy(nttb200_rns_keyswitch *ks);
NTTB200_API int nttb200_rns_keyswitch_apply(nttb200_rns_keyswitch *ks, const int32_t *d_in, size_t in_stride,
                                      const int32_t *d_keys, const uint32_t *galois, uint32_t count,
                                      int32_t *d_out, size_t batch, uint32_t flags, void *cuda_stream);

/* ---- Plaintext matrix-vector products (new) -------------------------------------
 * y = M z on the slots of every ciphertext of a batch, M given by its generalised diagonals:
 *     y[s] = sum_{k in offsets} d_k[s] * z[(s + k) mod n],   n = N/2,
 * over the n complex CKKS slots, or over each of the two rows of packed BFV / BGV slots (each row
 * its own n x n matrix).  Rotation by r is galois_rotation(N, r) = 5^r mod 2N.  Baby-step
 * giant-step schedule: k = n1 i + j with 0 <= j < n1,
 *     W_i = sum_j sigma_{-n1 i}(pt_{n1 i + j}) (.) rot_j(ct),   y = W_0 + sum_{i >= 1} rot_{n1 i}(W_i);
 * the babies rot_j (j >= 1) come from one hoisted key switch of c1 (rot_0 = ct), each giant is a
 * key switch of W_i.c1, and only the babies and giants that occur are computed.
 *
 * nttb200_rns_lintrans_keys: the Galois elements whose keys the call needs, in the order it reads
 * them: the babies j >= 1 that occur in ascending order (5^j mod 2N), then the giants i >= 1 that
 * occur in ascending order (5^(n1 i) mod 2N).  *nkeys receives their number; galois_out, when not
 * null, receives the elements (room for *nkeys: ask with galois_out = null first).  Host only.
 * A null offsets or nkeys, count == 0, n1 outside [1, 64], logn outside [12, 16], an offset >= N/2
 * or a duplicated one -> NTTB200_ERR_INVALID_ARG.
 *
 * nttb200_rns_lintrans_apply: ks a key switcher with L = q_limbs.  d_ct [batch][2][L][N] in the
 * rns_ct order on Q.  d_diags [count][L][N]: d_k encoded (CKKS scale Delta_pt, or packed), in the
 * rns_ct order, in the order of offsets, not rotated (sigma_{-n1 i} is applied inside); one matrix
 * for the whole batch.  d_keys [nkeys][dnum][2][L + K][N] in the order of nttb200_rns_lintrans_keys,
 * each key in the format of nttb200_rns_keyswitch_apply.  d_out [batch][2][L][N] in the rns_ct
 * order, not rescaled (CKKS scale Delta Delta_pt).  The result is bit for bit the one of the
 * composed calls: nttb200_rns_keyswitch_apply hoisted over the babies, nttb200_rns_automorphism(EVAL)
 * of c0 plus rns_pointwise ADD, automorphism(EVAL) of each diagonal by sigma_{-n1 i},
 * rns_pointwise MUL / ADD per term, one nttb200_rns_keyswitch_apply per giant, automorphism of
 * W_i.c0 and the adds.  The offsets are read before the call returns.
 * A null ks, the errors of nttb200_rns_lintrans_keys, or nkeys different from its count ->
 * NTTB200_ERR_INVALID_ARG, also when batch == 0; a null buffer with batch > 0 (d_keys may be null
 * when nkeys == 0), or d_out overlapping d_ct, d_diags or d_keys (no in-place form) -> INVALID_ARG;
 * batch == 0 -> NTTB200_OK with nothing launched; a buffer that is not 16-byte aligned ->
 * NTTB200_ERR_UNSUPPORTED (nothing is written in either case); indexing is 64-bit; the transforms
 * of a key-switch pass must stay below 2^31 tiles (else UNSUPPORTED), as in
 * nttb200_rns_keyswitch_apply.  With nb babies, ng giants >= 1 and nw giants (0 included):
 * stream-ordered scratch of (nb + nw + ng) * batch * 2 * L * N words (nb + ng when the only giant is
 * 0) plus 16 * (2 nw + count + 1) bytes of schedule, and per key-switch pass of c elements the
 * scratch of nttb200_rns_keyswitch_apply with c * batch inputs for the giants.
 * Launches per call, with P = 2 dnum + 5 at N = 4096 and 2 dnum + 9 above:
 *     [nb > 0] P + 1 + [ng > 0] (ceil(ng / 64) P + 1);   one offset 0 alone is one launch. */
NTTB200_API int nttb200_rns_lintrans_keys(uint32_t logn, const uint32_t *offsets, uint32_t count, uint32_t n1,
                                          uint32_t *galois_out, uint32_t *nkeys);
NTTB200_API int nttb200_rns_lintrans_apply(nttb200_rns_keyswitch *ks, const int32_t *d_ct, const int32_t *d_diags,
                                           const uint32_t *offsets, uint32_t count, uint32_t n1,
                                           const int32_t *d_keys, uint32_t nkeys, int32_t *d_out, size_t batch,
                                           void *cuda_stream);

/* ---- introspection ---------------------------------------------------------- */
NTTB200_API const char *nttb200_strerror(int status);
/* text of the last CUDA error seen by the calling thread ("" if none) */
NTTB200_API const char *nttb200_last_error(void);
/* how many kernels this library has launched since load (all plans, all threads) */
NTTB200_API uint64_t nttb200_kernel_launches(void);
/* name of the kernel path the last nttb200_gs_batch/ct_batch on this plan took */
NTTB200_API const char *nttb200_plan_last_path(const nttb200_plan *plan);
NTTB200_API uint32_t nttb200_plan_logn(const nttb200_plan *plan);
NTTB200_API uint32_t nttb200_plan_modulus(const nttb200_plan *plan);
NTTB200_API const char *nttb200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* NTTB200_H */
