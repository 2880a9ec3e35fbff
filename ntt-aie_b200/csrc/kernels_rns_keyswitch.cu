// kernels_rns_keyswitch.cu -- hybrid key switching on RNS batches: the key inner product fused with
// the evaluation-domain Galois permutation, and the call pipeline around it.
//
//   rns_ks_dot_kernel<G>  U[c][b][p][l] = sum_{i < dnum} sigma_{g_c}(D[i][b][l]) * K[c][i][p][l]  mod q_l
//                         for both key parts p (b, a), every element c of the call and every
//                         channel l of Q P, in the rns_ct order.  D: [dnum][batch][L+K][N] digits,
//                         K: [count][dnum][2][L+K][N] keys, U: [count][batch][2][L+K][N].
//     Work item = one 4096-word output block t of one channel row, for one element c and a group
//     of G polynomials of the batch.  The evaluation-domain permutation of rns_auto_eval_kernel
//     maps output block t to the single source block brev_s((g brev_s(t) + (g-1)/2) mod 2^s),
//     s = logn - 12, so each digit's source block is staged in 16 KiB of shared memory (128-bit
//     loads, the next digit's block in flight in registers while this one is gathered) and the
//     words are gathered from there.  g = 1 is a uniform branch that reads the digits directly.
//     The key words are read once per item with 128-bit loads and serve the G polynomials.  Both
//     key parts accumulate exactly in 64 bits and are folded every 16 digits, the rns_dot bound
//     q + 16 (q-1)^2 < 2^64 for q <= 2^30; one store each for U_b and U_a.  The element index is
//     the fastest-moving part of the item index, so the digit rows under way stay L2-resident
//     while the count elements gather from them.
//     Paired (P): D is [dnum][count][batch][L+K][N] and element c reads only its own polynomials
//     c * batch + b, so one pass switches count different inputs, each under its own element
//     (the giant steps of nttb200_rns_lintrans_apply).  A group of G stays inside one element.
// Every pointer is 16-byte aligned (checked by the host), every index 64-bit.
#include <algorithm>
#include <vector>

#include "modarith.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kK_Threads = 512;
constexpr int kK_BlockVecs = 1024;                          // uint4 of one 4096-word block
constexpr int kK_Vecs = kK_BlockVecs / kK_Threads;          // uint4 per thread
constexpr int kK_GroupOwn = 2;                              // G for batch > 1 (ptxas: no spills)

// items = groups * rows * 2^(logn - 12) * count
template <int G, bool P = false>
__global__ void __launch_bounds__(kK_Threads)
rns_ks_dot_kernel(const uint4 *d, const uint4 *key, uint4 *u, uint64_t batch, uint32_t rows, uint32_t logn,
                  uint32_t dnum, uint32_t count, uint64_t items, const __grid_constant__ RnsKsConsts k) {
    __shared__ uint4 s4[G][kK_BlockVecs];
    const uint32_t log_b = logn - 12, bmask = (1u << log_b) - 1, nmask = (1u << logn) - 1;
    const uint64_t row_vecs = (uint64_t) 1 << (logn - 2);
    const uint64_t poly_vecs = row_vecs * rows, digit_vecs = poly_vecs * batch * (P ? count : 1);
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint32_t c = (uint32_t) (it % count);
        const uint64_t rest = it / count;
        const uint32_t t = (uint32_t) rest & bmask;
        const uint32_t l = (uint32_t) ((rest >> log_b) % rows);
        const uint64_t b0 = (rest >> log_b) / rows * G;
        const int gn = batch - b0 < (uint64_t) G ? (int) (batch - b0) : G;   // uniform: ragged last group
        const uint32_t q = k.q[l], g = k.g[c], off = k.off[c];
        const uint64_t mu = k.mu[l];
        const bool ident = g == 1;   // uniform across the block
        const uint32_t src_t = log_b ? __brev((g * (__brev(t) >> (32 - log_b)) + off) & bmask) >> (32 - log_b) : 0;
        const uint64_t blk = l * row_vecs + ((uint64_t) t << 10) + threadIdx.x;
        const uint64_t sblk = l * row_vecs + ((uint64_t) (ident ? t : src_t) << 10) + threadIdx.x;
        uint64_t pb[G];   // polynomial offsets; the last one of a ragged group stands in for the missing ones
#pragma unroll
        for (int p = 0; p < G; p++) pb[p] = ((P ? (uint64_t) c * batch : 0) + b0 + (p < gn ? p : gn - 1)) * poly_vecs;
        uint32_t idx[kK_Vecs][4];   // source word of every output word, inside the staged block
#pragma unroll
        for (int j = 0; j < kK_Vecs; j++) {
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const uint32_t k0 = (t << 12) + (threadIdx.x + j * kK_Threads) * 4 + e;
                idx[j][e] = brev_n((g * brev_n(k0, logn) + off) & nmask, logn) & (kK_BlockVecs * 4 - 1);
            }
        }
        uint64_t acc[G][2][kK_Vecs][4];
#pragma unroll
        for (int p = 0; p < G; p++) {
#pragma unroll
            for (int j = 0; j < kK_Vecs; j++) {
#pragma unroll
                for (int e = 0; e < 4; e++) acc[p][0][j][e] = acc[p][1][j][e] = 0;
            }
        }
        uint4 nxt[G][kK_Vecs];
#pragma unroll
        for (int p = 0; p < G; p++) {
#pragma unroll
            for (int j = 0; j < kK_Vecs; j++) nxt[p][j] = __ldg(d + pb[p] + sblk + j * kK_Threads);
        }
        for (uint32_t i = 0; i < dnum; i++) {
            uint32_t x[G][kK_Vecs][4];
            if (ident) {
#pragma unroll
                for (int p = 0; p < G; p++) {
#pragma unroll
                    for (int j = 0; j < kK_Vecs; j++) {
                        const uint4 v = nxt[p][j];
                        x[p][j][0] = v.x, x[p][j][1] = v.y, x[p][j][2] = v.z, x[p][j][3] = v.w;
                    }
                }
            } else {
                __syncthreads();   // the previous digit's gathers are done
#pragma unroll
                for (int p = 0; p < G; p++) {
#pragma unroll
                    for (int j = 0; j < kK_Vecs; j++) s4[p][threadIdx.x + j * kK_Threads] = nxt[p][j];
                }
                __syncthreads();
            }
            if (i + 1 < dnum) {
#pragma unroll
                for (int p = 0; p < G; p++) {
#pragma unroll
                    for (int j = 0; j < kK_Vecs; j++) {
                        nxt[p][j] = __ldg(d + (i + 1) * digit_vecs + pb[p] + sblk + j * kK_Threads);
                    }
                }
            }
            if (!ident) {
#pragma unroll
                for (int p = 0; p < G; p++) {
                    const uint32_t *s = reinterpret_cast<const uint32_t *>(s4[p]);
#pragma unroll
                    for (int j = 0; j < kK_Vecs; j++) {
#pragma unroll
                        for (int e = 0; e < 4; e++) x[p][j][e] = s[idx[j][e]];
                    }
                }
            }
            const uint4 *kc = key + ((uint64_t) c * dnum + i) * 2 * poly_vecs + blk;
#pragma unroll
            for (int j = 0; j < kK_Vecs; j++) {
                const uint4 kb = __ldg(kc + j * kK_Threads), ka = __ldg(kc + poly_vecs + j * kK_Threads);
                const uint32_t wb[4] = {kb.x, kb.y, kb.z, kb.w}, wa[4] = {ka.x, ka.y, ka.z, ka.w};
#pragma unroll
                for (int p = 0; p < G; p++) {
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        acc[p][0][j][e] += (uint64_t) x[p][j][e] * wb[e];
                        acc[p][1][j][e] += (uint64_t) x[p][j][e] * wa[e];
                    }
                }
            }
            if ((i & 15) == 15 || i + 1 == dnum) {   // fold: every accumulator back below q
#pragma unroll
                for (int p = 0; p < G; p++) {
#pragma unroll
                    for (int j = 0; j < kK_Vecs; j++) {
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            acc[p][0][j][e] = reduce64(acc[p][0][j][e], q, mu);
                            acc[p][1][j][e] = reduce64(acc[p][1][j][e], q, mu);
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int p = 0; p < G; p++) {
            if (p < gn) {
                uint4 *up = u + ((uint64_t) c * batch + b0 + p) * 2 * poly_vecs + blk;
#pragma unroll
                for (int j = 0; j < kK_Vecs; j++) {
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const uint64_t *a = acc[p][h][j];
                        __stcs(up + h * poly_vecs + j * kK_Threads,
                               make_uint4((uint32_t) a[0], (uint32_t) a[1], (uint32_t) a[2], (uint32_t) a[3]));
                    }
                }
            }
        }
    }
}

template <int G, bool P>
static int ks_dot_launch(const nttb200_rns_keyswitch *ks, const int32_t *digits, const int32_t *keys, int32_t *u,
                         size_t batch, uint32_t count, const RnsKsConsts &k, cudaStream_t st) {
    int per = 0;
    NTTB200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, rns_ks_dot_kernel<G, P>, kK_Threads, 0));
    const uint64_t items = ((((uint64_t) batch + G - 1) / G * ks->limbs) << (ks->logn - 12)) * count;
    const uint64_t cap = (uint64_t) ks->sm_count * (per > 0 ? per : 1);
    rns_ks_dot_kernel<G, P><<<(unsigned) (items < cap ? items : cap), kK_Threads, 0, st>>>(
        reinterpret_cast<const uint4 *>(digits), reinterpret_cast<const uint4 *>(keys), reinterpret_cast<uint4 *>(u),
        batch, ks->limbs, ks->logn, ks->dnum, count, items, k);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

static int ks_dot(const nttb200_rns_keyswitch *ks, const int32_t *digits, const int32_t *keys, int32_t *u,
                  size_t batch, const uint32_t *galois, uint32_t count, bool paired, cudaStream_t st) {
    RnsKsConsts k{};
    const uint32_t nmask = (1u << ks->logn) - 1;
    for (uint32_t c = 0; c < count; c++) {
        k.g[c] = galois[c];
        k.off[c] = ((galois[c] - 1) / 2) & nmask;
    }
    for (uint32_t l = 0; l < ks->limbs; l++) {
        k.q[l] = ks->qp_fwd->pos[l].x;
        k.mu[l] = (uint64_t) ((((unsigned __int128) 1) << 64) / k.q[l]);
    }
    if (paired) {
        return batch == 1 ? ks_dot_launch<1, true>(ks, digits, keys, u, batch, count, k, st)
                          : ks_dot_launch<kK_GroupOwn, true>(ks, digits, keys, u, batch, count, k, st);
    }
    return batch == 1 ? ks_dot_launch<1, false>(ks, digits, keys, u, batch, count, k, st)
                      : ks_dot_launch<kK_GroupOwn, false>(ks, digits, keys, u, batch, count, k, st);
}

// ---------------------------------------------------------------------------- host side
static int conv_init(nttb200_rns_conv *cv, const nttb200_rns_keyswitch *ks, const uint32_t *q, uint32_t s0,
                     uint32_t s1, uint32_t t0, uint32_t t1) {
    cv->device = ks->device;
    cv->logn = ks->logn;
    cv->src = s1 - s0;
    cv->dst = t1 - t0;
    cv->sm_count = ks->sm_count;
    return rns_conv_prepare(cv, q + s0, q + t0);
}

int keyswitch_prepare(nttb200_rns_keyswitch *ks, const nttb200_rns_plan *qp_fwd, const nttb200_rns_plan *qp_inv) {
    const uint32_t L = ks->q_limbs, LK = ks->limbs, n = 1u << ks->logn;
    std::vector<uint32_t> q(LK);
    for (uint32_t l = 0; l < LK; l++) q[l] = qp_fwd->pos[l].x;
    // own plans from the tables of the given ones: [L + K][N] host words each
    std::vector<int32_t> tf((size_t) LK * n), ti((size_t) LK * n);
    std::vector<const int32_t *> pf(LK), pi(LK);
    for (uint32_t l = 0; l < LK; l++) {
        pf[l] = tf.data() + (size_t) l * n;
        pi[l] = ti.data() + (size_t) l * n;
        int rc = nttb200_plan_table(qp_fwd->sub[l], tf.data() + (size_t) l * n);
        if (rc == NTTB200_OK) rc = nttb200_plan_table(qp_inv->sub[l], ti.data() + (size_t) l * n);
        if (rc != NTTB200_OK) return rc;
    }
    int rc = nttb200_rns_plan_create_logn(&ks->qp_fwd, ks->device, ks->logn, LK, q.data(), pf.data(), 0);
    if (rc == NTTB200_OK) rc = nttb200_rns_plan_create_logn(&ks->qp_inv, ks->device, ks->logn, LK, q.data(), pi.data(), 0);
    if (rc == NTTB200_OK) rc = nttb200_rns_plan_create_logn(&ks->q_fwd, ks->device, ks->logn, L, q.data(), pf.data(), 0);
    if (rc == NTTB200_OK) rc = nttb200_rns_plan_create_logn(&ks->q_inv, ks->device, ks->logn, L, q.data(), pi.data(), 0);
    if (rc != NTTB200_OK) return rc;
    ks->sm_count = ks->qp_fwd->sm_count;
    // ModUp: digit i into [0, i alpha) (i >= 1) and into [end of digit i, L + K); ModDown: P -> Q
    ks->up_lo.resize(ks->dnum - 1);
    ks->up_hi.resize(ks->dnum);
    for (uint32_t i = 0; i < ks->dnum && rc == NTTB200_OK; i++) {
        const uint32_t lo = i * ks->alpha, hi = std::min(lo + ks->alpha, L);
        if (i) rc = conv_init(&ks->up_lo[i - 1], ks, q.data(), lo, hi, 0, lo);
        if (rc == NTTB200_OK) rc = conv_init(&ks->up_hi[i], ks, q.data(), lo, hi, hi, LK);
    }
    if (rc == NTTB200_OK) rc = conv_init(&ks->down, ks, q.data(), L, LK, 0, L);
    return rc;
}

void keyswitch_release(nttb200_rns_keyswitch *ks) {
    nttb200_rns_plan_destroy(ks->q_fwd);
    nttb200_rns_plan_destroy(ks->q_inv);
    nttb200_rns_plan_destroy(ks->qp_fwd);
    nttb200_rns_plan_destroy(ks->qp_inv);
}

// rows rows of `width` words from src (pitch sp words) to dst (pitch dp words)
static int copy_rows(int32_t *dst, uint64_t dp, const int32_t *src, uint64_t sp, uint64_t width, size_t rows,
                     cudaStream_t st) {
    NTTB200_CUDA(cudaMemcpy2DAsync(dst, dp * sizeof(int32_t), src, sp * sizeof(int32_t), width * sizeof(int32_t),
                                   rows, cudaMemcpyDeviceToDevice, st));
    return NTTB200_OK;
}

int launch_keyswitch(const nttb200_rns_keyswitch *ks, const int32_t *in, uint64_t in_stride, const int32_t *keys,
                     const uint32_t *galois, uint32_t count, int32_t *out, size_t batch, bool coeff_in,
                     bool coeff_out, bool paired, cudaStream_t st) {
    const uint64_t n = (uint64_t) 1 << ks->logn, qw = ks->q_limbs * n, rw = ks->limbs * n;
    const uint64_t prods = (uint64_t) 2 * count * batch;   // (u0, u1) polynomials on Q P
    const size_t polys = paired ? (size_t) count * batch : batch;   // input polynomials
    int32_t *dig = nullptr;
    int rc = scratch_alloc_async((void **) &dig, sizeof(int32_t) * ((uint64_t) ks->dnum * polys + prods) * rw, st);
    if (rc != NTTB200_OK) return rc;
    int32_t *prod = dig + (uint64_t) ks->dnum * polys * rw;
    // x in coefficients: the input itself, or its inverse transform in the (still unused) product buffer
    const int32_t *x = in;
    uint64_t xs = in_stride;
    if (!coeff_in) {
        const int32_t *src = in;
        if (in_stride != qw) {   // the transform reads dense rows
            rc = copy_rows(prod, qw, in, in_stride, qw, polys, st);
            src = prod;
        }
        if (rc == NTTB200_OK) rc = rns_launch(ks->q_inv, 3, src, nullptr, prod, polys, st);
        x = prod;
        xs = qw;
    }
    // ModUp straight into the digit rows, then every digit to the evaluation domain on Q P
    for (uint32_t i = 0; i < ks->dnum && rc == NTTB200_OK; i++) {
        const uint32_t lo = i * ks->alpha, hi = std::min(lo + ks->alpha, ks->q_limbs);
        int32_t *di = dig + (uint64_t) i * polys * rw;
        const int32_t *xi = x + lo * n;
        if (i) rc = launch_rns_conv(&ks->up_lo[i - 1], xi, nullptr, xs, di, rw, polys, ConvMode::Fast, false, 0, st);
        if (rc == NTTB200_OK) {
            rc = launch_rns_conv(&ks->up_hi[i], xi, nullptr, xs, di + hi * n, rw, polys, ConvMode::Fast, false, 0, st);
        }
        if (rc == NTTB200_OK) rc = copy_rows(di + lo * n, rw, xi, xs, (hi - lo) * n, polys, st);
    }
    if (rc == NTTB200_OK) rc = rns_launch(ks->qp_fwd, 1, dig, nullptr, dig, (size_t) ks->dnum * polys, st);
    if (rc == NTTB200_OK) rc = ks_dot(ks, dig, keys, prod, batch, galois, count, paired, st);
    if (rc == NTTB200_OK) rc = rns_launch(ks->qp_inv, 3, prod, nullptr, prod, prods, st);
    if (rc == NTTB200_OK) {
        rc = launch_rns_conv(&ks->down, prod + qw, prod, rw, out, qw, prods, ConvMode::Down, true, 0, st);
    }
    if (rc == NTTB200_OK && !coeff_out) rc = rns_launch(ks->q_fwd, 1, out, nullptr, out, prods, st);
    const cudaError_t e = cudaFreeAsync(dig, st);
    if (rc == NTTB200_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync");
    return rc;
}

}  // namespace nttb200
