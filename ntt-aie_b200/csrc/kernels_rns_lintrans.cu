// kernels_rns_lintrans.cu -- plaintext matrix-vector products on RNS ciphertext batches: the
// baby-step giant-step linear transform over hoisted rotations, and the call pipeline around it.
//
//   rns_lt_kernel<G, Pt>  for every output o of the call and every ciphertext b of the batch
//       Y[o][b] = sum_{terms (g, s, a, d) of o} w_d * (sigma_g(S[s][b].c0) + A[a][b].u0, A[a][b].u1)
//   mod q_l, both parts, in the rns_ct order, with w_d = sigma_h(D[d]) (h per output) when Pt and
//   w_d = 1 otherwise; a = none stands for A = (0, S[s][b].c1).
//     Inner (Pt):  S = ct, A = the hoisted baby rotations U, D = the diagonals, one output W_i per
//                  giant i, h = the rotation by -n1 i.
//     Final (!Pt): S = W, A = the giant key switches V, one output y, terms (g_i, W_i, V_i) and
//                  (1, W_0, none).
//   Work item = one 4096-word output block t of one channel row, for one output o and a group of
//   G ciphertexts (the tiling of rns_ks_dot_kernel).  The evaluation-domain permutation maps
//   output block t to the single source block brev_s((g brev_s(t) + (g-1)/2) mod 2^s), s = logn-12,
//   so each term stages the G c0 source blocks and the diagonal's source block (shared by the G
//   ciphertexts) in shared memory with cp.async, double-buffered: the next term's blocks are in
//   flight while this term's words are gathered.  The addends are read directly with 128-bit
//   loads.  No rotated copy of c0 or of a diagonal is ever written.  The products w * R accumulate
//   exactly in 64 bits and are folded every 16 terms, the rns_dot bound q + 16 (q-1)^2 < 2^64 for
//   q <= 2^30.  The output index is the fastest-moving part of the item index, so the source and
//   addend rows under way stay L2-resident while the outputs read them.
// Every pointer is 16-byte aligned (checked by the host), every index 64-bit.
#include <cuda_pipeline.h>

#include <algorithm>
#include <vector>

#include "modarith.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kL_Threads = 512;
constexpr int kL_BlockVecs = 1024;                          // uint4 of one 4096-word block
constexpr int kL_Vecs = kL_BlockVecs / kL_Threads;          // uint4 per thread
constexpr int kL_GroupOwn = 2;                              // G for batch > 1 (ptxas: no spills)
constexpr uint32_t kL_None = 0xffffffffu;                   // a term without an addend

struct RnsLtConsts {
    uint64_t mu[kConvMaxChannels];   // floor(2^64 / q_l) for reduce64
    uint32_t q[kConvMaxChannels];    // q_l
};

// table: [nout] outputs (first term, end, h, -) then the terms (g, s, a, d); items = groups * rows
// * 2^(logn - 12) * nout
template <int G, bool Pt>
__global__ void __launch_bounds__(kL_Threads, 1)
rns_lt_kernel(const uint4 *src, const uint4 *add, const uint4 *diag, const uint4 *tab, uint32_t nout, uint4 *out,
              uint64_t batch, uint32_t rows, uint32_t logn, uint64_t items, const __grid_constant__ RnsLtConsts k) {
    constexpr int kStaged = G + (Pt ? 1 : 0);   // blocks per buffer: G c0 blocks, the diagonal's
    extern __shared__ uint4 s4[];               // [2][kStaged][kL_BlockVecs]
    const uint32_t log_b = logn - 12, bmask = (1u << log_b) - 1, nmask = (1u << logn) - 1;
    const uint64_t row_vecs = (uint64_t) 1 << (logn - 2);
    const uint64_t poly_vecs = row_vecs * rows, ct_vecs = 2 * poly_vecs;
    const uint4 *terms = tab + nout;
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint32_t o = (uint32_t) (it % nout);
        const uint64_t rest = it / nout;
        const uint32_t t = (uint32_t) rest & bmask;
        const uint32_t l = (uint32_t) ((rest >> log_b) % rows);
        const uint64_t b0 = (rest >> log_b) / rows * G;
        const int gn = batch - b0 < (uint64_t) G ? (int) (batch - b0) : G;   // uniform: ragged last group
        const uint32_t q = k.q[l];
        const uint64_t mu = k.mu[l];
        const uint4 od = __ldg(tab + o);
        const uint32_t t0 = od.x, t1 = od.y;
        const uint64_t rblk = l * row_vecs + ((uint64_t) t << 10) + threadIdx.x;   // this row's block
        uint64_t cb[G];   // ciphertext offsets; the last one of a ragged group stands in for the missing ones
#pragma unroll
        for (int p = 0; p < G; p++) cb[p] = (b0 + (p < gn ? p : gn - 1)) * ct_vecs;
        // brev(k0) of every output word k0 of this thread, and the diagonal's gather index
        uint32_t bk[kL_Vecs][4], pidx[kL_Vecs][4];
        const uint32_t h = od.z, hoff = ((h - 1) / 2) & nmask;
#pragma unroll
        for (int j = 0; j < kL_Vecs; j++) {
#pragma unroll
            for (int e = 0; e < 4; e++) {
                bk[j][e] = brev_n((t << 12) + (threadIdx.x + j * kL_Threads) * 4 + e, logn);
                pidx[j][e] = brev_n((h * bk[j][e] + hoff) & nmask, logn) & (kL_BlockVecs * 4 - 1);
            }
        }
        const uint32_t ptb = log_b ? __brev((h * (__brev(t) >> (32 - log_b)) + hoff) & bmask) >> (32 - log_b) : 0;
        // issue the cp.async copies of term ti into buffer buf
        auto stage = [&](uint32_t ti, int buf) {
            const uint4 tm = __ldg(terms + ti);
            const uint32_t g = tm.x, off = ((g - 1) / 2) & nmask;
            const uint32_t sb = log_b ? __brev((g * (__brev(t) >> (32 - log_b)) + off) & bmask) >> (32 - log_b) : 0;
            const uint64_t sblk = l * row_vecs + ((uint64_t) sb << 10) + threadIdx.x;
            uint4 *s = s4 + (uint64_t) buf * kStaged * kL_BlockVecs;
#pragma unroll
            for (int p = 0; p < G; p++) {
#pragma unroll
                for (int j = 0; j < kL_Vecs; j++) {
                    __pipeline_memcpy_async(s + p * kL_BlockVecs + threadIdx.x + j * kL_Threads,
                                            src + (uint64_t) tm.y * batch * ct_vecs + cb[p] + sblk + j * kL_Threads,
                                            sizeof(uint4));
                }
            }
            if (Pt) {
                const uint64_t pblk = (uint64_t) tm.w * poly_vecs + l * row_vecs + ((uint64_t) ptb << 10) + threadIdx.x;
#pragma unroll
                for (int j = 0; j < kL_Vecs; j++) {
                    __pipeline_memcpy_async(s + G * kL_BlockVecs + threadIdx.x + j * kL_Threads,
                                            diag + pblk + j * kL_Threads, sizeof(uint4));
                }
            }
            __pipeline_commit();
        };
        uint64_t acc[G][2][kL_Vecs][4];
#pragma unroll
        for (int p = 0; p < G; p++) {
#pragma unroll
            for (int j = 0; j < kL_Vecs; j++) {
#pragma unroll
                for (int e = 0; e < 4; e++) acc[p][0][j][e] = acc[p][1][j][e] = 0;
            }
        }
        stage(t0, 0);
        for (uint32_t ti = t0; ti < t1; ti++) {
            const int cur = (ti - t0) & 1;
            if (ti + 1 < t1) stage(ti + 1, cur ^ 1);
            else __pipeline_commit();   // an empty group keeps the wait count uniform
            __pipeline_wait_prior(1);
            __syncthreads();            // this term's blocks have landed for every thread
            const uint4 tm = __ldg(terms + ti);
            const uint32_t g = tm.x, off = ((g - 1) / 2) & nmask;
            const uint32_t *s = reinterpret_cast<const uint32_t *>(s4 + (uint64_t) cur * kStaged * kL_BlockVecs);
            const uint64_t sbase = (uint64_t) tm.y * batch * ct_vecs;
            const uint64_t abase = tm.z == kL_None ? sbase : (uint64_t) tm.z * batch * ct_vecs;
#pragma unroll
            for (int j = 0; j < kL_Vecs; j++) {
                uint32_t w[4] = {1, 1, 1, 1}, gi[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    gi[e] = brev_n((g * bk[j][e] + off) & nmask, logn) & (kL_BlockVecs * 4 - 1);
                    if (Pt) w[e] = s[G * kL_BlockVecs * 4 + pidx[j][e]];
                }
#pragma unroll
                for (int p = 0; p < G; p++) {
                    uint4 a0 = make_uint4(0, 0, 0, 0), a1;
                    const uint4 *ap = (tm.z == kL_None ? src : add) + abase + cb[p] + rblk + j * kL_Threads;
                    if (tm.z == kL_None) {
                        a1 = __ldg(ap + poly_vecs);
                    } else {
                        a0 = __ldg(ap);
                        a1 = __ldg(ap + poly_vecs);
                    }
                    const uint32_t u0[4] = {a0.x, a0.y, a0.z, a0.w}, u1[4] = {a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        const uint32_t r0 = add_mod(s[p * kL_BlockVecs * 4 + gi[e]], u0[e], q);
                        acc[p][0][j][e] += (uint64_t) w[e] * r0;
                        acc[p][1][j][e] += (uint64_t) w[e] * u1[e];
                    }
                }
            }
            if (((ti - t0) & 15) == 15 || ti + 1 == t1) {   // fold: every accumulator back below q
#pragma unroll
                for (int p = 0; p < G; p++) {
#pragma unroll
                    for (int j = 0; j < kL_Vecs; j++) {
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            acc[p][0][j][e] = reduce64(acc[p][0][j][e], q, mu);
                            acc[p][1][j][e] = reduce64(acc[p][1][j][e], q, mu);
                        }
                    }
                }
            }
            __syncthreads();   // every gather from this buffer is done before it is staged again
        }
#pragma unroll
        for (int p = 0; p < G; p++) {
            if (p < gn) {
                uint4 *op = out + (uint64_t) o * batch * ct_vecs + cb[p] + rblk;
#pragma unroll
                for (int j = 0; j < kL_Vecs; j++) {
#pragma unroll
                    for (int hp = 0; hp < 2; hp++) {
                        const uint64_t *a = acc[p][hp][j];
                        __stcs(op + hp * poly_vecs + j * kL_Threads,
                               make_uint4((uint32_t) a[0], (uint32_t) a[1], (uint32_t) a[2], (uint32_t) a[3]));
                    }
                }
            }
        }
    }
}

template <int G, bool Pt>
static int lt_launch(const nttb200_rns_keyswitch *ks, const int32_t *src, const int32_t *add, const int32_t *diag,
                     const uint4 *tab, uint32_t nout, int32_t *out, size_t batch, const RnsLtConsts &k,
                     cudaStream_t st) {
    const int smem = 2 * (G + (Pt ? 1 : 0)) * kL_BlockVecs * (int) sizeof(uint4);
    NTTB200_CUDA(cudaFuncSetAttribute(rns_lt_kernel<G, Pt>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per = 0;
    NTTB200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, rns_lt_kernel<G, Pt>, kL_Threads, smem));
    const uint32_t L = ks->q_limbs;
    const uint64_t items = ((((uint64_t) batch + G - 1) / G * L) << (ks->logn - 12)) * nout;
    const uint64_t cap = (uint64_t) ks->sm_count * (per > 0 ? per : 1);
    rns_lt_kernel<G, Pt><<<(unsigned) (items < cap ? items : cap), kL_Threads, smem, st>>>(
        reinterpret_cast<const uint4 *>(src), reinterpret_cast<const uint4 *>(add),
        reinterpret_cast<const uint4 *>(diag), tab, nout, reinterpret_cast<uint4 *>(out), batch, L, ks->logn, items,
        k);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

template <bool Pt>
static int lt_run(const nttb200_rns_keyswitch *ks, const int32_t *src, const int32_t *add, const int32_t *diag,
                  const uint4 *tab, uint32_t nout, int32_t *out, size_t batch, const RnsLtConsts &k, cudaStream_t st) {
    return batch == 1 ? lt_launch<1, Pt>(ks, src, add, diag, tab, nout, out, batch, k, st)
                      : lt_launch<kL_GroupOwn, Pt>(ks, src, add, diag, tab, nout, out, batch, k, st);
}

// ---------------------------------------------------------------------------- host side
// 5^r mod 2N for a rotation by r (negative: the other way); 5 has order N/2 modulo 2N
static uint32_t rotation_element(uint32_t logn, int64_t r) {
    const uint64_t half = (uint64_t) 1 << (logn - 1), two_n = (uint64_t) 2 << logn;
    uint64_t e = (uint64_t) (((r % (int64_t) half) + (int64_t) half) % (int64_t) half), b = 5, x = 1;
    for (; e; e >>= 1, b = b * b % two_n) {
        if (e & 1) x = x * b % two_n;
    }
    return (uint32_t) x;
}

int lintrans_schedule(uint32_t logn, const uint32_t *offsets, uint32_t count, uint32_t n1, LintransSchedule *s) {
    if (logn < 12 || logn > 16 || !offsets || count == 0 || n1 < 1 || n1 > kAutoMaxElems) {
        return NTTB200_ERR_INVALID_ARG;
    }
    const uint32_t half = 1u << (logn - 1);
    std::vector<char> seen(half, 0), baby(n1, 0);
    std::vector<int32_t> giant_of((half + n1 - 1) / n1, -1);
    for (uint32_t c = 0; c < count; c++) {
        if (offsets[c] >= half || seen[offsets[c]]) return NTTB200_ERR_INVALID_ARG;
        seen[offsets[c]] = 1;
        baby[offsets[c] % n1] = 1;
        giant_of[offsets[c] / n1] = 0;
    }
    s->babies.clear();
    s->giants.clear();
    for (uint32_t j = 1; j < n1; j++) {
        if (baby[j]) s->babies.push_back(j);
    }
    for (uint32_t i = 0; i < giant_of.size(); i++) {
        if (giant_of[i] == 0) {
            giant_of[i] = (int32_t) s->giants.size();
            s->giants.push_back(i);
        }
    }
    s->offsets.assign(offsets, offsets + count);
    s->terms.assign(s->giants.size(), {});
    for (uint32_t c = 0; c < count; c++) s->terms[giant_of[offsets[c] / n1]].push_back(c);
    for (auto &tl : s->terms) {   // ascending baby step inside a giant
        std::sort(tl.begin(), tl.end(), [&](uint32_t a, uint32_t b) { return offsets[a] < offsets[b]; });
    }
    return NTTB200_OK;
}

int launch_lintrans(const nttb200_rns_keyswitch *ks, const int32_t *ct, const int32_t *diags,
                    const LintransSchedule &s, uint32_t n1, const int32_t *keys, int32_t *out, size_t batch,
                    cudaStream_t st) {
    const uint32_t logn = ks->logn;
    const uint64_t n = (uint64_t) 1 << logn, qw = ks->q_limbs * n, ctw = 2 * qw, rw = ks->limbs * n;
    const uint32_t nb = (uint32_t) s.babies.size(), nw = (uint32_t) s.giants.size();
    const uint32_t lo = s.giants[0] == 0 ? 1 : 0, ng = nw - lo;   // the giants >= 1 are W[lo..nw)
    // the tables: the inner outputs and terms, then the final output and terms
    std::vector<uint32_t> baby_at(n1, kL_None);
    for (uint32_t b = 0; b < nb; b++) baby_at[s.babies[b]] = b;
    std::vector<uint4> tab;
    uint32_t at = 0;   // term indices count from the first term, after the outputs
    for (uint32_t w = 0; w < nw; w++) {
        const uint32_t sz = (uint32_t) s.terms[w].size();
        tab.push_back(make_uint4(at, at + sz, rotation_element(logn, -(int64_t) n1 * s.giants[w]), 0));
        at += sz;
    }
    for (uint32_t w = 0; w < nw; w++) {
        for (uint32_t c : s.terms[w]) {
            const uint32_t j = s.offsets[c] % n1;
            tab.push_back(make_uint4(rotation_element(logn, j), 0, baby_at[j], c));
        }
    }
    const uint32_t fin = (uint32_t) tab.size();
    tab.push_back(make_uint4(0, nw, 1, 0));
    for (uint32_t w = 0; w < nw; w++) {
        tab.push_back(make_uint4(rotation_element(logn, (int64_t) n1 * s.giants[w]), w, w < lo ? kL_None : w - lo, 0));
    }
    std::vector<uint32_t> bg, gg;   // the Galois elements of the baby and of the giant key switches
    for (uint32_t j : s.babies) bg.push_back(rotation_element(logn, j));
    for (uint32_t w = lo; w < nw; w++) gg.push_back(rotation_element(logn, (int64_t) n1 * s.giants[w]));
    RnsLtConsts k{};
    for (uint32_t l = 0; l < ks->q_limbs; l++) {
        k.q[l] = ks->qp_fwd->pos[l].x;
        k.mu[l] = (uint64_t) ((((unsigned __int128) 1) << 64) / k.q[l]);
    }
    // scratch: the tables, U [nb][batch][2][L][N], W [nw][batch][2][L][N] (none when the only giant
    // is 0: the inner kernel writes the output), V [ng][batch][2][L][N]
    const bool direct = ng == 0;
    const uint64_t tab_words = (uint64_t) tab.size() * 4;
    const uint64_t u_words = (uint64_t) nb * batch * ctw, w_words = direct ? 0 : (uint64_t) nw * batch * ctw;
    int32_t *scr = nullptr;
    int rc = scratch_alloc_async((void **) &scr,
                                 sizeof(int32_t) * (tab_words + u_words + w_words + (uint64_t) ng * batch * ctw), st);
    if (rc != NTTB200_OK) return rc;
    const uint4 *dtab = reinterpret_cast<const uint4 *>(scr);
    int32_t *U = scr + tab_words, *W = U + u_words, *V = W + w_words;
    const cudaError_t ce = cudaMemcpyAsync(scr, tab.data(), tab.size() * sizeof(uint4), cudaMemcpyHostToDevice, st);
    if (ce != cudaSuccess) rc = cuda_fail(ce, "cudaMemcpyAsync");
    if (rc == NTTB200_OK && nb) {   // the hoisted baby rotations of every c1
        rc = launch_keyswitch(ks, ct + qw, ctw, keys, bg.data(), nb, U, batch, false, false, false, st);
    }
    if (rc == NTTB200_OK) rc = lt_run<true>(ks, ct, U, diags, dtab, nw, direct ? out : W, batch, k, st);
    // the giants: one paired key switch of W_i.c1 under key i, kAutoMaxElems at a time
    for (uint32_t c0 = 0; c0 < ng && rc == NTTB200_OK; c0 += kAutoMaxElems) {
        const uint32_t cnt = std::min<uint32_t>(ng - c0, kAutoMaxElems);
        const int32_t *kc = keys + (uint64_t) (nb + c0) * ks->dnum * 2 * rw;
        rc = launch_keyswitch(ks, W + (lo + c0) * batch * ctw + qw, ctw, kc, gg.data() + c0, cnt, V + c0 * batch * ctw,
                              batch, false, false, true, st);
    }
    if (rc == NTTB200_OK && !direct) rc = lt_run<false>(ks, W, V, nullptr, dtab + fin, 1, out, batch, k, st);
    const cudaError_t e = cudaFreeAsync(scr, st);
    if (rc == NTTB200_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync");
    return rc;
}

}  // namespace nttb200
