// kernels_packed.cu -- packed integer slots mod t for BFV and BGV on RNS batches (DESIGN 3.6).
//
// t prime, t == 1 (mod 2N), t < 2^30; slot i holds m(psi^e_i) mod t and sits at index k_i of the
// rns_ct order of a one-channel plan of modulus t (include/nttb200.h).  The transforms mod t are
// the existing RNS transforms on two one-channel plans owned by the encoder; this file adds the
// two permutations around them and the lift onto the L channels of Q:
//   encode  packed_gather<kEncode>  v[k] = x[i(k)] mod t (signed words), into pool scratch
//           rns_gs_scaled (psi^-1 plan) in place: m, coefficients in [0, t)
//           packed_lift             m -> round(Q m / t) mod q_l (SCALED) or m_c mod q_l (CENTRED)
//   decode  rns_ct (psi plan) into pool scratch: v[k] = m(psi^(2 brev(k) + 1))
//           packed_gather<kDecode / kDecodeCentred>  z[i] = v[k_i], centred if asked
// The gathers store 128-bit words on the output side and read their 4-byte sources from L2: a
// thread owns 4 consecutive outputs of one polynomial, consecutive threads the next ones, so the
// source polynomials in flight stay L2-resident while they are read.  The lift reads m once and
// writes the L rows with 128-bit stores, a thread owning 4 consecutive coefficients (the layout of
// the CKKS encode store).  No integer division on the device: reduce64 with floor(2^64 / m).
#include <vector>

#include "modarith.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kP_Threads = 256;

enum PackedGather : int { kEncode, kDecode, kDecodeCentred };

// vecs = batch * N / 4.  out[b][j] = f(in[b][perm[j]]) for 4 consecutive j per thread:
//   kEncode         f(x) = x mod t for the signed word x: (x + off) mod t, off = t ceil(2^31 / t)
//   kDecode         f(x) = x
//   kDecodeCentred  f(x) = x - t for x > t/2, else x
template <int MODE>
__global__ void __launch_bounds__(kP_Threads)
packed_gather(const uint32_t *__restrict__ in, const uint4 *perm, uint4 *out, uint64_t vecs, uint32_t logn,
              uint32_t t, uint64_t mu_t, uint64_t off) {
    const uint32_t lv = logn - 2, vmask = (1u << lv) - 1;
    for (uint64_t v = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; v < vecs;
         v += (uint64_t) gridDim.x * blockDim.x) {
        const uint4 p = __ldg(perm + (v & vmask));
        const uint32_t *src = in + ((v >> lv) << logn);
        uint32_t r[4] = {__ldg(src + p.x), __ldg(src + p.y), __ldg(src + p.z), __ldg(src + p.w)};
#pragma unroll
        for (int e = 0; e < 4; e++) {
            if (MODE == kEncode) r[e] = reduce64((uint64_t) (int64_t) (int32_t) r[e] + off, t, mu_t);
            if (MODE == kDecodeCentred) r[e] = r[e] > (t >> 1) ? r[e] - t : r[e];
        }
        __stcs(out + v, make_uint4(r[0], r[1], r[2], r[3]));
    }
}

// vecs = batch * N / 4; m [batch][N] in [0, t), out [batch][L][N].
//   SCALED   out_l = (delta_l m + rho) mod q_l, rho = round(r m / t) = floor((r m + (t-1)/2) / t);
//            delta_l m + rho < 2^60 + 2^30: one reduce64.
//   CENTRED  out_l = (m + (m > t/2 ? -t mod q_l : 0)) mod q_l; m may exceed q_l (q_l >= 2).
template <bool CENTRED>
__global__ void __launch_bounds__(kP_Threads)
packed_lift(const uint4 *m, uint4 *out, uint64_t vecs, uint32_t logn, uint32_t L,
            const __grid_constant__ PackedConsts k) {
    const uint32_t lv = logn - 2, vmask = (1u << lv) - 1;
    for (uint64_t v = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; v < vecs;
         v += (uint64_t) gridDim.x * blockDim.x) {
        const uint4 x = __ldcs(m + v);
        const uint32_t a[4] = {x.x, x.y, x.z, x.w};
        uint64_t rho[4];
        bool neg[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
            if (CENTRED) {
                neg[e] = a[e] > (k.t >> 1);
            } else {
                // floor(y / t) for y < 2^61: the estimate is exact or one short, remainder in [0, 2t)
                const uint64_t y = (uint64_t) k.r * a[e] + (k.t >> 1);
                const uint64_t qh = __umul64hi(y, k.mu_t);
                rho[e] = qh + ((uint32_t) y - (uint32_t) qh * k.t >= k.t ? 1 : 0);
            }
        }
        uint4 *o = out + (((v >> lv) * L) << lv) + (v & vmask);
        for (uint32_t l = 0; l < L; l++) {
            const uint32_t q = k.q[l];
            const uint64_t mu = k.mu[l];
            uint32_t r[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
                r[e] = CENTRED ? reduce64((uint64_t) a[e] + (neg[e] ? k.negt[l] : 0u), q, mu)
                               : reduce64((uint64_t) k.delta[l] * a[e] + rho[e], q, mu);
            }
            __stcs(o + ((uint64_t) l << lv), make_uint4(r[0], r[1], r[2], r[3]));
        }
    }
}

// ---------------------------------------------------------------------------- host side
static uint64_t mulmod(uint64_t a, uint64_t b, uint64_t m) { return a * b % m; }   // a, b < m < 2^32

// a^-1 mod m for gcd(a, m) = 1 (m need not be prime)
static uint32_t inv_mod(uint64_t a, uint64_t m) {
    int64_t r0 = (int64_t) m, r1 = (int64_t) (a % m), t0 = 0, t1 = 1;
    while (r1) {
        const int64_t qt = r0 / r1, r2 = r0 - qt * r1, t2 = t0 - qt * t1;
        r0 = r1, r1 = r2, t0 = t1, t1 = t2;
    }
    return (uint32_t) ((t0 < 0 ? t0 + (int64_t) m : t0) % (int64_t) m);
}

// The smallest primitive 2N-th root of unity mod the prime t == 1 (mod 2N): psi_0 = x^((t-1)/2N)
// for a non-residue x has order 2N (psi_0^N = x^((t-1)/2) = -1); the primitive roots are its odd
// powers.
static uint32_t smallest_psi(uint32_t t, uint32_t logn) {
    const uint64_t two_n = 2ull << logn;
    uint32_t x = 2;
    while ((uint32_t) nttb200_powmod((int32_t) x, (t - 1) / 2, (int32_t) t) != t - 1) x++;
    const uint64_t psi0 = (uint64_t) nttb200_powmod((int32_t) x, (int64_t) ((t - 1) / two_n), (int32_t) t);
    const uint64_t sq = mulmod(psi0, psi0, t);
    uint64_t best = psi0, w = psi0;
    for (uint64_t i = 1; i < two_n / 2; i++) {
        w = mulmod(w, sq, t);
        if (w < best) best = w;
    }
    return (uint32_t) best;
}

int packed_prepare(nttb200_packed_encoder *enc) {
    PackedConsts &k = enc->k;
    const uint32_t logn = enc->logn, N = 1u << logn, t = k.t;
    uint64_t r = 1;
    for (uint32_t l = 0; l < enc->limbs; l++) {
        const uint32_t q = k.q[l];
        k.mu[l] = (uint64_t) ((((unsigned __int128) 1) << 64) / q);
        r = mulmod(r, q % t, t);
    }
    k.r = (uint32_t) r;
    k.mu_t = (uint64_t) ((((unsigned __int128) 1) << 64) / t);
    for (uint32_t l = 0; l < enc->limbs; l++) {
        const uint32_t q = k.q[l];
        k.delta[l] = (uint32_t) ((q - mulmod(r % q, inv_mod(t, q), q)) % q);
        k.negt[l] = (q - t % q) % q;
    }
    const uint32_t psi = smallest_psi(t, logn);
    const uint32_t psi_inv = (uint32_t) nttb200_powmod((int32_t) psi, t - 2, (int32_t) t);
    int rc = nttb200_rns_plan_create_generated(&enc->fwd, enc->device, logn, 1, &t, NTTB200_GEN_BITREV, &psi, 0);
    if (rc == NTTB200_OK) {
        rc = nttb200_rns_plan_create_generated(&enc->inv, enc->device, logn, 1, &t, NTTB200_GEN_BITREV, &psi_inv, 0);
    }
    if (rc != NTTB200_OK) return rc;
    std::vector<uint32_t> slot(N), islot(N);
    const uint64_t two_n = 2ull << logn;
    auto brev = [logn](uint64_t x) {
        uint32_t y = 0;
        for (uint32_t b = 0; b < logn; b++) y |= (uint32_t) ((x >> b) & 1) << (logn - 1 - b);
        return y;
    };
    uint64_t g = 1;
    for (uint32_t j = 0; j < N / 2; j++, g = g * 5 % two_n) {   // slot i sits at brev((e_i - 1) / 2)
        slot[j] = brev((g - 1) / 2);
        slot[N / 2 + j] = brev((two_n - g - 1) / 2);
    }
    for (uint32_t i = 0; i < N; i++) islot[slot[i]] = i;
    NTTB200_CUDA(cudaMalloc(&enc->d_slot, N * sizeof(uint32_t)));
    NTTB200_CUDA(cudaMalloc(&enc->d_islot, N * sizeof(uint32_t)));
    NTTB200_CUDA(cudaMemcpy(enc->d_slot, slot.data(), N * sizeof(uint32_t), cudaMemcpyHostToDevice));
    NTTB200_CUDA(cudaMemcpy(enc->d_islot, islot.data(), N * sizeof(uint32_t), cudaMemcpyHostToDevice));
    return NTTB200_OK;
}

void packed_release(nttb200_packed_encoder *enc) {
    nttb200_rns_plan_destroy(enc->fwd);
    nttb200_rns_plan_destroy(enc->inv);
    cudaFree(enc->d_slot);
    cudaFree(enc->d_islot);
}

// a grid of resident CTAs (the lift holds 48 registers: 5 CTAs of 256 threads per SM, not 8)
template <class Kernel>
static int packed_grid(const nttb200_packed_encoder *enc, Kernel kernel, uint64_t vecs, int *grid) {
    int per = 0;
    NTTB200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kernel, kP_Threads, 0));
    const uint64_t blocks = (vecs + kP_Threads - 1) / kP_Threads, cap = (uint64_t) enc->sm_count * per;
    *grid = (int) (blocks < cap ? blocks : cap);
    return NTTB200_OK;
}

int launch_packed_encode(const nttb200_packed_encoder *enc, const int32_t *slots, bool centred, int32_t *out,
                         size_t batch, cudaStream_t st) {
    const uint32_t logn = enc->logn, t = enc->k.t;
    const uint64_t vecs = (uint64_t) batch << (logn - 2);
    const auto lift = centred ? packed_lift<true> : packed_lift<false>;
    int g_grid, l_grid;
    int rc = packed_grid(enc, packed_gather<kEncode>, vecs, &g_grid);
    if (rc == NTTB200_OK) rc = packed_grid(enc, lift, vecs, &l_grid);
    uint32_t *m = nullptr;
    if (rc == NTTB200_OK) rc = scratch_alloc_async((void **) &m, (sizeof(uint32_t) * batch) << logn, st);
    if (rc != NTTB200_OK) return rc;
    const uint64_t off = (uint64_t) t * (((1ull << 31) + t - 1) / t);
    packed_gather<kEncode><<<g_grid, kP_Threads, 0, st>>>(reinterpret_cast<const uint32_t *>(slots),
                                                          reinterpret_cast<const uint4 *>(enc->d_islot),
                                                          reinterpret_cast<uint4 *>(m), vecs, logn, t, enc->k.mu_t, off);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = cuda_fail(e, "packed_gather");
    if (rc == NTTB200_OK) rc = rns_launch(enc->inv, 3, (const int32_t *) m, nullptr, (int32_t *) m, batch, st);
    if (rc == NTTB200_OK) {
        lift<<<l_grid, kP_Threads, 0, st>>>(reinterpret_cast<const uint4 *>(m), reinterpret_cast<uint4 *>(out), vecs,
                                           logn, enc->limbs, enc->k);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        e = cudaGetLastError();
        if (e != cudaSuccess) rc = cuda_fail(e, "packed_lift");
    }
    cudaFreeAsync(m, st);
    return rc;
}

int launch_packed_decode(const nttb200_packed_encoder *enc, const int32_t *in, bool centred, int32_t *slots,
                         size_t batch, cudaStream_t st) {
    const uint32_t logn = enc->logn;
    const uint64_t vecs = (uint64_t) batch << (logn - 2);
    const auto gather = centred ? packed_gather<kDecodeCentred> : packed_gather<kDecode>;
    int grid;
    int rc = packed_grid(enc, gather, vecs, &grid);
    uint32_t *v = nullptr;
    if (rc == NTTB200_OK) rc = scratch_alloc_async((void **) &v, (sizeof(uint32_t) * batch) << logn, st);
    if (rc != NTTB200_OK) return rc;
    rc = rns_launch(enc->fwd, 1, in, nullptr, (int32_t *) v, batch, st);
    if (rc == NTTB200_OK) {
        gather<<<grid, kP_Threads, 0, st>>>(v, reinterpret_cast<const uint4 *>(enc->d_slot),
                                            reinterpret_cast<uint4 *>(slots), vecs, logn, enc->k.t, 0, 0);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) rc = cuda_fail(e, "packed_gather");
    }
    cudaFreeAsync(v, st);
    return rc;
}

}  // namespace nttb200
