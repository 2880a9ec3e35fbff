// kernels_ckks.cu -- CKKS slot encoding and decoding on RNS batches: the canonical embedding as an
// FP64 negacyclic FFT (DESIGN 3.6).
//
// n = N/2 slots, zeta = e^(i pi / N), w = e^(2 pi i / n), s_j = (5^j mod 2N - 1) / 4.
//   decode: y_k = (x_k + i x_(k+n)) zeta^k (k < n), Y_s = sum_k y_k w^(sk), z_j = Y_(s_j) / scale
//   encode: v_(s_j) = z_j, Y_k = sum_s v_s w^(-sk), a_k + i a_(k+n) = rint(scale / n * Y_k zeta^-k)
// The transform is a radix-2 decimation-in-frequency DFT in shared memory (natural order in,
// bit-reversed order out); the fold-and-twist, the permutation s_j and the bit reversal ride on
// its load and store.
//   n <= 2^13  one CTA per polynomial, one launch (ckks_encode_cta / ckks_decode_cta).
//   n >= 2^14  n = n1 * 2^13 with n1 = 2 or 4, two launches through pool scratch T:
//     encode  rows: per (poly, j1) the 2^13-point DFT of v_(j1 + n1 j2) over j2, times
//                   w^(-j1 k2), into T[j1][k2];  cols: the n1-point DFTs over j1 and the store.
//     decode  cols: the load and the n1-point DFTs over j1 of y_(j2 + 2^13 j1), times w^(k1 j2),
//                   into T[k1][j2];  rows: per (poly, k1) the 2^13-point DFT over j2 and the store.
//   Encode ends with rint (half to even) and fans each rounded coefficient out to the L channel
//   rows, reduced once per channel, with 128-bit stores.  Decode starts with the exact CRT of up to
//   four channels in 128-bit integers.  No step goes through float.
#include <math.h>

#include <algorithm>
#include <numeric>
#include <utility>

#include "modarith.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kCkThreads = 512;        // CTA and row kernels
constexpr int kColThreads = 256;       // column kernels
constexpr uint32_t kRowLog = 13;       // 2^13 complex doubles = 128 KiB of shared memory
constexpr uint32_t kRowLen = 1u << kRowLog;

typedef unsigned __int128 u128;

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 conj2(double2 a) { return make_double2(a.x, -a.y); }
__device__ __forceinline__ uint32_t brev(uint32_t x, uint32_t bits) { return __brev(x) >> (32 - bits); }

// In place, length m = 2^lm in shared memory: X_k = sum_j x_j u^(jk) with u = w^(n/m) (INV) or its
// conjugate, X_k left at position brev(k).  W[t] = w^t; ts = n / m.
template <bool INV>
__device__ __forceinline__ void fft_dif(double2 *x, uint32_t lm, const double2 *W, uint32_t ts) {
    const uint32_t half = 1u << (lm - 1);
    for (int lh = (int) lm - 1; lh >= 0; lh--) {
        const uint32_t h = 1u << lh;
        for (uint32_t i = threadIdx.x; i < half; i += blockDim.x) {
            const uint32_t r = i & (h - 1), j = ((i >> lh) << (lh + 1)) | r;
            double2 w = __ldg(W + (r << (lm - 1 - lh)) * ts);
            if (!INV) w.y = -w.y;
            const double2 a = x[j], b = x[j + h];
            x[j] = make_double2(a.x + b.x, a.y + b.y);
            x[j + h] = cmul(make_double2(a.x - b.x, a.y - b.y), w);
        }
        __syncthreads();
    }
}

// |x| >= 2^63 (or not finite): |x| = M 2^e with M < 2^53, so x mod q = +-(M mod q)(2^e mod q).
__device__ __noinline__ uint32_t big_residue(double x, uint32_t q, uint64_t mu) {
    const uint64_t bits = (uint64_t) __double_as_longlong(x);
    uint32_t e = (uint32_t) ((bits >> 52) & 0x7ff) - 1075;
    uint32_t r = reduce64((bits & ((1ull << 52) - 1)) | (1ull << 52), q, mu);
    uint32_t base = reduce64(2, q, mu);
    for (; e; e >>= 1) {
        if (e & 1) r = reduce64((uint64_t) r * base, q, mu);
        base = reduce64((uint64_t) base * base, q, mu);
    }
    return (x < 0 && r) ? q - r : r;
}

// a = rint(x[e]) for coefficients k0 + e (e < 4) and n + k0 + e (e >= 4), written as residues to
// the L rows at o (row pitch N words): each value is rounded once and reduced once per channel.
__device__ __forceinline__ void encode_store(uint32_t *o, uint32_t logn, uint32_t k0, uint32_t L, const double (&x)[8],
                                             const CkksEncConsts &k) {
    const uint32_t n = 1u << (logn - 1);
    uint64_t u[8];
    bool neg[8], big = false;
#pragma unroll
    for (int e = 0; e < 8; e++) {
        const bool small = fabs(x[e]) < 0x1p63;
        const long long a = small ? __double2ll_rn(x[e]) : 0;
        neg[e] = a < 0;
        u[e] = neg[e] ? 0ull - (uint64_t) a : (uint64_t) a;
        big |= !small;
    }
    for (uint32_t l = 0; l < L; l++) {
        const uint32_t q = k.q[l];
        const uint64_t mu = k.mu[l];
        uint32_t r[8];
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const uint32_t t = reduce64(u[e], q, mu);
            r[e] = (neg[e] && t) ? q - t : t;
        }
        if (big) {
#pragma unroll
            for (int e = 0; e < 8; e++) {
                if (!(fabs(x[e]) < 0x1p63)) r[e] = big_residue(x[e], q, mu);
            }
        }
        uint32_t *row = o + ((uint64_t) l << logn) + k0;
        __stcs(reinterpret_cast<uint4 *>(row), make_uint4(r[0], r[1], r[2], r[3]));
        __stcs(reinterpret_cast<uint4 *>(row + n), make_uint4(r[4], r[5], r[6], r[7]));
    }
}

__device__ __forceinline__ u128 u128_of(const uint64_t (&v)[2]) { return ((u128) v[1] << 64) | v[0]; }

// correctly rounded: the top 64 bits with a sticky bit for the rest, one rounding to 53 bits
__device__ __forceinline__ double u128_to_double(u128 u) {
    const uint64_t hi = (uint64_t) (u >> 64);
    if (hi == 0) return __ull2double_rn((uint64_t) u);
    const int lz = __clzll(hi);
    const u128 t = u << lz;
    const uint64_t top = (uint64_t) (t >> 64) | (uint64_t) ((uint64_t) t != 0);
    return __ull2double_rn(top) * __hiloint2double((1023 + 64 - lz) << 20, 0);
}

// The centred CRT value x_c in (-B/2, B/2] of 4 consecutive columns at p over the first C rows
// (row pitch N words): S = sum_i y_i (B/b_i) < C B, v = #{k : 2S > (2k+1) B}, x_c = S - v B.
__device__ __forceinline__ void crt_centred(const uint32_t *p, uint32_t logn, uint32_t C, const CkksDecConsts &k,
                                            double (&x)[4]) {
    u128 s[4] = {0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < kCkksMaxDecode; i++) {
        if (i < (int) C) {
            const uint4 v = __ldcs(reinterpret_cast<const uint4 *>(p + ((uint64_t) i << logn)));
            const uint32_t r[4] = {v.x, v.y, v.z, v.w};
            const u128 m = u128_of(k.m[i]);
#pragma unroll
            for (int e = 0; e < 4; e++) s[e] += (u128) shoup_mul(r[e], k.w[i], k.wp[i], k.b[i]) * m;
        }
    }
    const u128 B = u128_of(k.bb);
#pragma unroll
    for (int e = 0; e < 4; e++) {
        const u128 s2 = s[e] << 1;
        uint32_t v = 0;
#pragma unroll
        for (int t = 0; t < kCkksMaxDecode; t++) v += s2 > u128_of(k.t[t]) ? 1u : 0u;
        const u128 vb = (u128) v * B;
        x[e] = s[e] >= vb ? u128_to_double(s[e] - vb) : -u128_to_double(vb - s[e]);
    }
}

// ------------------------------------------------------------------ n <= 2^13: one CTA per polynomial
__global__ void __launch_bounds__(kCkThreads)
ckks_encode_cta(const double2 *slots, uint32_t *out, uint32_t logn, uint32_t L, uint64_t batch, double scale_n,
                const double2 *W, const double2 *zeta, const uint32_t *perm, const __grid_constant__ CkksEncConsts k) {
    extern __shared__ double2 sh[];
    const uint32_t lm = logn - 1, n = 1u << lm;
    for (uint64_t poly = blockIdx.x; poly < batch; poly += gridDim.x) {
        const double2 *z = slots + poly * n;
        for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) sh[__ldg(perm + j)] = __ldcs(z + j);
        __syncthreads();
        fft_dif<false>(sh, lm, W, 1);
        uint32_t *o = out + ((poly * L) << logn);
        for (uint32_t k0 = threadIdx.x * 4; k0 < n; k0 += blockDim.x * 4) {
            double x[8];
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const double2 m = cmul(sh[brev(k0 + e, lm)], conj2(__ldg(zeta + k0 + e)));
                x[e] = m.x * scale_n;
                x[4 + e] = m.y * scale_n;
            }
            encode_store(o, logn, k0, L, x, k);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kCkThreads)
ckks_decode_cta(const uint32_t *in, uint64_t in_stride, uint32_t C, double2 *slots, uint32_t logn, uint64_t batch,
                const double2 *W, const double2 *zeta, const uint32_t *perm, const __grid_constant__ CkksDecConsts k) {
    extern __shared__ double2 sh[];
    const uint32_t lm = logn - 1, n = 1u << lm;
    for (uint64_t poly = blockIdx.x; poly < batch; poly += gridDim.x) {
        const uint32_t *p = in + poly * in_stride;
        for (uint32_t k0 = threadIdx.x * 4; k0 < n; k0 += blockDim.x * 4) {
            double re[4], im[4];
            crt_centred(p + k0, logn, C, k, re);
            crt_centred(p + n + k0, logn, C, k, im);
#pragma unroll
            for (int e = 0; e < 4; e++) sh[k0 + e] = cmul(make_double2(re[e], im[e]), __ldg(zeta + k0 + e));
        }
        __syncthreads();
        fft_dif<true>(sh, lm, W, 1);
        double2 *z = slots + poly * n;
        for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
            const double2 v = sh[brev(__ldg(perm + j), lm)];
            __stcs(z + j, make_double2(v.x * k.inv_scale, v.y * k.inv_scale));
        }
        __syncthreads();
    }
}

// ------------------------------------------------------- n = N1 * 2^13: row and column passes
// items = batch * n1; row it = poly * n1 + j1 of T
__global__ void __launch_bounds__(kCkThreads)
ckks_encode_rows(const double2 *slots, double2 *T, uint32_t logn, uint64_t items, const double2 *W,
                 const uint32_t *iperm) {
    extern __shared__ double2 sh[];
    const uint32_t lm = logn - 1, ln1 = lm - kRowLog, n1 = 1u << ln1;
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint32_t j1 = (uint32_t) it & (n1 - 1);
        const double2 *z = slots + (it >> ln1 << lm);
        for (uint32_t j2 = threadIdx.x; j2 < kRowLen; j2 += blockDim.x) sh[j2] = z[__ldg(iperm + j1 + (j2 << ln1))];
        __syncthreads();
        fft_dif<false>(sh, kRowLog, W, n1);
        double2 *t = T + it * kRowLen;
        for (uint32_t k2 = threadIdx.x; k2 < kRowLen; k2 += blockDim.x) {
            t[k2] = cmul(sh[brev(k2, kRowLog)], conj2(__ldg(W + j1 * k2)));
        }
        __syncthreads();
    }
}

// items = batch * 2^13 / 4; a thread owns columns k2 .. k2 + 3 of one polynomial
template <int N1>
__global__ void __launch_bounds__(kColThreads)
ckks_encode_cols(const double2 *T, uint32_t *out, uint32_t logn, uint32_t L, uint64_t items, double scale_n,
                 const double2 *W, const double2 *zeta, const __grid_constant__ CkksEncConsts k) {
    for (uint64_t it = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; it < items;
         it += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t poly = it >> (kRowLog - 2);
        const uint32_t k2 = ((uint32_t) it & (kRowLen / 4 - 1)) * 4;
        const double2 *t = T + poly * N1 * kRowLen + k2;
        double2 v[N1][4];
#pragma unroll
        for (int j1 = 0; j1 < N1; j1++) {
#pragma unroll
            for (int e = 0; e < 4; e++) v[j1][e] = __ldcs(t + j1 * kRowLen + e);
        }
        uint32_t *o = out + ((poly * L) << logn);
#pragma unroll
        for (int k1 = 0; k1 < N1; k1++) {
            double x[8];
#pragma unroll
            for (int e = 0; e < 4; e++) {
                double2 acc = v[0][e];
#pragma unroll
                for (int j1 = 1; j1 < N1; j1++) {
                    const double2 p = cmul(v[j1][e], conj2(__ldg(W + (((j1 * k1) & (N1 - 1)) << kRowLog))));
                    acc = make_double2(acc.x + p.x, acc.y + p.y);
                }
                const double2 m = cmul(acc, conj2(__ldg(zeta + (k1 << kRowLog) + k2 + e)));
                x[e] = m.x * scale_n;
                x[4 + e] = m.y * scale_n;
            }
            encode_store(o, logn, (k1 << kRowLog) + k2, L, x, k);
        }
    }
}

// items = batch * 2^13 / 4; a thread owns columns j2 .. j2 + 3 of one polynomial
template <int N1>
__global__ void __launch_bounds__(kColThreads)
ckks_decode_cols(const uint32_t *in, uint64_t in_stride, uint32_t C, double2 *T, uint32_t logn, uint64_t items,
                 const double2 *W, const double2 *zeta, const __grid_constant__ CkksDecConsts k) {
    const uint32_t n = 1u << (logn - 1);
    for (uint64_t it = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; it < items;
         it += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t poly = it >> (kRowLog - 2);
        const uint32_t j2 = ((uint32_t) it & (kRowLen / 4 - 1)) * 4;
        const uint32_t *p = in + poly * in_stride + j2;
        double2 y[N1][4];
#pragma unroll
        for (int j1 = 0; j1 < N1; j1++) {
            double re[4], im[4];
            crt_centred(p + (j1 << kRowLog), logn, C, k, re);
            crt_centred(p + n + (j1 << kRowLog), logn, C, k, im);
#pragma unroll
            for (int e = 0; e < 4; e++) {
                y[j1][e] = cmul(make_double2(re[e], im[e]), __ldg(zeta + (j1 << kRowLog) + j2 + e));
            }
        }
        double2 *t = T + poly * N1 * kRowLen + j2;
#pragma unroll
        for (int k1 = 0; k1 < N1; k1++) {
#pragma unroll
            for (int e = 0; e < 4; e++) {
                double2 acc = y[0][e];
#pragma unroll
                for (int j1 = 1; j1 < N1; j1++) {
                    const double2 q = cmul(y[j1][e], __ldg(W + (((j1 * k1) & (N1 - 1)) << kRowLog)));
                    acc = make_double2(acc.x + q.x, acc.y + q.y);
                }
                t[k1 * kRowLen + e] = k1 ? cmul(acc, __ldg(W + k1 * (j2 + e))) : acc;
            }
        }
    }
}

// items = batch * n1; row it = poly * n1 + k1 of T
__global__ void __launch_bounds__(kCkThreads)
ckks_decode_rows(const double2 *T, double2 *slots, uint32_t logn, uint64_t items, const double2 *W,
                 const uint32_t *iperm, double inv_scale) {
    extern __shared__ double2 sh[];
    const uint32_t lm = logn - 1, ln1 = lm - kRowLog, n1 = 1u << ln1;
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint32_t k1 = (uint32_t) it & (n1 - 1);
        const double2 *t = T + it * kRowLen;
        for (uint32_t j2 = threadIdx.x; j2 < kRowLen; j2 += blockDim.x) sh[j2] = __ldcs(t + j2);
        __syncthreads();
        fft_dif<true>(sh, kRowLog, W, n1);
        double2 *z = slots + (it >> ln1 << lm);
        for (uint32_t pos = threadIdx.x; pos < kRowLen; pos += blockDim.x) {
            const double2 v = sh[pos];
            z[__ldg(iperm + k1 + (brev(pos, kRowLog) << ln1))] = make_double2(v.x * inv_scale, v.y * inv_scale);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------- host side
// e^(2 pi i t / M) for M a power of two >= 8, within 1 ulp: the angle is reduced to [0, pi/4] on
// the integer t, then evaluated in long double (64-bit significand) and rounded once.
static double2 unit_root(uint64_t t, uint64_t M) {
    const long double two_pi = 6.283185307179586476925286766559005768L;
    t %= M;
    const uint64_t quarter = M / 4, qd = t / quarter, r = t % quarter;
    const bool swap = 2 * r > quarter;
    const long double phi = two_pi * ((long double) (swap ? quarter - r : r) / (long double) M);
    long double c = cosl(phi), s = sinl(phi);
    if (swap) std::swap(c, s);
    long double re = c, im = s;
    switch (qd) {
        case 1: re = -s, im = c; break;
        case 2: re = -c, im = -s; break;
        case 3: re = s, im = -c; break;
        default: break;
    }
    return make_double2((double) re, (double) im);
}

int ckks_prepare(nttb200_ckks_encoder *enc) {
    const uint32_t n = 1u << (enc->logn - 1);
    const uint64_t two_n = 2ull << enc->logn;
    std::vector<double2> w(n), zeta(n);
    std::vector<uint32_t> perm(n), iperm(n);
    for (uint32_t t = 0; t < n; t++) {
        w[t] = unit_root(t, n);
        zeta[t] = unit_root(t, two_n);
    }
    uint64_t g = 1;
    for (uint32_t j = 0; j < n; j++, g = g * 5 % two_n) {
        perm[j] = (uint32_t) ((g - 1) / 4);
        iperm[perm[j]] = j;
    }
    NTTB200_CUDA(cudaMalloc(&enc->d_w, n * sizeof(double2)));
    NTTB200_CUDA(cudaMalloc(&enc->d_zeta, n * sizeof(double2)));
    NTTB200_CUDA(cudaMalloc(&enc->d_perm, n * sizeof(uint32_t)));
    NTTB200_CUDA(cudaMalloc(&enc->d_iperm, n * sizeof(uint32_t)));
    NTTB200_CUDA(cudaMemcpy(enc->d_w, w.data(), n * sizeof(double2), cudaMemcpyHostToDevice));
    NTTB200_CUDA(cudaMemcpy(enc->d_zeta, zeta.data(), n * sizeof(double2), cudaMemcpyHostToDevice));
    NTTB200_CUDA(cudaMemcpy(enc->d_perm, perm.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice));
    NTTB200_CUDA(cudaMemcpy(enc->d_iperm, iperm.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice));
    const int smem = (int) (kRowLen * sizeof(double2));
    NTTB200_CUDA(cudaFuncSetAttribute(ckks_encode_cta, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    NTTB200_CUDA(cudaFuncSetAttribute(ckks_decode_cta, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    NTTB200_CUDA(cudaFuncSetAttribute(ckks_encode_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    NTTB200_CUDA(cudaFuncSetAttribute(ckks_decode_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    return NTTB200_OK;
}

// a^-1 mod m for gcd(a, m) = 1 (the moduli need not be prime)
static uint32_t inv_mod(uint64_t a, uint64_t m) {
    int64_t r0 = (int64_t) m, r1 = (int64_t) (a % m), t0 = 0, t1 = 1;
    while (r1) {
        const int64_t qt = r0 / r1, r2 = r0 - qt * r1, t2 = t0 - qt * t1;
        r0 = r1, r1 = r2, t0 = t1, t1 = t2;
    }
    return (uint32_t) ((t0 < 0 ? t0 + (int64_t) m : t0) % (int64_t) m);
}

int ckks_decode_consts(const nttb200_ckks_encoder *enc, uint32_t channels, double scale, CkksDecConsts *k) {
    const uint32_t *b = enc->k.q;
    for (uint32_t x = 0; x < channels; x++) {
        for (uint32_t z = x + 1; z < channels; z++) {
            if (std::gcd(b[x], b[z]) != 1) return NTTB200_ERR_MODULUS;
        }
    }
    *k = CkksDecConsts{};
    u128 B = 1;
    for (uint32_t i = 0; i < channels; i++) B *= b[i];
    for (uint32_t i = 0; i < channels; i++) {
        const u128 m = B / b[i];
        k->m[i][0] = (uint64_t) m, k->m[i][1] = (uint64_t) (m >> 64);
        k->b[i] = b[i];
        k->w[i] = inv_mod((uint64_t) (m % b[i]), b[i]);
        k->wp[i] = (uint32_t) (((uint64_t) k->w[i] << 32) / b[i]);
    }
    for (int t = 0; t < kCkksMaxDecode; t++) {
        const u128 th = (u128) (2 * t + 1) * B;
        k->t[t][0] = (uint64_t) th, k->t[t][1] = (uint64_t) (th >> 64);
    }
    k->bb[0] = (uint64_t) B, k->bb[1] = (uint64_t) (B >> 64);
    k->inv_scale = 1.0 / scale;
    return NTTB200_OK;
}

void ckks_release(nttb200_ckks_encoder *enc) {
    cudaFree(enc->d_w);
    cudaFree(enc->d_zeta);
    cudaFree(enc->d_perm);
    cudaFree(enc->d_iperm);
}

// resident CTAs of a shared-memory kernel: at most 2048 threads and 228 KiB per SM
static int cta_grid(const nttb200_ckks_encoder *enc, uint64_t items, size_t smem) {
    const uint64_t per = std::min<uint64_t>(2048 / kCkThreads, (228u << 10) / (smem + 1024));
    const uint64_t cap = (uint64_t) enc->sm_count * per;
    return (int) (items < cap ? items : cap);
}

static int col_grid(const nttb200_ckks_encoder *enc, uint64_t items) {
    const uint64_t blocks = (items + kColThreads - 1) / kColThreads, cap = (uint64_t) enc->sm_count * 8;
    return (int) (blocks < cap ? blocks : cap);
}

int launch_ckks_encode(const nttb200_ckks_encoder *enc, const double2 *slots, double scale, int32_t *out,
                       size_t batch, cudaStream_t st) {
    if (batch == 0) return NTTB200_OK;
    const uint32_t logn = enc->logn, lm = logn - 1;
    const double scale_n = scale / (double) (1u << lm);
    uint32_t *o = reinterpret_cast<uint32_t *>(out);
    if (lm <= kRowLog) {
        const size_t smem = sizeof(double2) << lm;
        ckks_encode_cta<<<cta_grid(enc, batch, smem), kCkThreads, smem, st>>>(
            slots, o, logn, enc->limbs, batch, scale_n, enc->d_w, enc->d_zeta, enc->d_perm, enc->k);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        NTTB200_CUDA(cudaGetLastError());
        return NTTB200_OK;
    }
    double2 *T = nullptr;
    const int rc = scratch_alloc_async((void **) &T, (sizeof(double2) * batch) << lm, st);
    if (rc != NTTB200_OK) return rc;
    const uint64_t rows = (uint64_t) batch << (lm - kRowLog), cols = (uint64_t) batch * (kRowLen / 4);
    const size_t smem = sizeof(double2) * kRowLen;
    ckks_encode_rows<<<cta_grid(enc, rows, smem), kCkThreads, smem, st>>>(slots, T, logn, rows, enc->d_w,
                                                                           enc->d_iperm);
    if (lm - kRowLog == 1) {
        ckks_encode_cols<2><<<col_grid(enc, cols), kColThreads, 0, st>>>(T, o, logn, enc->limbs, cols, scale_n,
                                                                         enc->d_w, enc->d_zeta, enc->k);
    } else {
        ckks_encode_cols<4><<<col_grid(enc, cols), kColThreads, 0, st>>>(T, o, logn, enc->limbs, cols, scale_n,
                                                                         enc->d_w, enc->d_zeta, enc->k);
    }
    g_launches.fetch_add(2, std::memory_order_relaxed);
    const cudaError_t e = cudaGetLastError();
    cudaFreeAsync(T, st);
    NTTB200_CUDA(e);
    return NTTB200_OK;
}

int launch_ckks_decode(const nttb200_ckks_encoder *enc, const int32_t *in, uint64_t in_stride, uint32_t channels,
                       const CkksDecConsts &k, double2 *slots, size_t batch, cudaStream_t st) {
    if (batch == 0) return NTTB200_OK;
    const uint32_t logn = enc->logn, lm = logn - 1;
    const uint32_t *src = reinterpret_cast<const uint32_t *>(in);
    if (lm <= kRowLog) {
        const size_t smem = sizeof(double2) << lm;
        ckks_decode_cta<<<cta_grid(enc, batch, smem), kCkThreads, smem, st>>>(
            src, in_stride, channels, slots, logn, batch, enc->d_w, enc->d_zeta, enc->d_perm, k);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        NTTB200_CUDA(cudaGetLastError());
        return NTTB200_OK;
    }
    double2 *T = nullptr;
    const int rc = scratch_alloc_async((void **) &T, (sizeof(double2) * batch) << lm, st);
    if (rc != NTTB200_OK) return rc;
    const uint64_t rows = (uint64_t) batch << (lm - kRowLog), cols = (uint64_t) batch * (kRowLen / 4);
    const size_t smem = sizeof(double2) * kRowLen;
    if (lm - kRowLog == 1) {
        ckks_decode_cols<2><<<col_grid(enc, cols), kColThreads, 0, st>>>(src, in_stride, channels, T, logn, cols,
                                                                         enc->d_w, enc->d_zeta, k);
    } else {
        ckks_decode_cols<4><<<col_grid(enc, cols), kColThreads, 0, st>>>(src, in_stride, channels, T, logn, cols,
                                                                         enc->d_w, enc->d_zeta, k);
    }
    ckks_decode_rows<<<cta_grid(enc, rows, smem), kCkThreads, smem, st>>>(T, slots, logn, rows, enc->d_w,
                                                                           enc->d_iperm, k.inv_scale);
    g_launches.fetch_add(2, std::memory_order_relaxed);
    const cudaError_t e = cudaGetLastError();
    cudaFreeAsync(T, st);
    NTTB200_CUDA(e);
    return NTTB200_OK;
}

}  // namespace nttb200
