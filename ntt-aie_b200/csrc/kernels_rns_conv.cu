// kernels_rns_conv.cu -- basis conversion between the primes of two RNS plans
// ([batch][channels][N] rows, coefficient domain).
//
//   rns_conv_kernel<S, V, M>  one kernel for four operations (ConvMode M):
//       Fast   the fast base conversion, x + alpha B;
//       Down   the division by B (with or without rounding: the host zeroes h);
//       Exact  the exact base conversion of the centred x;
//       Scale  round(t X / B) (t folded into w / wp and tc / tcp by the host).
//     Work item = one chunk of 256 * V consecutive columns of one polynomial; a thread owns V
//     consecutive columns (one V-word load or store per channel row, coalesced along the columns).
//     phase 1: the S source residues are loaded and turned into y_i = x_i (B/b_i)^-1 mod b_i
//              with one Shoup multiply each (Down: x_i + h_B,i first); all of them stay in
//              registers, one instantiation per S.  Exact / Scale also compute
//              v = rint(sum_i y_i / b_i) in FP64 (HPS): one exact I2F.F64 and one DFMA per term
//              with 1/b_i from the parameter block; the rint is the low word of the sum plus
//              2^52.  (Building the double as 2^52 + y_i less 2^52 instead needs a register pair
//              per term and doubles the register count: DESIGN 3.6.)
//     phase 2: for each target channel j (warp-uniform, so m[j][i] is a broadcast constant
//              operand): sum_i y_i m[j][i] exactly in 64 bits, folded with reduce64 after 16
//              terms -- c + 16 (2^30 - 1)^2 < 2^64 for moduli <= 2^30, the bound of rns_dot --
//              and reduced mod c_j.  Down: (x_C,j + h_C,j - sum) * B^-1 mod c_j (Shoup).
//              Exact / Scale start the sum at v (-B mod c_j) <= S (c_j - 1), which keeps
//              the bound: S (c - 1) + 16 (c - 1)^2 < 2^64.  Scale: (t x_C,j - sum) * B^-1.
#include <array>
#include <numeric>
#include <utility>

#include "modarith.cuh"
#include "plan.h"

namespace nttb200 {

constexpr int kC_Threads = 256;

template <int V> struct ConvVec;
template <> struct ConvVec<4> {
    using T = uint4;
    static __device__ __forceinline__ void get(const T &v, uint32_t *x) { x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w; }
    static __device__ __forceinline__ T make(const uint32_t *x) { return make_uint4(x[0], x[1], x[2], x[3]); }
};
template <> struct ConvVec<2> {
    using T = uint2;
    static __device__ __forceinline__ void get(const T &v, uint32_t *x) { x[0] = v.x; x[1] = v.y; }
    static __device__ __forceinline__ T make(const uint32_t *x) { return make_uint2(x[0], x[1]); }
};

// items = batch << log_chunks (2^log_chunks chunks of 256 * V columns per polynomial)
template <int S, int V, ConvMode M>
__global__ void __launch_bounds__(kC_Threads)
rns_conv_kernel(const uint32_t *src, const uint32_t *tin, uint32_t *out, uint64_t src_stride, uint64_t out_stride,
                uint32_t logn, uint32_t T, uint64_t items, uint32_t log_chunks,
                const __grid_constant__ RnsConvConsts k) {
    constexpr bool DOWN = M == ConvMode::Down;
    constexpr bool HPS = M == ConvMode::Exact || M == ConvMode::Scale;
    using Vec = typename ConvVec<V>::T;
    for (uint64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const uint64_t poly = it >> log_chunks;
        const uint64_t col = ((it & ((1u << log_chunks) - 1)) * kC_Threads + threadIdx.x) * V;
        const uint32_t *s = src + poly * src_stride + col;
        uint32_t y[S][V];
#pragma unroll
        for (int i = 0; i < S; i++) {
            ConvVec<V>::get(__ldcs(reinterpret_cast<const Vec *>(s + ((uint64_t) i << logn))), y[i]);
        }
#pragma unroll
        for (int i = 0; i < S; i++) {
#pragma unroll
            for (int e = 0; e < V; e++) {
                const uint32_t x = DOWN ? add_mod(y[i][e], k.hb[i], k.b[i]) : y[i][e];
                y[i][e] = shoup_mul(x, k.w[i], k.wp[i], k.b[i]);
            }
        }
        uint32_t v[V];
        if constexpr (HPS) {
            double f[V];
#pragma unroll
            for (int e = 0; e < V; e++) f[e] = 0.0;
#pragma unroll
            for (int i = 0; i < S; i++) {
#pragma unroll
                for (int e = 0; e < V; e++) f[e] = __fma_rn(__uint2double_rn(y[i][e]), k.binvd[i], f[e]);
            }
#pragma unroll
            for (int e = 0; e < V; e++) v[e] = (uint32_t) __double2loint(__dadd_rn(f[e], 0x1p52));
        }
        for (uint32_t j = 0; j < T; j++) {
            const uint32_t c = k.c[j];
            const uint64_t mu = k.mu[j];
            uint64_t acc[V];
#pragma unroll
            for (int e = 0; e < V; e++) {
                if constexpr (HPS) {
                    acc[e] = (uint64_t) v[e] * k.nbc[j];
                } else {
                    acc[e] = 0;
                }
            }
#pragma unroll
            for (int i = 0; i < S; i++) {
                if (i == 16) {
#pragma unroll
                    for (int e = 0; e < V; e++) acc[e] = reduce64(acc[e], c, mu);
                }
                const uint32_t m = k.m[j][i];
#pragma unroll
                for (int e = 0; e < V; e++) acc[e] += (uint64_t) y[i][e] * m;
            }
            uint32_t r[V];
#pragma unroll
            for (int e = 0; e < V; e++) r[e] = reduce64(acc[e], c, mu);
            const uint64_t row = (uint64_t) j << logn;
            if constexpr (DOWN || M == ConvMode::Scale) {
                uint32_t x[V];
                ConvVec<V>::get(__ldcs(reinterpret_cast<const Vec *>(tin + poly * src_stride + row + col)), x);
#pragma unroll
                for (int e = 0; e < V; e++) {
                    const uint32_t tx = DOWN ? add_mod(x[e], k.hc[j], c) : shoup_mul(x[e], k.tc[j], k.tcp[j], c);
                    r[e] = shoup_mul(sub_mod(tx, r[e], c), k.binv[j], k.binvp[j], c);
                }
            }
            __stcs(reinterpret_cast<Vec *>(out + poly * out_stride + row + col), ConvVec<V>::make(r));
        }
    }
}

// ---------------------------------------------------------------------------- host side
static uint64_t mulmod64(uint64_t a, uint64_t b, uint64_t m) {
    return (uint64_t) ((unsigned __int128) a * b % m);
}

// a^-1 mod m for gcd(a, m) = 1 (extended Euclid: the moduli need not be prime)
static uint32_t inv_mod(uint64_t a, uint64_t m) {
    int64_t r0 = (int64_t) m, r1 = (int64_t) (a % m), t0 = 0, t1 = 1;
    while (r1) {
        const int64_t qt = r0 / r1, r2 = r0 - qt * r1, t2 = t0 - qt * t1;
        r0 = r1, r1 = r2, t0 = t1, t1 = t2;
    }
    return (uint32_t) (t0 < 0 ? t0 + (int64_t) m : t0) % (uint32_t) m;
}

// prod_{k != skip} b_k mod m (skip = S: the whole product B)
static uint64_t prod_mod(const uint32_t *b, uint32_t S, uint32_t skip, uint64_t m) {
    uint64_t p = 1 % m;
    for (uint32_t k = 0; k < S; k++) {
        if (k != skip) p = mulmod64(p, b[k], m);
    }
    return p;
}

int rns_conv_prepare(nttb200_rns_conv *cv, const uint32_t *b, const uint32_t *c) {
    const uint32_t S = cv->src, T = cv->dst;
    std::vector<uint32_t> all(b, b + S);
    all.insert(all.end(), c, c + T);
    for (size_t x = 0; x < all.size(); x++) {
        for (size_t z = x + 1; z < all.size(); z++) {
            if (std::gcd(all[x], all[z]) != 1) return NTTB200_ERR_MODULUS;
        }
    }
    RnsConvConsts &k = cv->k;
    k = RnsConvConsts{};
    // floor(B/2) mod m = floor((B mod 2m) / 2), also when one modulus is even
    for (uint32_t i = 0; i < S; i++) {
        k.b[i] = b[i];
        k.w[i] = inv_mod(prod_mod(b, S, i, b[i]), b[i]);
        k.wp[i] = (uint32_t) (((uint64_t) k.w[i] << 32) / b[i]);
        k.hb[i] = (uint32_t) (prod_mod(b, S, S, 2ull * b[i]) / 2);
        k.binvd[i] = 1.0 / b[i];   // correctly rounded: relative error <= 2^-53
    }
    for (uint32_t j = 0; j < T; j++) {
        k.c[j] = c[j];
        k.mu[j] = (uint64_t) ((((unsigned __int128) 1) << 64) / c[j]);
        for (uint32_t i = 0; i < S; i++) k.m[j][i] = (uint32_t) prod_mod(b, S, i, c[j]);
        k.binv[j] = inv_mod(prod_mod(b, S, S, c[j]), c[j]);
        k.binvp[j] = (uint32_t) (((uint64_t) k.binv[j] << 32) / c[j]);
        k.hc[j] = (uint32_t) (prod_mod(b, S, S, 2ull * c[j]) / 2);
        k.nbc[j] = (uint32_t) ((c[j] - prod_mod(b, S, S, c[j])) % c[j]);
    }
    return NTTB200_OK;
}

// columns per thread, by measurement (profiles/r5_conv_columns_per_thread.jsonl, B200): 4 is
// faster for S <= 16 (2 costs 3-22 %), 2 for S > 16 (4 costs 6-22 %; it needs 185 registers at S = 32)
template <int S>
constexpr int conv_cols() { return S <= 16 ? 4 : 2; }

template <int S, ConvMode M>
static void conv_launch(const nttb200_rns_conv *cv, const int32_t *src, const int32_t *tin, uint64_t src_stride,
                        int32_t *out, uint64_t out_stride, size_t batch, const RnsConvConsts &k, cudaStream_t st) {
    constexpr int V = conv_cols<S>();
    const uint32_t log_chunks = cv->logn - (V == 4 ? 10 : 9);   // chunk = kC_Threads * V columns
    const uint64_t items = (uint64_t) batch << log_chunks;
    const uint64_t cap = (uint64_t) cv->sm_count * 8;
    const int grid = (int) (items < cap ? items : cap);
    rns_conv_kernel<S, V, M><<<grid, kC_Threads, 0, st>>>(
        reinterpret_cast<const uint32_t *>(src), reinterpret_cast<const uint32_t *>(tin),
        reinterpret_cast<uint32_t *>(out), src_stride, out_stride, cv->logn, cv->dst, items, log_chunks, k);
}

using ConvLaunch = void (*)(const nttb200_rns_conv *, const int32_t *, const int32_t *, uint64_t, int32_t *,
                            uint64_t, size_t, const RnsConvConsts &, cudaStream_t);

// one instantiation per S = 1..32: the phase-2 sum is straight-line code with no tail guard
template <ConvMode M, int... I>
static constexpr std::array<ConvLaunch, sizeof...(I)> conv_table(std::integer_sequence<int, I...>) {
    return {{&conv_launch<I + 1, M>...}};
}

static constexpr std::array<std::array<ConvLaunch, kConvMaxChannels>, 4> kConvLaunch = {
    conv_table<ConvMode::Fast>(std::make_integer_sequence<int, kConvMaxChannels>()),
    conv_table<ConvMode::Down>(std::make_integer_sequence<int, kConvMaxChannels>()),
    conv_table<ConvMode::Exact>(std::make_integer_sequence<int, kConvMaxChannels>()),
    conv_table<ConvMode::Scale>(std::make_integer_sequence<int, kConvMaxChannels>())};

int launch_rns_conv(const nttb200_rns_conv *cv, const int32_t *src, const int32_t *tin, uint64_t src_stride,
                    int32_t *out, uint64_t out_stride, size_t batch, ConvMode mode, bool round, uint32_t t,
                    cudaStream_t st) {
    if (batch == 0) return NTTB200_OK;
    const ConvLaunch launch = kConvLaunch[(int) mode][cv->src - 1];
    if (mode == ConvMode::Down && !round) {
        RnsConvConsts k = cv->k;
        for (int x = 0; x < kConvMaxChannels; x++) k.hb[x] = k.hc[x] = 0;
        launch(cv, src, tin, src_stride, out, out_stride, batch, k, st);
    } else if (mode == ConvMode::Scale) {
        // y'_i = [t x_i (B/b_i)^-1]_{b_i}; the target row is multiplied by t mod c_j
        RnsConvConsts k = cv->k;
        for (uint32_t i = 0; i < cv->src; i++) {
            k.w[i] = (uint32_t) mulmod64(k.w[i], t % k.b[i], k.b[i]);
            k.wp[i] = (uint32_t) (((uint64_t) k.w[i] << 32) / k.b[i]);
        }
        for (uint32_t j = 0; j < cv->dst; j++) {
            k.tc[j] = t % k.c[j];
            k.tcp[j] = (uint32_t) (((uint64_t) k.tc[j] << 32) / k.c[j]);
        }
        launch(cv, src, tin, src_stride, out, out_stride, batch, k, st);
    } else {
        launch(cv, src, tin, src_stride, out, out_stride, batch, cv->k, st);
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    NTTB200_CUDA(cudaGetLastError());
    return NTTB200_OK;
}

}  // namespace nttb200
