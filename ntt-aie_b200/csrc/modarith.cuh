// modarith.cuh -- 32-bit modular arithmetic for sm_100a.
//
// Replaces the AIE vector helpers vector_modadd / vector_modsub / vector_barrett
// (reference src/aie_core.cc:41-102; scalar spec :11-39).  The reference reduces
// every product with a 3-multiply Barrett (t=a*b; s=((t>>(w-2))*u)>>(w+2);
// c=t-s*p; one conditional subtract).  On the GPU the twiddle is a table value
// known at plan time, so the butterfly uses Shoup/Harvey multiplication with a
// precomputed companion w' = floor(w * 2^32 / q):
//     h = mulhi(x, w');  r = x*w - h*q   (mod 2^32)   =>  r in [0, 2q) for ANY
//     32-bit x and 0 <= w < q                              (IMAD.HI + 2 IMAD)
// Results are made canonical before they leave a kernel, so the outputs are the
// same integers the golden's `%` produces (src/test.cpp:48-50).
// Valid for q <= 2^30 (4q fits 32 bits) -- the golden's own domain.
#pragma once
#include <stdint.h>

namespace nttb200 {

// r = x*w mod q, lazy: result in [0, 2q).  x: any u32, w in [0,q), wp = floor(w*2^32/q).
__device__ __forceinline__ uint32_t shoup_mul_lazy(uint32_t x, uint32_t w, uint32_t wp,
                                                   uint32_t q) {
    uint32_t h = __umulhi(x, wp);
    return x * w - h * q;
}

// min(x, x - m) with unsigned wrap: conditional subtract of m for x in [0, 2m)
__device__ __forceinline__ uint32_t csub(uint32_t x, uint32_t m) {
    return min(x, x - m);
}

// canonical modular add / sub for canonical inputs (src/aie_core.cc:11-25)
__device__ __forceinline__ uint32_t add_mod(uint32_t a, uint32_t b, uint32_t q) {
    return csub(a + b, q);
}
__device__ __forceinline__ uint32_t sub_mod(uint32_t a, uint32_t b, uint32_t q) {
    return csub(a + q - b, q);
}

// canonical x*w mod q through Shoup
__device__ __forceinline__ uint32_t shoup_mul(uint32_t x, uint32_t w, uint32_t wp, uint32_t q) {
    return csub(shoup_mul_lazy(x, w, wp, q), q);
}

// t mod q for any t < 2^64, q <= 2^30, mu = floor(2^64 / q):
// t/q - 1 < t*mu/2^64 <= t/q, so qhat = floor(t*mu/2^64) is floor(t/q) or one less and the
// remainder t - qhat*q lies in [0, 2q) (computed mod 2^32, where it fits).
__device__ __forceinline__ uint32_t reduce64(uint64_t t, uint32_t q, uint64_t mu) {
    const uint64_t qhat = __umul64hi(t, mu);
    return csub((uint32_t) t - (uint32_t) qhat * q, q);
}

// General a*b mod q for two data operands (pointwise product): 64-bit product
// and a Barrett quotient estimate.  mu = floor(2^62 / q); for a,b < q <= 2^30 the
// product t < 2^60 and qhat = floor(t*mu / 2^62) is floor(t/q) or one less, so
// r = t - qhat*q lies in [0, 2q) and one conditional subtract makes it canonical.
__device__ __forceinline__ uint32_t barrett_mul(uint32_t a, uint32_t b, uint32_t q, uint64_t mu) {
    uint64_t t = (uint64_t) a * b;
    uint64_t qhat = __umul64hi(t << 2, mu);  // floor(t*4*mu / 2^64) = floor(t*mu / 2^62)
    uint32_t r = (uint32_t) t - (uint32_t) qhat * q;
    return csub(r, q);
}

// logn-bit reversal of x < 2^logn (logn >= 12): the index map of the rns_ct order
__device__ __forceinline__ uint32_t brev_n(uint32_t x, uint32_t logn) { return __brev(x) >> (32 - logn); }

}  // namespace nttb200
