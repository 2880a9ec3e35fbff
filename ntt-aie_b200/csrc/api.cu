// api.cu -- the C ABI of libnttb200.so (include/nttb200.h): plan management, the
// dispatch between the fused and the generic kernels, the host-buffer pipeline.
//
// This file is the successor of the reference host harness around one launch
// (src/test.cpp:110-190): load device image + allocate/sync buffer objects ->
// nttb200_plan_create; kernel(bo_inA, bo_root, bo_outC) + run.wait() ->
// nttb200_gs_batch / nttb200_gs_host.  There is no CPU compute path in here:
// without a usable CUDA device every compute entry point returns an error.
#include <float.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <numeric>
#include <stdexcept>
#include <vector>

#include "plan.h"

namespace nttb200 {

std::atomic<uint64_t> g_launches{0};

static std::mutex g_pool_mu;
static cudaMemPool_t g_pool[64] = {};
static std::atomic<int> g_live_plans{0};

int scratch_alloc_async(void **p, size_t bytes, cudaStream_t st) {
    int dev = 0;
    NTTB200_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return NTTB200_ERR_UNSUPPORTED;
    cudaMemPool_t pool;
    {
        std::lock_guard<std::mutex> lock(g_pool_mu);
        if (!g_pool[dev]) {
            cudaMemPoolProps props = {};
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = dev;
            NTTB200_CUDA(cudaMemPoolCreate(&g_pool[dev], &props));
            uint64_t keep = ~0ull;
            NTTB200_CUDA(cudaMemPoolSetAttribute(g_pool[dev], cudaMemPoolAttrReleaseThreshold, &keep));
        }
        pool = g_pool[dev];
    }
    NTTB200_CUDA(cudaMallocFromPoolAsync(p, bytes, pool, st));
    return NTTB200_OK;
}

static void scratch_trim_all() {
    std::lock_guard<std::mutex> lock(g_pool_mu);
    for (int d = 0; d < 64; d++) {
        if (g_pool[d]) cudaMemPoolTrimTo(g_pool[d], 0);
    }
}
static thread_local char t_err[512] = "";

int cuda_fail(cudaError_t e, const char *what) {
    snprintf(t_err, sizeof(t_err), "%s: %s (%s)", what, cudaGetErrorName(e),
             cudaGetErrorString(e));
    cudaGetLastError();  // clear the sticky-free error state
    return e == cudaErrorNoDevice || e == cudaErrorInvalidDevice ||
                   e == cudaErrorInsufficientDriver
               ? NTTB200_ERR_NO_DEVICE
               : NTTB200_ERR_CUDA;
}

int fail_msg(int status, const char *msg) {
    snprintf(t_err, sizeof(t_err), "%s", msg);
    return status;
}

static uint64_t powmod64(uint64_t b, uint64_t e, uint64_t m) {
    uint64_t r = 1 % m;
    b %= m;
    while (e) {
        if (e & 1) r = (unsigned __int128) r * b % m;
        b = (unsigned __int128) b * b % m;
        e >>= 1;
    }
    return r;
}

static uint32_t shoup_companion(uint32_t w, uint32_t q) {
    return (uint32_t) (((uint64_t) w << 32) / q);
}

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// puts the caller's current device back when a constructor that switched devices returns
struct DeviceRestore {
    int prev = -1;
    DeviceRestore() {
        if (cudaGetDevice(&prev) != cudaSuccess) {
            prev = -1;
            cudaGetLastError();
        }
    }
    ~DeviceRestore() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

static bool full_depth(const nttb200_plan *p, int stage_limit) {
    return stage_limit < 0 || stage_limit > (int) p->logn - 2;
}

}  // namespace nttb200

using namespace nttb200;

extern "C" {

/* ---------------------------------------------------------------- tables */
int nttb200_make_roots(int32_t n, int32_t *roots, int32_t p, int32_t g) {
    if (!roots || n < 1 || p < 2 || g < 0) return NTTB200_ERR_INVALID_ARG;  // p < 2^31 by type
    // src/test.cpp:137-139 (roots[0] = 1) and :27-32 (w = g^((p-1)/n), running product)
    uint64_t w = powmod64((uint64_t) g, (uint64_t) ((p - 1) / n), (uint64_t) p);
    roots[0] = 1;
    uint64_t cur = 1;
    for (int32_t i = 1; i < n; i++) {
        cur = cur * w % (uint64_t) p;
        roots[i] = (int32_t) cur;
    }
    return NTTB200_OK;
}

int nttb200_make_bitrev_table(int32_t n, int32_t *table, int32_t p, int32_t base) {
    if (!table || n < 1 || (n & (n - 1)) || p < 2 || base < 0) {
        return NTTB200_ERR_INVALID_ARG;
    }
    int logn = 0;
    while ((1 << logn) < n) logn++;
    uint64_t cur = 1 % (uint64_t) p;
    for (int32_t i = 0; i < n; i++) {
        uint32_t r = 0;
        for (int b = 0; b < logn; b++) r |= ((uint32_t) (i >> b) & 1u) << (logn - 1 - b);
        table[r] = (int32_t) cur;  // table[bitrev(i)] = base^i  <=>  table[k] = base^bitrev(k)
        cur = cur * (uint64_t) base % (uint64_t) p;
    }
    return NTTB200_OK;
}

int32_t nttb200_powmod(int32_t b, int64_t e, int32_t m) {
    if (m < 1 || e < 0 || b < 0) return -1;
    return (int32_t) powmod64((uint64_t) b, (uint64_t) e, (uint64_t) m);
}

/* ------------------------------------------------------------------ plan */
}  // extern "C"

// argument checks, device selection, plan object and the (w, w') table allocation shared by
// the two constructors; on success the plan's device is current (guard)
static int plan_begin(nttb200_plan **out, int device, uint32_t logn, uint32_t q, uint32_t flags,
                      nttb200_plan **pp) {
    if (!out) return NTTB200_ERR_INVALID_ARG;
    *out = nullptr;
    if (logn < 1 || logn > NTTB200_MAX_LOGN) return NTTB200_ERR_INVALID_ARG;
    if (flags & ~(NTTB200_ORDER_AIE_DEVICE | NTTB200_FORCE_GENERIC | NTTB200_REDUCE_INPUT |
                  NTTB200_INPUT_BITREV | NTTB200_OUTPUT_BITREV)) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if ((flags & NTTB200_ORDER_AIE_DEVICE) && (flags & (NTTB200_INPUT_BITREV | NTTB200_OUTPUT_BITREV))) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if ((flags & NTTB200_ORDER_AIE_DEVICE) && logn < 4) return NTTB200_ERR_INVALID_ARG;
    if (q < 2 || q > 0x7fffffffu) return NTTB200_ERR_MODULUS;
    // 2^30 < q < 2^31 (outside the golden's int32 domain, SURVEY 8f.4): the lazy [0,2q) /
    // [0,4q) butterflies of the register-radix kernels need 4q <= 2^32, so these moduli run
    // on the stage-pass kernels, whose intermediates are canonical (sums below 2q < 2^32)
    if (q > (1u << 30)) flags |= NTTB200_FORCE_GENERIC;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
    if (count == 0 || device < 0 || device >= count) {
        snprintf(t_err, sizeof(t_err), "device %d not available (%d CUDA devices)", device, count);
        return NTTB200_ERR_NO_DEVICE;
    }
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    nttb200_plan *p = new (std::nothrow) nttb200_plan();
    if (!p) return NTTB200_ERR_ALLOC;
    p->device = device;
    p->logn = logn;
    p->n = 1u << logn;
    p->q = q;
    p->flags = flags;
    p->mu = (uint64_t) ((((unsigned __int128) 1) << 62) / q);
    cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, device);
    // N^-1 mod q exists iff q is odd; found by the extended Euclid-free route
    // n_inv = ((q+1)/2)^logn, valid for every odd q (prime or not)
    if (q & 1u) {
        p->n_inv = (uint32_t) powmod64((uint64_t) (q + 1) / 2, logn, q);
        p->n_inv_shoup = shoup_companion(p->n_inv, q);
    }
    e = cudaMalloc(&p->d_tw, sizeof(uint2) * (size_t) p->n);
    if (e != cudaSuccess) {
        delete p;
        return e == cudaErrorMemoryAllocation ? (cudaGetLastError(), NTTB200_ERR_ALLOC)
                                              : cuda_fail(e, "cudaMalloc(table)");
    }
    *pp = p;
    return NTTB200_OK;
}

static void plan_abort(nttb200_plan *p) {
    fused_release(p);
    multi_release(p);
    tilecol_release(p);
    if (p->d_tw) cudaFree(p->d_tw);
    delete p;
}

// kernel-family layouts derived from d_tw (all built on the device)
static int plan_finish(nttb200_plan **out, nttb200_plan *p) {
    int rc = generic_prepare();
    if (rc == NTTB200_OK) rc = polymul_prepare();
    try {  // the per-family staging vectors are small (<= 64 KiB) but no exception may cross the ABI
        if (rc == NTTB200_OK && !(p->flags & NTTB200_FORCE_GENERIC)) {
            rc = fused_prepare(p);
            if (rc == NTTB200_ERR_UNSUPPORTED) rc = small_prepare(p);
            if (rc == NTTB200_OK || rc == NTTB200_ERR_UNSUPPORTED) {
                int rc2 = multi_prepare(p);
                if (rc2 != NTTB200_ERR_UNSUPPORTED) rc = rc2;
            }
            if (rc == NTTB200_ERR_UNSUPPORTED) rc = NTTB200_OK;
        }
    } catch (...) {
        rc = NTTB200_ERR_ALLOC;
    }
    if (rc != NTTB200_OK) {
        plan_abort(p);
        return rc;
    }
    g_live_plans.fetch_add(1);
    *out = p;
    return NTTB200_OK;
}

extern "C" {

int nttb200_plan_create(nttb200_plan **out, int device, uint32_t logn, uint32_t q,
                        const int32_t *table_host, uint32_t flags) {
    if (out) *out = nullptr;
    if (!table_host || logn < 1 || logn > NTTB200_MAX_LOGN) return NTTB200_ERR_INVALID_ARG;
    if (q >= 2 && q <= 0x7fffffffu) {
        const uint32_t n = 1u << logn;
        for (uint32_t i = 1; i < n; i++) {  // table[0] is never read (src/test.cpp:45: h >= 1)
            if (table_host[i] < 0 || (uint32_t) table_host[i] >= q) return NTTB200_ERR_TABLE;
        }
    }
    DeviceRestore restore;
    nttb200_plan *p = nullptr;
    int rc = plan_begin(out, device, logn, q, flags, &p);
    if (rc != NTTB200_OK) return rc;
    // ship the caller's int32 table; the Shoup companions are computed on the device
    int32_t *d_table = nullptr;
    cudaError_t e = cudaMalloc(&d_table, sizeof(int32_t) * (size_t) p->n);
    if (e == cudaSuccess) {
        e = cudaMemcpy(d_table, table_host, sizeof(int32_t) * (size_t) p->n, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) {
        rc = build_shoup_table(p, d_table);
        if (rc == NTTB200_OK) e = cudaDeviceSynchronize();
    }
    if (d_table) cudaFree(d_table);
    if (e != cudaSuccess || rc != NTTB200_OK) {
        plan_abort(p);
        if (rc != NTTB200_OK) return rc;
        return e == cudaErrorMemoryAllocation ? (cudaGetLastError(), NTTB200_ERR_ALLOC)
                                              : cuda_fail(e, "table upload");
    }
    return plan_finish(out, p);
}

int nttb200_plan_create_generated(nttb200_plan **out, int device, uint32_t logn, uint32_t q,
                                  uint32_t kind, uint32_t base, uint32_t gen_logn,
                                  uint32_t block_mult, uint32_t flags) {
    if (out) *out = nullptr;
    if (kind > NTTB200_GEN_BITREV || gen_logn < logn || gen_logn > 31 || block_mult < 1) {
        return NTTB200_ERR_INVALID_ARG;
    }
    // largest exponent: (N/2) * block_mult + N/2 - 1 must stay below 2^gen_logn
    if (logn >= 1 && logn <= NTTB200_MAX_LOGN &&
        ((uint64_t) 1 << (logn - 1)) * ((uint64_t) block_mult + 1) > ((uint64_t) 1 << gen_logn)) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if (q >= 2 && base >= q) return NTTB200_ERR_TABLE;
    DeviceRestore restore;
    nttb200_plan *p = nullptr;
    int rc = plan_begin(out, device, logn, q, flags, &p);
    if (rc != NTTB200_OK) return rc;
    rc = build_generated_table(p, kind, base, gen_logn, block_mult);
    if (rc != NTTB200_OK) {
        plan_abort(p);
        return rc;
    }
    return plan_finish(out, p);
}

int nttb200_plan_table(const nttb200_plan *p, int32_t *table_host) {
    if (!p || !table_host) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    // the w halves of the (w, w') pairs, strided copy
    NTTB200_CUDA(cudaMemcpy2D(table_host, sizeof(int32_t), p->d_tw, sizeof(uint2), sizeof(int32_t),
                              p->n, cudaMemcpyDeviceToHost));
    table_host[0] = 1;  // never read by the networks; the reference host sets roots[0] = 1
    return NTTB200_OK;
}

static void host_release(nttb200_plan *p);

int nttb200_plan_destroy(nttb200_plan *p) {
    if (!p) return NTTB200_OK;
    DeviceGuard guard(p->device);
    host_release(p);
    fused_release(p);
    multi_release(p);
    tilecol_release(p);
    if (p->d_tw) cudaFree(p->d_tw);
    delete p;
    if (g_live_plans.fetch_sub(1) == 1) scratch_trim_all();   // last plan: give the scratch pages back
    return NTTB200_OK;
}

/* -------------------------------------------------------------- hot path */
static int run_gs_core(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                       int stage_limit, cudaStream_t st);

static int run_gs(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                  int stage_limit, cudaStream_t st, bool reduce_first = false) {
    if (batch == 0) return NTTB200_OK;
    if (reduce_first || (p->flags & NTTB200_REDUCE_INPUT)) {
        // the golden's `%` on first touch (src/test.cpp:46-50): canonicalise, then in place
        int rc = launch_reduce(p, d_in, d_out, batch * p->n, st);
        if (rc != NTTB200_OK) return rc;
        d_in = d_out;
    }
    const bool in_br = p->flags & NTTB200_INPUT_BITREV, out_br = p->flags & NTTB200_OUTPUT_BITREV;
    if (in_br || out_br) {
        // fused into the N = 4096 kernel's load / store; one permutation pass elsewhere
        if (full_depth(p, stage_limit) && !(p->flags & NTTB200_FORCE_GENERIC)) {
            int rc = launch_fused_gs_bitrev(p, d_in, d_out, batch, in_br, out_br, st);
            if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
        }
        if (in_br) {
            int rc = launch_bitrev_permute(p, d_in, d_out, batch, st);
            if (rc != NTTB200_OK) return rc;
            d_in = d_out;
        }
        int rc = run_gs_core(p, d_in, d_out, batch, stage_limit, st);
        if (rc == NTTB200_OK && out_br) rc = launch_bitrev_permute(p, d_out, d_out, batch, st);
        return rc;
    }
    return run_gs_core(p, d_in, d_out, batch, stage_limit, st);
}

static int run_gs_core(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                       int stage_limit, cudaStream_t st) {
    const bool full = full_depth(p, stage_limit);
    const bool permute = full && (p->flags & NTTB200_ORDER_AIE_DEVICE);
    if (full && !(p->flags & NTTB200_FORCE_GENERIC)) {
        int rc = launch_fused_gs(p, d_in, d_out, batch, permute, st);
        if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
        if (!permute) {
            rc = launch_multi_gs(p, d_in, d_out, batch, st);
            if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
        }
        size_t done = 0;
        rc = launch_small_gs(p, d_in, d_out, batch, permute, st, &done);
        if (rc == NTTB200_OK) {
            if (done == batch) return rc;
            // ragged tail (< one 2048-coefficient block) through the generic pass
            const char *path = p->last_path;
            rc = launch_generic(p, d_in + done * p->n, d_out + done * p->n, batch - done, 0,
                                (int) p->logn, false, permute, st);
            p->last_path = path;
            return rc;
        }
        if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    }
    p->last_path = "generic_stage_pass";
    int se = full ? (int) p->logn : stage_limit + 1;
    return launch_generic(p, d_in, d_out, batch, 0, se, /*ct=*/false, permute, st);
}

int nttb200_gs_batch(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                     int stage_limit, void *stream) {
    if (!p || (batch && (!d_in || !d_out))) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    return run_gs(p, d_in, d_out, batch, stage_limit, (cudaStream_t) stream);
}

}  // extern "C"
static int ct_core(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch, int stage_limit,
                   void *stream);
extern "C" {

int nttb200_ct_batch(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                     int stage_limit, void *stream) {
    if (!p || (batch && (!d_in || !d_out))) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    if (batch == 0) return NTTB200_OK;
    if (p->flags & NTTB200_REDUCE_INPUT) {
        int rc = launch_reduce(p, d_in, d_out, batch * p->n, (cudaStream_t) stream);
        if (rc != NTTB200_OK) return rc;
        d_in = d_out;
    }
    if (p->flags & NTTB200_INPUT_BITREV) {
        int rc = launch_bitrev_permute(p, d_in, d_out, batch, (cudaStream_t) stream);
        if (rc != NTTB200_OK) return rc;
        d_in = d_out;
    }
    if (p->flags & NTTB200_OUTPUT_BITREV) {
        int rc = ct_core(p, d_in, d_out, batch, stage_limit, (cudaStream_t) stream);
        if (rc == NTTB200_OK) rc = launch_bitrev_permute(p, d_out, d_out, batch, (cudaStream_t) stream);
        return rc;
    }
    return ct_core(p, d_in, d_out, batch, stage_limit, (cudaStream_t) stream);
}

}  // extern "C"

static int ct_core(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch, int stage_limit,
                   void *stream) {
    // CT stage idx (0 = stride N/2) acts on index bit logn-1-idx
    const bool full = full_depth(p, stage_limit);
    int sb = full ? 0 : (int) p->logn - 1 - stage_limit;
    if (full && !(p->flags & NTTB200_FORCE_GENERIC)) {
        int rc = launch_multi_ct(p, d_in, d_out, batch, (cudaStream_t) stream);
        if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
        size_t done = 0;
        rc = launch_small(p, 3, d_in, nullptr, d_out, batch, (cudaStream_t) stream, &done);
        if (rc == NTTB200_OK) {
            if (done == batch) return rc;
            const char *path = p->last_path;  // ragged tail through the generic pass
            rc = launch_generic(p, d_in + done * p->n, d_out + done * p->n, batch - done, 0,
                                (int) p->logn, true, false, (cudaStream_t) stream);
            p->last_path = path;
            return rc;
        }
        if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    }
    p->last_path = "generic_stage_pass";
    return launch_generic(p, d_in, d_out, batch, sb, (int) p->logn, /*ct=*/true, false,
                          (cudaStream_t) stream);
}

extern "C" {

int nttb200_bitrev_permute(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                           void *stream) {
    if (!p || (batch && (!d_in || !d_out))) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    return launch_bitrev_permute(p, d_in, d_out, batch, (cudaStream_t) stream);
}

int nttb200_transpose(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                      int to_batch_minor, void *stream) {
    if (!p || (batch && (!d_in || !d_out || d_in == d_out))) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    return to_batch_minor ? launch_transpose(p, d_in, d_out, batch, p->n, (cudaStream_t) stream)
                          : launch_transpose(p, d_in, d_out, p->n, batch, (cudaStream_t) stream);
}

int nttb200_gs_stage_range(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t batch,
                           int stage_begin, int stage_end, void *stream) {
    if (!p || (batch && (!d_in || !d_out))) return NTTB200_ERR_INVALID_ARG;
    if (stage_begin < 0 || stage_end > (int) p->logn || stage_begin > stage_end) {
        return NTTB200_ERR_INVALID_ARG;
    }
    DeviceGuard guard(p->device);
    if (batch == 0) return NTTB200_OK;
    if (stage_begin == stage_end) {
        if (d_in != d_out && batch) {
            NTTB200_CUDA(cudaMemcpyAsync(d_out, d_in, sizeof(int32_t) * batch * p->n,
                                         cudaMemcpyDeviceToDevice, (cudaStream_t) stream));
        }
        return NTTB200_OK;
    }
    cudaStream_t st = (cudaStream_t) stream;
    // stages that pair coefficients >= 4 apart run as register-radix column passes
    if (stage_begin >= 2 && !(p->flags & NTTB200_FORCE_GENERIC) && !((uintptr_t) d_in & 15u) &&
        !((uintptr_t) d_out & 15u)) {
        int rest = stage_end - stage_begin;
        int passes = (rest + 5) / 6;
        int s0 = stage_begin;
        const int32_t *src = d_in;
        int rc = NTTB200_OK;
        for (int k = 0; k < passes && rc == NTTB200_OK; k++) {
            int take = (rest + (passes - k) - 1) / (passes - k);
            rc = launch_column_pass(p, src, d_out, batch, s0, take, st);
            src = d_out;
            s0 += take;
            rest -= take;
        }
        p->last_path = "column_passes";
        return rc;
    }
    p->last_path = "generic_stage_pass";
    return launch_generic(p, d_in, d_out, batch, stage_begin, stage_end, false, false, st);
}

int nttb200_gs_stage_range_scatter(nttb200_plan *p, int32_t *d_buf, int stage_begin, int stage_end,
                                   void *const *peer_bufs, int world, int rank, void *stream) {
    if (!p || !d_buf || !peer_bufs) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    return launch_gs_range_scatter(p, d_buf, stage_begin, stage_end, peer_bufs, world, rank,
                                   (cudaStream_t) stream);
}

static void host_release(nttb200_plan *p) {
    for (int k = 0; k < kHostStreams; k++) {
        if (p->hstream[k]) cudaStreamSynchronize(p->hstream[k]);
        if (p->d_stage[k]) cudaFree(p->d_stage[k]);
        if (p->hstream[k]) cudaStreamDestroy(p->hstream[k]);
        p->d_stage[k] = nullptr;
        p->hstream[k] = nullptr;
    }
    p->host_ready = false;
}

// staging buffers of 32 MiB each: deep enough to hide the PCIe latency, small enough that the
// first kernel starts early (measured: 46.2 GB/s each way at 32 MiB vs 44.7 at 16)
constexpr size_t kHostChunkMB = 32;

static int host_prepare(nttb200_plan *p) {
    if (p->host_ready) return NTTB200_OK;
    size_t polys = (kHostChunkMB << 20) / (sizeof(int32_t) * p->n);
    if (polys < 1) polys = 1;
    for (int k = 0; k < kHostStreams; k++) {
        cudaError_t e = cudaStreamCreateWithFlags(&p->hstream[k], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaMalloc(&p->d_stage[k], sizeof(int32_t) * polys * p->n);
        if (e != cudaSuccess) {
            host_release(p);  // nothing half-built is left behind
            return e == cudaErrorMemoryAllocation ? (cudaGetLastError(), NTTB200_ERR_ALLOC)
                                                  : cuda_fail(e, "host pipeline setup");
        }
    }
    p->stage_polys = polys;
    p->host_ready = true;
    return NTTB200_OK;
}

int nttb200_gs_host(nttb200_plan *p, const int32_t *h_in, int32_t *h_out, size_t batch,
                    int stage_limit) {
    if (!p || (batch && (!h_in || !h_out))) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    std::lock_guard<std::mutex> lock(p->host_mu);
    int rc = host_prepare(p);
    if (rc != NTTB200_OK) return rc;
    const size_t n = p->n;
    size_t done = 0;
    int k = 0;
    cudaError_t e = cudaSuccess;
    while (done < batch && rc == NTTB200_OK && e == cudaSuccess) {
        size_t polys = batch - done < p->stage_polys ? batch - done : p->stage_polys;
        cudaStream_t st = p->hstream[k];
        int32_t *d = p->d_stage[k];
        // the stream is ordered: the previous D2H of this staging buffer has been
        // queued before this H2D, so the buffer is reused safely
        e = cudaMemcpyAsync(d, h_in + done * n, sizeof(int32_t) * polys * n, cudaMemcpyHostToDevice, st);
        // host inputs are whatever the caller's harness wrote (the reference fills a[i] = i,
        // src/test.cpp:141): reduce them as the golden's `%` would; hidden behind the copies
        if (e == cudaSuccess) rc = run_gs(p, d, d, polys, stage_limit, st, /*reduce_first=*/true);
        if (e == cudaSuccess && rc == NTTB200_OK) {
            e = cudaMemcpyAsync(h_out + done * n, d, sizeof(int32_t) * polys * n, cudaMemcpyDeviceToHost,
                                st);
        }
        done += polys;
        k = (k + 1) % kHostStreams;
    }
    // always drain: no copy may still be writing h_out after this synchronous call returns
    for (int s = 0; s < kHostStreams; s++) {
        cudaError_t es = cudaStreamSynchronize(p->hstream[s]);
        if (e == cudaSuccess) e = es;
    }
    if (rc != NTTB200_OK) return rc;
    if (e != cudaSuccess) return cuda_fail(e, "nttb200_gs_host");
    return NTTB200_OK;
}

int nttb200_reduce(nttb200_plan *p, const int32_t *d_in, int32_t *d_out, size_t count,
                   void *stream) {
    if (!p || (count && (!d_in || !d_out))) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    return launch_reduce(p, d_in, d_out, count, (cudaStream_t) stream);
}

int nttb200_host_alloc(void **ptr, size_t bytes, int write_combined) {
    if (!ptr || bytes == 0) return NTTB200_ERR_INVALID_ARG;
    *ptr = nullptr;
    cudaError_t e = cudaHostAlloc(ptr, bytes,
                                  cudaHostAllocPortable |
                                      (write_combined ? cudaHostAllocWriteCombined : 0));
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return NTTB200_ERR_ALLOC;
    }
    return e == cudaSuccess ? NTTB200_OK : cuda_fail(e, "cudaHostAlloc");
}

int nttb200_host_free(void *ptr) {
    if (!ptr) return NTTB200_OK;
    cudaError_t e = cudaFreeHost(ptr);
    return e == cudaSuccess ? NTTB200_OK : cuda_fail(e, "cudaFreeHost");
}

/* ---------------------------------------------------- multiplier operators */
int nttb200_pointwise(nttb200_plan *p, const int32_t *d_a, const int32_t *d_b, int32_t *d_c,
                      size_t count, void *stream) {
    if (!p || (count && (!d_a || !d_b || !d_c))) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    return launch_pointwise(p, d_a, d_b, d_c, count, (cudaStream_t) stream);
}

int nttb200_scale(nttb200_plan *p, const int32_t *d_a, int32_t *d_c, size_t count, int32_t scalar,
                  void *stream) {
    if (!p || (count && (!d_a || !d_c))) return NTTB200_ERR_INVALID_ARG;
    if (scalar < 0 || (uint32_t) scalar >= p->q) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(p->device);
    return launch_scale(p, d_a, d_c, count, (uint32_t) scalar,
                        shoup_companion((uint32_t) scalar, p->q), (cudaStream_t) stream);
}

int nttb200_polymul_negacyclic(nttb200_plan *fwd, nttb200_plan *inv, const int32_t *d_a,
                               const int32_t *d_b, int32_t *d_c, size_t batch, void *stream) {
    if (!fwd || !inv || (batch && (!d_a || !d_b || !d_c))) return NTTB200_ERR_INVALID_ARG;
    if (fwd->logn != inv->logn || fwd->q != inv->q || fwd->device != inv->device) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if (!(fwd->q & 1u)) return NTTB200_ERR_MODULUS;  // N^-1 must exist
    if ((fwd->flags | inv->flags) & NTTB200_ORDER_AIE_DEVICE) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    DeviceGuard guard(fwd->device);
    cudaStream_t st = (cudaStream_t) stream;
    const size_t words = batch * fwd->n;
    if (fwd->logn == 12 && !((fwd->flags | inv->flags) & NTTB200_FORCE_GENERIC)) {
        // N = 4096: one kernel per product, operands and result cross HBM once (12 N bytes).
        // It declines (launching nothing) on operands that are not 16-byte aligned, a d_c that
        // is not 4-byte aligned or 2^31 tiles; the transform kernels would decline as well, so
        // the generic pipeline below serves these calls.
        int rc = launch_polymul4096(fwd, inv, d_a, d_b, d_c, batch, st);
        if (rc != NTTB200_ERR_UNSUPPORTED) return rc;
    }
    // scratch for NTT(b) (and NTT(a) when the output aliases b)
    int32_t *tmp = nullptr;
    const bool fast = fwd->logn > 12 && !((fwd->flags | inv->flags) & NTTB200_FORCE_GENERIC) &&
                      fwd->d_tw_tile && inv->d_tw_tile;
    if (fast) {
        // NTT(a), NTT(b) into scratch; pointwise product, inverse transform and the
        // N^-1 scaling in one pass over them
        {
            int rca = scratch_alloc_async((void **) &tmp, sizeof(int32_t) * words * 2, st);
            if (rca != NTTB200_OK) return rca;
        }
        int rc = launch_multi_ct(fwd, d_a, tmp, batch, st);
        if (rc == NTTB200_OK) rc = launch_multi_ct(fwd, d_b, tmp + words, batch, st);
        if (rc == NTTB200_OK) rc = launch_multi_gs_dual(inv, tmp, tmp + words, d_c, batch, st);
        cudaError_t e = cudaFreeAsync(tmp, st);
        if (rc != NTTB200_ERR_UNSUPPORTED) {
            if (rc == NTTB200_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync");
            return rc;
        }
        tmp = nullptr;  // fall through to the generic pipeline (nothing was written to d_c)
    }
    if (!((fwd->flags | inv->flags) & NTTB200_FORCE_GENERIC) && fwd->logn >= 6 && fwd->logn <= 11 &&
        fwd->d_tw_r1 && inv->d_tw_r1 && batch % ((size_t) 2048 >> fwd->logn) == 0) {
        // N = 512..2048: warp-per-block CT, CT, then pointwise + inverse + scaling in one kernel
        {
            int rca = scratch_alloc_async((void **) &tmp, sizeof(int32_t) * words * 2, st);
            if (rca != NTTB200_OK) return rca;
        }
        size_t done = 0;
        int rc = launch_small(fwd, 3, d_a, nullptr, tmp, batch, st, &done);
        if (rc == NTTB200_OK) rc = launch_small(fwd, 3, d_b, nullptr, tmp + words, batch, st, &done);
        if (rc == NTTB200_OK) rc = launch_small(inv, 2, tmp, tmp + words, d_c, batch, st, &done);
        cudaError_t e = cudaFreeAsync(tmp, st);
        if (rc != NTTB200_ERR_UNSUPPORTED) {
            if (rc == NTTB200_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync");
            return rc;
        }
        tmp = nullptr;
    }
    {
        int rca = scratch_alloc_async((void **) &tmp, sizeof(int32_t) * words, st);
        if (rca != NTTB200_OK) return rca;
    }
    int rc = launch_generic(fwd, d_b, tmp, batch, 0, (int) fwd->logn, true, false, st);
    if (rc == NTTB200_OK) rc = launch_generic(fwd, d_a, d_c, batch, 0, (int) fwd->logn, true, false, st);
    if (rc == NTTB200_OK) rc = launch_pointwise(fwd, d_c, tmp, d_c, words, st);
    if (rc == NTTB200_OK) rc = run_gs(inv, d_c, d_c, batch, -1, st);
    if (rc == NTTB200_OK) rc = launch_scale(inv, d_c, d_c, words, inv->n_inv, inv->n_inv_shoup, st);
    cudaError_t e = cudaFreeAsync(tmp, st);
    if (rc == NTTB200_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync");
    return rc;
}

/* --------------------------------------------------------------------- RNS */
}  // extern "C"

// Argument checks shared by the RNS constructors, all before any device is touched.
// `tables` (host tables) or `bases` (device-generated tables) is non-null.
static int rns_check_args(nttb200_rns_plan **out, uint32_t logn, uint32_t limbs, const uint32_t *q,
                          const int32_t *const *tables, const uint32_t *bases, uint32_t flags) {
    if (!out) return NTTB200_ERR_INVALID_ARG;
    *out = nullptr;
    if (!q || (!tables && !bases) || limbs < 1 || limbs > 32 || flags != 0) return NTTB200_ERR_INVALID_ARG;
    if (logn < 1 || logn > NTTB200_MAX_LOGN) return NTTB200_ERR_INVALID_ARG;
    if (logn < 12 || logn > 16) return NTTB200_ERR_UNSUPPORTED;
    if (tables) {
        for (uint32_t l = 0; l < limbs; l++) {
            if (!tables[l]) return NTTB200_ERR_INVALID_ARG;
        }
    }
    // the sub-plans' own checks, for every channel before the first one reaches the device
    for (uint32_t l = 0; l < limbs; l++) {
        if (q[l] < 2 || q[l] > 0x7fffffffu) return NTTB200_ERR_MODULUS;
        if (bases && bases[l] >= q[l]) return NTTB200_ERR_TABLE;
        for (uint32_t i = 1; tables && i < (1u << logn); i++) {
            if (tables[l][i] < 0 || (uint32_t) tables[l][i] >= q[l]) return NTTB200_ERR_TABLE;
        }
    }
    return NTTB200_OK;
}

// One sub-plan per channel exists: concatenate their tile tables ([L][G][32][65]), for
// N > 4096 their (w, w') tables ([L][N]), and derive the per-channel constants.
static int rns_plan_finish(nttb200_rns_plan *rp) {
    const uint32_t limbs = rp->limbs;
    for (nttb200_plan *sp : rp->sub) {
        if (!sp->d_tw_tile) return NTTB200_ERR_UNSUPPORTED;   // q > 2^30: no tile kernels
    }
    DeviceGuard guard(rp->device);
    rp->sm_count = rp->sub[0]->sm_count;
    const size_t tile_words = (size_t) kRnsTwTile << (rp->logn - 12), n = (size_t) 1 << rp->logn;
    NTTB200_CUDA(cudaMalloc(&rp->d_tw_tile, sizeof(uint4) * tile_words * limbs));
    if (rp->logn > 12) NTTB200_CUDA(cudaMalloc(&rp->d_tw, sizeof(uint2) * n * limbs));
    try {
        for (uint32_t l = 0; l < limbs; l++) {
            const nttb200_plan *sp = rp->sub[l];
            NTTB200_CUDA(cudaMemcpy(rp->d_tw_tile + l * tile_words, sp->d_tw_tile, sizeof(uint4) * tile_words,
                                    cudaMemcpyDeviceToDevice));
            if (rp->d_tw) {
                NTTB200_CUDA(cudaMemcpy(rp->d_tw + l * n, sp->d_tw, sizeof(uint2) * n,
                                        cudaMemcpyDeviceToDevice));
            }
            uint4 pc = make_uint4(sp->q, 0, 0, 0), ps = pc;
            if (sp->q & 1u) {
                pc.y = inv_mod_2_32(sp->q);
                uint64_t sc = ((uint64_t) sp->n_inv << 32) % sp->q;
                pc.z = (uint32_t) sc;
                pc.w = (uint32_t) ((sc << 32) / sp->q);
                ps = make_uint4(sp->q, pc.y, sp->n_inv, sp->n_inv_shoup);
            }
            rp->pos.push_back(pc);
            rp->pos_scaled.push_back(ps);
        }
    } catch (...) {
        return NTTB200_ERR_ALLOC;
    }
    return NTTB200_OK;
}

// make_sub(l, &sp) builds channel l's sub-plan (host table or device-generated)
template <class MakeSub>
static int rns_plan_build(nttb200_rns_plan **out, int device, uint32_t logn, uint32_t limbs,
                          MakeSub make_sub) {
    DeviceRestore restore;
    nttb200_rns_plan *rp = new (std::nothrow) nttb200_rns_plan();
    if (!rp) return NTTB200_ERR_ALLOC;
    rp->device = device;
    rp->logn = logn;
    rp->limbs = limbs;
    int rc = NTTB200_OK;
    try {
        rp->sub.reserve(limbs);
    } catch (...) {
        rc = NTTB200_ERR_ALLOC;
    }
    for (uint32_t l = 0; l < limbs && rc == NTTB200_OK; l++) {
        nttb200_plan *sp = nullptr;
        rc = make_sub(l, &sp);
        if (rc == NTTB200_OK) rp->sub.push_back(sp);   // capacity reserved: does not throw
    }
    if (rc == NTTB200_OK) rc = rns_plan_finish(rp);
    if (rc != NTTB200_OK) {
        nttb200_rns_plan_destroy(rp);
        return rc;
    }
    *out = rp;
    return NTTB200_OK;
}

extern "C" {

int nttb200_rns_plan_create_logn(nttb200_rns_plan **out, int device, uint32_t logn, uint32_t limbs,
                                 const uint32_t *q, const int32_t *const *tables_host, uint32_t flags) {
    if (out) *out = nullptr;
    if (!tables_host) return NTTB200_ERR_INVALID_ARG;
    int rc = rns_check_args(out, logn, limbs, q, tables_host, nullptr, flags);
    if (rc != NTTB200_OK) return rc;
    return rns_plan_build(out, device, logn, limbs, [&](uint32_t l, nttb200_plan **sp) {
        return nttb200_plan_create(sp, device, logn, q[l], tables_host[l], 0);
    });
}

int nttb200_rns_plan_create(nttb200_rns_plan **out, int device, uint32_t limbs, const uint32_t *q,
                            const int32_t *const *tables_host, uint32_t flags) {
    return nttb200_rns_plan_create_logn(out, device, 12, limbs, q, tables_host, flags);
}

int nttb200_rns_plan_create_generated(nttb200_rns_plan **out, int device, uint32_t logn, uint32_t limbs,
                                      const uint32_t *q, uint32_t kind, const uint32_t *bases,
                                      uint32_t flags) {
    if (out) *out = nullptr;
    if (!bases || kind > NTTB200_GEN_BITREV) return NTTB200_ERR_INVALID_ARG;
    int rc = rns_check_args(out, logn, limbs, q, nullptr, bases, flags);
    if (rc != NTTB200_OK) return rc;
    return rns_plan_build(out, device, logn, limbs, [&](uint32_t l, nttb200_plan **sp) {
        return nttb200_plan_create_generated(sp, device, logn, q[l], kind, bases[l], logn, 1, 0);
    });
}

int nttb200_rns_plan_destroy(nttb200_rns_plan *rp) {
    if (!rp) return NTTB200_OK;
    {
        DeviceGuard guard(rp->device);
        if (rp->d_tw_tile) cudaFree(rp->d_tw_tile);
        if (rp->d_tw) cudaFree(rp->d_tw);
    }
    for (nttb200_plan *sp : rp->sub) nttb200_plan_destroy(sp);
    delete rp;
    return NTTB200_OK;
}

static int rns_run(nttb200_rns_plan *rp, int kind, const int32_t *d_a, const int32_t *d_b,
                   int32_t *d_out, size_t batch, void *stream) {
    if (!rp || (batch && (!d_a || !d_out))) return NTTB200_ERR_INVALID_ARG;
    DeviceGuard guard(rp->device);
    return rns_launch(rp, kind, d_a, d_b, d_out, batch, (cudaStream_t) stream);
}

int nttb200_rns_gs_batch(nttb200_rns_plan *rp, const int32_t *d_in, int32_t *d_out, size_t batch,
                         void *stream) {
    return rns_run(rp, 0, d_in, nullptr, d_out, batch, stream);
}

int nttb200_rns_ct_batch(nttb200_rns_plan *rp, const int32_t *d_in, int32_t *d_out, size_t batch,
                         void *stream) {
    return rns_run(rp, 1, d_in, nullptr, d_out, batch, stream);
}

int nttb200_rns_polymul_negacyclic(nttb200_rns_plan *fwd, nttb200_rns_plan *inv, const int32_t *d_a,
                                   const int32_t *d_b, int32_t *d_c, size_t batch, void *stream) {
    if (!fwd || !inv || (batch && (!d_a || !d_b || !d_c))) return NTTB200_ERR_INVALID_ARG;
    if (fwd->limbs != inv->limbs || fwd->device != inv->device || fwd->logn != inv->logn) {
        return NTTB200_ERR_INVALID_ARG;
    }
    for (uint32_t l = 0; l < fwd->limbs; l++) {
        if (fwd->pos[l].x != inv->pos[l].x) return NTTB200_ERR_INVALID_ARG;
        if (!(fwd->pos[l].x & 1u)) return NTTB200_ERR_MODULUS;
    }
    if (batch == 0) return NTTB200_OK;
    // N > 4096: the output is written by the tile pass's vector stores, so it must be aligned
    // like the operands; checked here so that nothing runs on an unaligned request
    if (fwd->logn > 12 && (((uintptr_t) d_a | (uintptr_t) d_b | (uintptr_t) d_c) & 15u)) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    DeviceGuard guard(fwd->device);
    cudaStream_t st = (cudaStream_t) stream;
    // N = 4096, one kernel per channel: both operands enter the SM once, the product leaves once
    // (12 N bytes per channel product instead of 28 N through the scratch buffers below).  It
    // declines for the first channel already (launching nothing) where the transform kernels
    // would decline as well: unaligned buffers, 2^31 tiles.
    if (fwd->logn == 12) {
        int rc = NTTB200_OK;
        for (uint32_t l = 0; l < fwd->limbs && rc == NTTB200_OK; l++) {
            rc = launch_polymul4096_strided(fwd->sub[l], inv->sub[l], d_a, d_b, d_c, batch, fwd->limbs, l, st);
        }
        return rc;
    }
    // N > 4096: CT(a), CT(b) into scratch (column pass + tile pass each); the DUAL tile pass
    // multiplies them at load and scales by N^-1 at the store, then the GS column pass
    if (batch > 0xffffffffull || ((uint64_t) batch * fwd->limbs << (fwd->logn - 12)) > 0x7fffffffull) {
        return NTTB200_ERR_UNSUPPORTED;   // the tile kernels count tiles in 31 bits
    }
    const size_t words = (batch * fwd->limbs) << fwd->logn;
    int32_t *tmp = nullptr;
    {
        int rca = scratch_alloc_async((void **) &tmp, sizeof(int32_t) * words * 2, st);
        if (rca != NTTB200_OK) return rca;
    }
    int rc = rns_run(fwd, 1, d_a, nullptr, tmp, batch, stream);
    if (rc == NTTB200_OK) rc = rns_run(fwd, 1, d_b, nullptr, tmp + words, batch, stream);
    if (rc == NTTB200_OK) rc = rns_run(inv, 2, tmp, tmp + words, d_c, batch, stream);
    cudaError_t e = cudaFreeAsync(tmp, st);
    if (rc == NTTB200_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync");
    return rc;
}

int nttb200_rns_gs_scaled_batch(nttb200_rns_plan *rp, const int32_t *d_in, int32_t *d_out, size_t batch,
                                void *stream) {
    if (!rp || (batch && (!d_in || !d_out))) return NTTB200_ERR_INVALID_ARG;
    for (uint32_t l = 0; l < rp->limbs; l++) {
        if (!(rp->pos[l].x & 1u)) return NTTB200_ERR_MODULUS;   // N^-1 must exist
    }
    return rns_run(rp, 3, d_in, nullptr, d_out, batch, stream);
}

}  // extern "C"

// Evaluation-domain operators: [lo, hi) byte ranges of the buffers, for the aliasing rules
struct ByteRange {
    uintptr_t lo, hi;
    bool overlaps(const ByteRange &o) const { return lo < o.hi && o.lo < hi; }
};

static ByteRange byte_range(const void *p, uint64_t words) {
    return {(uintptr_t) p, (uintptr_t) p + words * sizeof(int32_t)};
}

static bool aligned16(const void *a, const void *b, const void *c) {
    return !(((uintptr_t) a | (uintptr_t) b | (uintptr_t) c) & 15u);
}

// words of `polys` polynomials of the plan, or 0 when the byte count would not fit 62 bits
static uint64_t rns_words(const nttb200_rns_plan *rp, uint64_t polys) {
    const uint64_t per = (uint64_t) rp->limbs << rp->logn;
    return polys > ((uint64_t) 1 << 60) / per ? 0 : polys * per;
}

extern "C" {

int nttb200_rns_pointwise(nttb200_rns_plan *rp, uint32_t op, const int32_t *d_a, const int32_t *d_b,
                          int32_t *d_c, size_t batch, size_t b_batch, void *stream) {
    if (!rp || (batch && (!d_a || !d_b || !d_c))) return NTTB200_ERR_INVALID_ARG;
    if (op > NTTB200_RNS_MUL || (b_batch != batch && b_batch != 1)) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    const uint64_t words = rns_words(rp, batch);
    if (!words) return NTTB200_ERR_UNSUPPORTED;
    const bool bcast = b_batch != batch;   // b_batch == 1 < batch
    const ByteRange a = byte_range(d_a, words), c = byte_range(d_c, words);
    const ByteRange b = byte_range(d_b, bcast ? words / batch : words);
    if ((c.overlaps(a) && d_c != d_a) || (c.overlaps(b) && (d_c != d_b || bcast))) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if (!aligned16(d_a, d_b, d_c)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(rp->device);
    return launch_rns_stream(rp, op, d_a, d_b, d_c, batch, bcast, nullptr, (cudaStream_t) stream);
}

int nttb200_rns_scale(nttb200_rns_plan *rp, const int32_t *d_a, int32_t *d_c, size_t batch,
                      const uint32_t *scalars, void *stream) {
    if (!rp || !scalars || (batch && (!d_a || !d_c))) return NTTB200_ERR_INVALID_ARG;
    for (uint32_t l = 0; l < rp->limbs; l++) {
        if (scalars[l] >= rp->pos[l].x) return NTTB200_ERR_INVALID_ARG;
    }
    if (batch == 0) return NTTB200_OK;
    const uint64_t words = rns_words(rp, batch);
    if (!words) return NTTB200_ERR_UNSUPPORTED;
    if (d_c != d_a && byte_range(d_c, words).overlaps(byte_range(d_a, words))) return NTTB200_ERR_INVALID_ARG;
    if (!aligned16(d_a, d_a, d_c)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(rp->device);
    return launch_rns_stream(rp, 3, d_a, nullptr, d_c, batch, false, scalars, (cudaStream_t) stream);
}

int nttb200_rns_dot(nttb200_rns_plan *rp, const int32_t *d_a, const int32_t *d_w, int32_t *d_c, uint32_t terms,
                    size_t batch, size_t w_batch, int accumulate, void *stream) {
    if (!rp || (batch && (!d_a || !d_w || !d_c))) return NTTB200_ERR_INVALID_ARG;
    if (terms < 1 || terms > 64 || (w_batch != batch && w_batch != 1)) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    const uint64_t words = rns_words(rp, batch), a_words = rns_words(rp, (uint64_t) terms * batch);
    if (!words || !a_words) return NTTB200_ERR_UNSUPPORTED;
    const bool w_shared = w_batch != batch;   // w_batch == 1 < batch
    const ByteRange c = byte_range(d_c, words);
    if (c.overlaps(byte_range(d_a, a_words)) ||
        c.overlaps(byte_range(d_w, w_shared ? a_words / batch : a_words))) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if (!aligned16(d_a, d_w, d_c)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(rp->device);
    return launch_rns_dot(rp, d_a, d_w, d_c, terms, batch, w_shared, accumulate != 0, (cudaStream_t) stream);
}

int nttb200_rns_automorphism(nttb200_rns_plan *rp, const int32_t *d_in, int32_t *d_out, size_t batch,
                             const uint32_t *galois, uint32_t count, uint32_t domain, void *stream) {
    if (!rp || !galois || count < 1 || count > kAutoMaxElems || domain > NTTB200_AUTO_EVAL) {
        return NTTB200_ERR_INVALID_ARG;
    }
    for (uint32_t c = 0; c < count; c++) {
        if (!(galois[c] & 1u) || galois[c] >= (2u << rp->logn)) return NTTB200_ERR_INVALID_ARG;
    }
    if (batch && (!d_in || !d_out)) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    const uint64_t words = rns_words(rp, batch), out_words = rns_words(rp, (uint64_t) count * batch);
    if (!words || !out_words) return NTTB200_ERR_UNSUPPORTED;
    if (byte_range(d_out, out_words).overlaps(byte_range(d_in, words))) return NTTB200_ERR_INVALID_ARG;
    if (!aligned16(d_in, d_in, d_out)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(rp->device);
    return launch_rns_automorph(rp, d_in, d_out, batch, galois, count, domain == NTTB200_AUTO_EVAL,
                                (cudaStream_t) stream);
}

/* ------------------------------------------------------- RNS basis conversion */
int nttb200_rns_conv_create(nttb200_rns_conv **conv, const nttb200_rns_plan *from, const nttb200_rns_plan *to,
                            uint32_t flags) {
    if (!conv) return NTTB200_ERR_INVALID_ARG;
    *conv = nullptr;
    if (!from || !to || flags != 0) return NTTB200_ERR_INVALID_ARG;
    if (from->device != to->device || from->logn != to->logn) return NTTB200_ERR_INVALID_ARG;
    nttb200_rns_conv *cv = new (std::nothrow) nttb200_rns_conv();
    if (!cv) return NTTB200_ERR_ALLOC;
    cv->device = from->device;
    cv->logn = from->logn;
    cv->src = from->limbs;
    cv->dst = to->limbs;
    cv->sm_count = from->sm_count;
    uint32_t b[kConvMaxChannels], c[kConvMaxChannels];
    for (uint32_t i = 0; i < cv->src; i++) b[i] = from->pos[i].x;
    for (uint32_t j = 0; j < cv->dst; j++) c[j] = to->pos[j].x;
    int rc;
    try {
        rc = rns_conv_prepare(cv, b, c);
    } catch (...) {
        rc = NTTB200_ERR_ALLOC;
    }
    if (rc != NTTB200_OK) {
        delete cv;
        return rc;
    }
    *conv = cv;
    return NTTB200_OK;
}

int nttb200_rns_conv_destroy(nttb200_rns_conv *conv) {
    delete conv;
    return NTTB200_OK;
}

}  // extern "C"

// Word offsets of the rows of an equal-stride pair of views overlap: input row b holds
// [I + b P, I + b P + SA), output row b' holds [O + b' P, O + b' P + TA) (bytes, P > 0, every
// row shorter than P).  They share a byte iff some k = b' - b in (-batch, batch) has
// I - O - TA < k P < I - O + SA.
static bool rows_overlap(uintptr_t in, uint64_t sa, uintptr_t out, uint64_t ta, uint64_t period, uint64_t batch) {
    const int64_t d = (int64_t) (in - out), p = (int64_t) period, lo = d - (int64_t) ta;
    int64_t k = (lo >= 0 ? lo / p : -((-lo + p - 1) / p)) + 1;   // floor(lo / p) + 1: least k with k P > lo
    if (k < 1 - (int64_t) batch) k = 1 - (int64_t) batch;
    return k <= (int64_t) batch - 1 && k * p < d + (int64_t) sa;
}

// The strided conversions (base_convert, base_convert_exact): null pointers, strides (0: dense),
// extents, the row overlap and the alignment are checked in that order, then one launch.
static int conv_strided(nttb200_rns_conv *conv, const int32_t *d_in, size_t in_stride, int32_t *d_out,
                        size_t out_stride, size_t batch, ConvMode mode, void *stream) {
    if (!conv || (batch && (!d_in || !d_out))) return NTTB200_ERR_INVALID_ARG;
    const uint64_t n = (uint64_t) 1 << conv->logn;
    const uint64_t s_words = conv->src * n, t_words = conv->dst * n;
    const uint64_t is = in_stride ? in_stride : s_words, os = out_stride ? out_stride : t_words;
    if (is % n || is < s_words || os % n || os < t_words) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    // extents, or 0 when the byte count would not fit 62 bits
    const uint64_t lim = (uint64_t) 1 << 60;
    if (is > lim || os > lim || batch - 1 > (lim - s_words) / is || batch - 1 > (lim - t_words) / os) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    const uintptr_t in = (uintptr_t) d_in, out = (uintptr_t) d_out;
    const bool overlap = is == os ? rows_overlap(in, 4 * s_words, out, 4 * t_words, 4 * is, batch)
                                  : byte_range(d_in, (batch - 1) * is + s_words)
                                        .overlaps(byte_range(d_out, (batch - 1) * os + t_words));
    if (overlap) return NTTB200_ERR_INVALID_ARG;
    if (!aligned16(d_in, d_in, d_out)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(conv->device);
    return launch_rns_conv(conv, d_in, nullptr, is, d_out, os, batch, mode, false, 0, (cudaStream_t) stream);
}

// The operations on [batch][T+S][N] (mod_down, scale_round; the source rows follow the T target
// rows of each polynomial): null pointers and a rejected option (bad_option), extents, overlap
// and alignment are checked in that order, then one launch.
static int conv_down(nttb200_rns_conv *conv, const int32_t *d_in, int32_t *d_out, size_t batch, bool bad_option,
                     ConvMode mode, bool round, uint32_t t, void *stream) {
    if (!conv || (batch && (!d_in || !d_out)) || bad_option) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    const uint64_t n = (uint64_t) 1 << conv->logn;
    const uint64_t row = (conv->src + conv->dst) * n, t_words = conv->dst * n;
    if (batch > ((uint64_t) 1 << 60) / row) return NTTB200_ERR_UNSUPPORTED;
    if (byte_range(d_in, batch * row).overlaps(byte_range(d_out, batch * t_words))) return NTTB200_ERR_INVALID_ARG;
    if (!aligned16(d_in, d_in, d_out)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(conv->device);
    return launch_rns_conv(conv, d_in + t_words, d_in, row, d_out, t_words, batch, mode, round, t,
                           (cudaStream_t) stream);
}

extern "C" {

int nttb200_rns_base_convert(nttb200_rns_conv *conv, const int32_t *d_in, size_t in_stride, int32_t *d_out,
                             size_t out_stride, size_t batch, void *stream) {
    return conv_strided(conv, d_in, in_stride, d_out, out_stride, batch, ConvMode::Fast, stream);
}

int nttb200_rns_base_convert_exact(nttb200_rns_conv *conv, const int32_t *d_in, size_t in_stride, int32_t *d_out,
                                   size_t out_stride, size_t batch, void *stream) {
    return conv_strided(conv, d_in, in_stride, d_out, out_stride, batch, ConvMode::Exact, stream);
}

int nttb200_rns_mod_down(nttb200_rns_conv *conv, const int32_t *d_in, int32_t *d_out, size_t batch, uint32_t flags,
                         void *stream) {
    return conv_down(conv, d_in, d_out, batch, (flags & ~NTTB200_RNS_ROUND) != 0, ConvMode::Down,
                     (flags & NTTB200_RNS_ROUND) != 0, 0, stream);
}

int nttb200_rns_scale_round(nttb200_rns_conv *conv, const int32_t *d_in, int32_t *d_out, size_t batch, uint32_t t,
                            void *stream) {
    return conv_down(conv, d_in, d_out, batch, t == 0, ConvMode::Scale, false, t, stream);
}

/* ------------------------------------------------------- CKKS slot encoding */
int nttb200_ckks_encoder_create(nttb200_ckks_encoder **enc, const nttb200_rns_plan *plan, uint32_t flags) {
    if (!enc) return NTTB200_ERR_INVALID_ARG;
    *enc = nullptr;
    if (!plan || flags != 0) return NTTB200_ERR_INVALID_ARG;
    nttb200_ckks_encoder *e = new (std::nothrow) nttb200_ckks_encoder();
    if (!e) return NTTB200_ERR_ALLOC;
    e->device = plan->device;
    e->logn = plan->logn;
    e->limbs = plan->limbs;
    e->sm_count = plan->sm_count;
    for (uint32_t l = 0; l < e->limbs; l++) {
        e->k.q[l] = plan->pos[l].x;
        e->k.mu[l] = (uint64_t) ((((unsigned __int128) 1) << 64) / e->k.q[l]);
    }
    int rc;
    {
        DeviceGuard guard(e->device);
        try {
            rc = ckks_prepare(e);
        } catch (...) {
            rc = NTTB200_ERR_ALLOC;
        }
        if (rc != NTTB200_OK) ckks_release(e);
    }
    if (rc != NTTB200_OK) {
        delete e;
        return rc;
    }
    *enc = e;
    return NTTB200_OK;
}

int nttb200_ckks_encoder_destroy(nttb200_ckks_encoder *enc) {
    if (!enc) return NTTB200_OK;
    {
        DeviceGuard guard(enc->device);
        ckks_release(enc);
    }
    delete enc;
    return NTTB200_OK;
}

static bool bad_scale(double scale) { return !(scale > 0.0 && scale <= DBL_MAX); }

int nttb200_ckks_encode(nttb200_ckks_encoder *enc, const void *d_slots, double scale, int32_t *d_out, size_t batch,
                        void *stream) {
    if (!enc || bad_scale(scale) || (batch && (!d_slots || !d_out))) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    const uint64_t n = (uint64_t) 1 << (enc->logn - 1), row = (uint64_t) enc->limbs << enc->logn;
    if (batch > ((uint64_t) 1 << 60) / row) return NTTB200_ERR_UNSUPPORTED;
    if (byte_range(d_out, batch * row).overlaps(byte_range(d_slots, 4 * batch * n))) return NTTB200_ERR_INVALID_ARG;
    if (!aligned16(d_slots, d_slots, d_out)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(enc->device);
    return launch_ckks_encode(enc, static_cast<const double2 *>(d_slots), scale, d_out, batch, (cudaStream_t) stream);
}

int nttb200_ckks_decode(nttb200_ckks_encoder *enc, const int32_t *d_in, size_t in_stride, uint32_t channels,
                        double scale, void *d_slots, size_t batch, void *stream) {
    if (!enc || bad_scale(scale) || (batch && (!d_in || !d_slots))) return NTTB200_ERR_INVALID_ARG;
    const uint64_t N = (uint64_t) 1 << enc->logn, c_words = channels * N;
    if (channels < 1 || channels > std::min<uint32_t>(enc->limbs, kCkksMaxDecode)) return NTTB200_ERR_INVALID_ARG;
    const uint64_t is = in_stride ? in_stride : c_words;
    if (is % N || is < c_words) return NTTB200_ERR_INVALID_ARG;
    CkksDecConsts k;
    const int rc = ckks_decode_consts(enc, channels, scale, &k);
    if (rc != NTTB200_OK) return rc;
    if (batch == 0) return NTTB200_OK;
    if (is > ((uint64_t) 1 << 60) || batch - 1 > (((uint64_t) 1 << 60) - c_words) / is ||
        batch > ((uint64_t) 1 << 60) / (2 * N)) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    if (byte_range(d_in, (batch - 1) * is + c_words).overlaps(byte_range(d_slots, 2 * N * batch))) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if (!aligned16(d_in, d_in, d_slots)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(enc->device);
    return launch_ckks_decode(enc, d_in, is, channels, k, static_cast<double2 *>(d_slots), batch,
                              (cudaStream_t) stream);
}

/* ------------------------------------------------------ packed integer slots */
// trial division: t < 2^30, so divisors up to 2^15
static bool is_prime(uint32_t t) {
    if (t < 2) return false;
    for (uint32_t d = 2; d * d <= t; d++) {
        if (t % d == 0) return false;
    }
    return true;
}

int nttb200_packed_encoder_create(nttb200_packed_encoder **enc, const nttb200_rns_plan *plan, uint32_t t,
                                  uint32_t flags) {
    if (!enc) return NTTB200_ERR_INVALID_ARG;
    *enc = nullptr;
    if (!plan || flags != 0) return NTTB200_ERR_INVALID_ARG;
    if (t >= (1u << 30) || !is_prime(t) || (t - 1) % (2u << plan->logn)) return NTTB200_ERR_MODULUS;
    for (uint32_t l = 0; l < plan->limbs; l++) {
        if (plan->pos[l].x % t == 0) return NTTB200_ERR_MODULUS;
    }
    nttb200_packed_encoder *e = new (std::nothrow) nttb200_packed_encoder();
    if (!e) return NTTB200_ERR_ALLOC;
    e->device = plan->device;
    e->logn = plan->logn;
    e->limbs = plan->limbs;
    e->sm_count = plan->sm_count;
    e->k.t = t;
    for (uint32_t l = 0; l < e->limbs; l++) e->k.q[l] = plan->pos[l].x;
    int rc;
    {
        DeviceGuard guard(e->device);
        try {
            rc = packed_prepare(e);
        } catch (...) {
            rc = NTTB200_ERR_ALLOC;
        }
        if (rc != NTTB200_OK) packed_release(e);
    }
    if (rc != NTTB200_OK) {
        delete e;
        return rc;
    }
    *enc = e;
    return NTTB200_OK;
}

int nttb200_packed_encoder_destroy(nttb200_packed_encoder *enc) {
    if (!enc) return NTTB200_OK;
    {
        DeviceGuard guard(enc->device);
        packed_release(enc);
    }
    delete enc;
    return NTTB200_OK;
}

// Shared checks of encode and decode after the mode / flag: in_words and out_words per polynomial.
static int packed_args(const nttb200_packed_encoder *enc, const int32_t *in, uint64_t in_words, const int32_t *out,
                       uint64_t out_words, size_t batch) {
    if (batch && (!in || !out)) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    if (batch > (0x7fffffffull >> (enc->logn - 12))) return NTTB200_ERR_UNSUPPORTED;   // the transforms mod t
    if (byte_range(in, batch * in_words).overlaps(byte_range(out, batch * out_words))) return NTTB200_ERR_INVALID_ARG;
    if (!aligned16(in, in, out)) return NTTB200_ERR_UNSUPPORTED;
    return NTTB200_OK;
}

int nttb200_packed_encode(nttb200_packed_encoder *enc, const int32_t *d_slots, uint32_t mode, int32_t *d_out,
                          size_t batch, void *stream) {
    if (!enc || mode > NTTB200_PACK_CENTRED) return NTTB200_ERR_INVALID_ARG;
    const uint64_t N = (uint64_t) 1 << enc->logn;
    const int rc = packed_args(enc, d_slots, N, d_out, enc->limbs * N, batch);
    if (rc != NTTB200_OK || batch == 0) return rc;
    DeviceGuard guard(enc->device);
    return launch_packed_encode(enc, d_slots, mode == NTTB200_PACK_CENTRED, d_out, batch, (cudaStream_t) stream);
}

int nttb200_packed_decode(nttb200_packed_encoder *enc, const int32_t *d_in, uint32_t flags, int32_t *d_slots,
                          size_t batch, void *stream) {
    if (!enc || (flags & ~NTTB200_PACK_CENTRED)) return NTTB200_ERR_INVALID_ARG;
    const uint64_t N = (uint64_t) 1 << enc->logn;
    const int rc = packed_args(enc, d_in, N, d_slots, N, batch);
    if (rc != NTTB200_OK || batch == 0) return rc;
    DeviceGuard guard(enc->device);
    return launch_packed_decode(enc, d_in, flags == NTTB200_PACK_CENTRED, d_slots, batch, (cudaStream_t) stream);
}

/* ------------------------------------------------------- hybrid key switching */
int nttb200_rns_keyswitch_create(nttb200_rns_keyswitch **ks, const nttb200_rns_plan *qp_fwd,
                                 const nttb200_rns_plan *qp_inv, uint32_t q_limbs, uint32_t alpha, uint32_t flags) {
    if (!ks) return NTTB200_ERR_INVALID_ARG;
    *ks = nullptr;
    if (!qp_fwd || !qp_inv || flags != 0) return NTTB200_ERR_INVALID_ARG;
    if (qp_fwd->logn != qp_inv->logn || qp_fwd->device != qp_inv->device || qp_fwd->limbs != qp_inv->limbs) {
        return NTTB200_ERR_INVALID_ARG;
    }
    const uint32_t LK = qp_fwd->limbs;
    if (q_limbs == 0 || q_limbs >= LK || alpha == 0 || alpha > q_limbs) return NTTB200_ERR_INVALID_ARG;
    for (uint32_t l = 0; l < LK; l++) {
        if (qp_fwd->pos[l].x != qp_inv->pos[l].x) return NTTB200_ERR_INVALID_ARG;
    }
    for (uint32_t l = 0; l < LK; l++) {
        const uint32_t q = qp_fwd->pos[l].x;
        if (!(q & 1u)) return NTTB200_ERR_MODULUS;   // N^-1 must exist
        for (uint32_t m = l + 1; m < LK; m++) {
            if (std::gcd(q, qp_fwd->pos[m].x) != 1) return NTTB200_ERR_MODULUS;
        }
    }
    nttb200_rns_keyswitch *k = new (std::nothrow) nttb200_rns_keyswitch();
    if (!k) return NTTB200_ERR_ALLOC;
    k->device = qp_fwd->device;
    k->logn = qp_fwd->logn;
    k->q_limbs = q_limbs;
    k->limbs = LK;
    k->alpha = alpha;
    k->dnum = (q_limbs + alpha - 1) / alpha;
    k->sm_count = qp_fwd->sm_count;
    int rc;
    {
        DeviceGuard guard(k->device);
        try {
            rc = keyswitch_prepare(k, qp_fwd, qp_inv);
        } catch (...) {
            rc = NTTB200_ERR_ALLOC;
        }
        if (rc != NTTB200_OK) keyswitch_release(k);
    }
    if (rc != NTTB200_OK) {
        delete k;
        return rc;
    }
    *ks = k;
    return NTTB200_OK;
}

int nttb200_rns_keyswitch_destroy(nttb200_rns_keyswitch *ks) {
    if (!ks) return NTTB200_OK;
    {
        DeviceGuard guard(ks->device);
        keyswitch_release(ks);
    }
    delete ks;
    return NTTB200_OK;
}

int nttb200_rns_keyswitch_apply(nttb200_rns_keyswitch *ks, const int32_t *d_in, size_t in_stride, const int32_t *d_keys,
                          const uint32_t *galois, uint32_t count, int32_t *d_out, size_t batch, uint32_t flags,
                          void *stream) {
    if (!ks || !galois || count < 1 || count > kAutoMaxElems) return NTTB200_ERR_INVALID_ARG;
    if (flags & ~(NTTB200_KS_COEFF_IN | NTTB200_KS_COEFF_OUT)) return NTTB200_ERR_INVALID_ARG;
    for (uint32_t c = 0; c < count; c++) {
        if (!(galois[c] & 1u) || galois[c] >= (2u << ks->logn)) return NTTB200_ERR_INVALID_ARG;
    }
    if (batch && (!d_in || !d_keys || !d_out)) return NTTB200_ERR_INVALID_ARG;
    const uint64_t n = (uint64_t) 1 << ks->logn, qw = ks->q_limbs * n, rw = ks->limbs * n;
    const uint64_t is = in_stride ? in_stride : qw;
    if (is % n || is < qw) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    // sizes: byte counts within 62 bits; the transforms count polynomials in 32 bits and tiles in 31
    const uint64_t lim = (uint64_t) 1 << 60, polys = (uint64_t) 2 * count * batch;
    if (is > lim || batch > lim / (2 * kAutoMaxElems * (ks->dnum + 2) * rw) || batch - 1 > (lim - qw) / is) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    const uint64_t tiles = std::max<uint64_t>(polys, (uint64_t) ks->dnum * batch) * ks->limbs << (ks->logn - 12);
    if (tiles > 0x7fffffffull || std::max<uint64_t>(polys, (uint64_t) ks->dnum * batch) > 0xffffffffull) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    const ByteRange out = byte_range(d_out, polys * qw);
    if (out.overlaps(byte_range(d_in, (batch - 1) * is + qw)) ||
        out.overlaps(byte_range(d_keys, (uint64_t) count * ks->dnum * 2 * rw))) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if (!aligned16(d_in, d_keys, d_out)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(ks->device);
    return launch_keyswitch(ks, d_in, is, d_keys, galois, count, d_out, batch, (flags & NTTB200_KS_COEFF_IN) != 0,
                            (flags & NTTB200_KS_COEFF_OUT) != 0, false, (cudaStream_t) stream);
}

/* ------------------------------------------------- matrix-vector products */
int nttb200_rns_lintrans_keys(uint32_t logn, const uint32_t *offsets, uint32_t count, uint32_t n1,
                              uint32_t *galois_out, uint32_t *nkeys) {
    if (!nkeys) return NTTB200_ERR_INVALID_ARG;
    LintransSchedule s;
    int rc;
    try {
        rc = lintrans_schedule(logn, offsets, count, n1, &s);
    } catch (...) {
        return NTTB200_ERR_ALLOC;
    }
    if (rc != NTTB200_OK) return rc;
    const uint64_t two_n = (uint64_t) 2 << logn, half = two_n / 4;
    auto rot = [&](uint64_t r) {   // 5^r mod 2N, r < N/2
        uint64_t x = 1, b = 5;
        for (; r; r >>= 1, b = b * b % two_n) {
            if (r & 1) x = x * b % two_n;
        }
        return (uint32_t) x;
    };
    uint32_t k = 0;
    for (uint32_t j : s.babies) {
        if (galois_out) galois_out[k] = rot(j);
        k++;
    }
    for (uint32_t i : s.giants) {
        if (i == 0) continue;
        if (galois_out) galois_out[k] = rot((uint64_t) n1 * i % half);
        k++;
    }
    *nkeys = k;
    return NTTB200_OK;
}

int nttb200_rns_lintrans_apply(nttb200_rns_keyswitch *ks, const int32_t *d_ct, const int32_t *d_diags,
                               const uint32_t *offsets, uint32_t count, uint32_t n1, const int32_t *d_keys,
                               uint32_t nkeys, int32_t *d_out, size_t batch, void *stream) {
    if (!ks) return NTTB200_ERR_INVALID_ARG;
    LintransSchedule s;
    int rc;
    try {
        rc = lintrans_schedule(ks->logn, offsets, count, n1, &s);
    } catch (...) {
        return NTTB200_ERR_ALLOC;
    }
    if (rc != NTTB200_OK) return rc;
    const uint32_t nb = (uint32_t) s.babies.size(), nw = (uint32_t) s.giants.size();
    const uint32_t ng = nw - (s.giants[0] == 0 ? 1 : 0);
    if (nkeys != nb + ng) return NTTB200_ERR_INVALID_ARG;
    if (batch && (!d_ct || !d_diags || !d_out || (nkeys && !d_keys))) return NTTB200_ERR_INVALID_ARG;
    if (batch == 0) return NTTB200_OK;
    const uint64_t n = (uint64_t) 1 << ks->logn, qw = ks->q_limbs * n, ctw = 2 * qw, rw = ks->limbs * n;
    // sizes: byte counts within 62 bits (the buffers, U, W, V and one key-switch pass of up to 64
    // elements); the transforms count polynomials in 32 bits and tiles in 31
    const uint64_t lim = (uint64_t) 1 << 60;
    const uint64_t per = ctw * (2 + nb + nw + ng) + rw * (ks->dnum + 2) * kAutoMaxElems;
    if (batch > lim / per) return NTTB200_ERR_UNSUPPORTED;
    const uint64_t polys = std::max<uint64_t>(std::max<uint64_t>(2 * nb, ks->dnum),
                                              std::max<uint64_t>(2, ks->dnum) * std::min<uint32_t>(ng, kAutoMaxElems)) *
                           batch;
    if ((polys * ks->limbs << (ks->logn - 12)) > 0x7fffffffull || polys > 0xffffffffull) {
        return NTTB200_ERR_UNSUPPORTED;
    }
    const ByteRange out = byte_range(d_out, batch * ctw);
    if (out.overlaps(byte_range(d_ct, batch * ctw)) || out.overlaps(byte_range(d_diags, (uint64_t) count * qw)) ||
        (nkeys && out.overlaps(byte_range(d_keys, (uint64_t) nkeys * ks->dnum * 2 * rw)))) {
        return NTTB200_ERR_INVALID_ARG;
    }
    if (!aligned16(d_ct, d_diags, d_out) || !aligned16(d_keys, d_keys, d_keys)) return NTTB200_ERR_UNSUPPORTED;
    DeviceGuard guard(ks->device);
    try {
        return launch_lintrans(ks, d_ct, d_diags, s, n1, d_keys, d_out, batch, (cudaStream_t) stream);
    } catch (...) {
        return NTTB200_ERR_ALLOC;
    }
}

/* ---------------------------------------------------------- introspection */
const char *nttb200_strerror(int status) {
    switch (status) {
        case NTTB200_OK: return "ok";
        case NTTB200_ERR_INVALID_ARG: return "invalid argument";
        case NTTB200_ERR_MODULUS: return "modulus outside [2, 2^31) (or even where N^-1 is needed)";
        case NTTB200_ERR_TABLE: return "twiddle table entry outside [0, q)";
        case NTTB200_ERR_CUDA: return "CUDA error (see nttb200_last_error)";
        case NTTB200_ERR_NO_DEVICE: return "no usable CUDA device; this library has no CPU path";
        case NTTB200_ERR_ALLOC: return "allocation failed";
        case NTTB200_ERR_UNSUPPORTED: return "unsupported configuration";
        default: return "unknown status";
    }
}

const char *nttb200_last_error(void) { return t_err; }
uint64_t nttb200_kernel_launches(void) { return g_launches.load(std::memory_order_relaxed); }
const char *nttb200_plan_last_path(const nttb200_plan *p) {
    return p ? p->last_path.load(std::memory_order_relaxed) : "none";
}
uint32_t nttb200_plan_logn(const nttb200_plan *p) { return p ? p->logn : 0; }
uint32_t nttb200_plan_modulus(const nttb200_plan *p) { return p ? p->q : 0; }
const char *nttb200_version(void) { return "nttb200 0.3 (sm_100a)"; }

}  // extern "C"
