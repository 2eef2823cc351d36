// b200va_capi.cu -- the C ABI of libb200va.so (declared in include/b200va.h).
//
// Host-side dispatch for the sm_100a vectorAdd kernels: argument checking, alignment
// peeling, geometry resolution, the in-process launch loop, the host-buffer staging
// pipeline.  Each entry point names the step of the reference's `./vectorAdd` process
// it replaces (cuda-test-deployment.yaml:18-19; SURVEY.md section 8(a)).
//
// There is deliberately NO CPU fallback: without a CUDA device every compute entry
// point returns an error code.
#include <cuda_runtime.h>

#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <atomic>
#include <cctype>
#include <condition_variable>
#include <functional>
#include <thread>
#include <vector>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>

#include "../../include/b200va.h"
#include "b200va_kernels.cuh"
#include "b200va_stream.cuh"

using namespace b200va;

namespace {

constexpr int kMaxDevices = 64;

inline int cuda_err(cudaError_t e) { return e == cudaSuccess ? B200VA_OK : -(1000 + static_cast<int>(e)); }

#define CU_TRY(expr)                                   \
    do {                                               \
        cudaError_t e__ = (expr);                      \
        if (e__ != cudaSuccess) return cuda_err(e__);  \
    } while (0)

#define RC_TRY(expr)                   \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != B200VA_OK) return rc__; \
    } while (0)

struct DevCache {
    std::once_flag once;
    int rc = B200VA_ERR_NO_DEVICE;
    b200va_devinfo_t info{};
};
DevCache g_dev[kMaxDevices];

int dev_info(int device, const b200va_devinfo_t** out)
{
    if (device < 0 || device >= kMaxDevices) return B200VA_ERR_INVALID;
    DevCache& dc = g_dev[device];
    std::call_once(dc.once, [&] {
        // individual attributes, not cudaGetDeviceProperties: the latter queries everything
        // and costs tens of milliseconds of every short-lived ./vectorAdd process
        int major = 0, minor = 0, sms = 0, smem = 0, l2 = 0;
        cudaError_t e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, device);
        if (e != cudaSuccess) { dc.rc = cuda_err(e); return; }
        dc.info.device = device;
        dc.info.cc_major = major;
        dc.info.cc_minor = minor;
        dc.info.sm_count = sms;
        dc.info.max_smem_optin = smem;
        dc.info.l2_bytes = l2;
        // the cubin is sm_100a SASS (+ compute_100a PTX): architecture-specific, it runs on CC 10.0 only
        dc.rc = (major == 10 && minor == 0) ? B200VA_OK : B200VA_ERR_NO_DEVICE;
    });
    if (out) *out = &dc.info;
    return dc.rc;
}

int current_dev_info(const b200va_devinfo_t** out)
{
    int device = -1;
    CU_TRY(cudaGetDevice(&device));
    return dev_info(device, out);
}

// ----------------------------------------------------------------------- vec dispatch
// libb200va.so carries the production set only (what AUTO and the named variants resolve to,
// plus close neighbours used by the parity tests); -DB200VA_TUNE_MATRIX (libb200va_tune.so, the
// A/B tool's library) instantiates every combination of b200va_tune_t.  A combination that is
// not compiled in makes the pick functions return nullptr -> B200VA_ERR_VARIANT.
using vec_fn = void (*)(const float*, const float*, float*, size_t, size_t, size_t, size_t);

template <int VW, int UNROLL, int LD, int ST>
vec_fn pick_early_hw(int early)
{
    switch (early) {
        case 0: return vadd_vec<VW, UNROLL, LD, ST, 0>;
        case 1: return vadd_vec<VW, UNROLL, LD, ST, 1>;
        case 2: return vadd_vec<VW, UNROLL, LD, ST, 2>;
    }
    return nullptr;
}

template <int VW, int UNROLL, int LD, int ST>
vec_fn pick_early_clc(int early)
{
    switch (early) {
        case 0: return vadd_vec_clc<VW, UNROLL, LD, ST, 0>;
        case 1: return vadd_vec_clc<VW, UNROLL, LD, ST, 1>;
        case 2: return vadd_vec_clc<VW, UNROLL, LD, ST, 2>;
    }
    return nullptr;
}

template <int VW, int UNROLL, int LD, int ST>
vec_fn pick_sched(int early, int sched)
{
    if (sched == 1) {
#ifdef B200VA_TUNE_MATRIX
        return pick_early_clc<VW, UNROLL, LD, ST>(early);
#else
        if constexpr (VW == 4 && LD == LD_PLAIN && ST == ST_NA && (UNROLL == 2 || UNROLL == 4))
            return pick_early_clc<VW, UNROLL, LD, ST>(early);
        else
            return nullptr;
#endif
    }
    return pick_early_hw<VW, UNROLL, LD, ST>(early);
}

template <int VW, int UNROLL, int LD>
vec_fn pick_st(int st, int early, int sched)
{
    switch (st) {
        case ST_PLAIN: return pick_sched<VW, UNROLL, LD, ST_PLAIN>(early, sched);
        case ST_NA:    return pick_sched<VW, UNROLL, LD, ST_NA>(early, sched);
#ifdef B200VA_TUNE_MATRIX
        case ST_CS:    return pick_sched<VW, UNROLL, LD, ST_CS>(early, sched);
        case ST_NA_EF: return pick_sched<VW, UNROLL, LD, ST_NA_EF>(early, sched);
#endif
    }
    return nullptr;
}

template <int VW, int UNROLL>
vec_fn pick_ld(int ld, int st, int early, int sched)
{
    switch (ld) {
        case LD_PLAIN: return pick_st<VW, UNROLL, LD_PLAIN>(st, early, sched);
        case LD_NA_EF: return pick_st<VW, UNROLL, LD_NA_EF>(st, early, sched);
#ifdef B200VA_TUNE_MATRIX
        case LD_NA:    return pick_st<VW, UNROLL, LD_NA>(st, early, sched);
        case LD_NC_NA: return pick_st<VW, UNROLL, LD_NC_NA>(st, early, sched);
        case LD_CS:    return pick_st<VW, UNROLL, LD_CS>(st, early, sched);
        case LD_NA_256: return pick_st<VW, UNROLL, LD_NA_256>(st, early, sched);
#endif
    }
    return nullptr;
}

template <int VW>
vec_fn pick_unroll(int unroll, int ld, int st, int early, int sched)
{
    switch (unroll) {
        case 1: return pick_ld<VW, 1>(ld, st, early, sched);
        case 2: return pick_ld<VW, 2>(ld, st, early, sched);
        case 4: return pick_ld<VW, 4>(ld, st, early, sched);
#ifdef B200VA_TUNE_MATRIX
        case 8: return pick_ld<VW, 8>(ld, st, early, sched);
#endif
    }
    return nullptr;
}

vec_fn pick_vec(int vw, int unroll, int ld, int st, int early, int sched)
{
    return vw == 8 ? pick_unroll<8>(unroll, ld, st, early, sched) : pick_unroll<4>(unroll, ld, st, early, sched);
}

// ----------------------------------------------------------------------- tma dispatch
using tma_fn = void (*)(const float*, const float*, float*, size_t, size_t, size_t, uint32_t, uint32_t);

#ifdef B200VA_TUNE_MATRIX
template <int MODE, bool HINT>
tma_fn pick_tma_st(int st)
{
    switch (st) {
        case ST_PLAIN: return vadd_tma<MODE, HINT, ST_PLAIN>;
        case ST_NA:    return vadd_tma<MODE, HINT, ST_NA>;
        case ST_CS:    return vadd_tma<MODE, HINT, ST_CS>;
        case ST_NA_EF: return vadd_tma<MODE, HINT, ST_NA_EF>;
    }
    return nullptr;
}
#endif

template <bool HINT>
tma_fn pick_tma_clc_st(int st)
{
    switch (st) {
        case ST_PLAIN: return vadd_tma_clc<HINT, ST_PLAIN>;
        case ST_NA:    return vadd_tma_clc<HINT, ST_NA>;
#ifdef B200VA_TUNE_MATRIX
        case ST_CS:    return vadd_tma_clc<HINT, ST_CS>;
        case ST_NA_EF: return vadd_tma_clc<HINT, ST_NA_EF>;
#endif
    }
    return nullptr;
}

tma_fn pick_tma(int store_mode, bool l2_hint, int st)
{
    if (store_mode == 2)  // cluster-launch-control tile scheduler, register stores
        return l2_hint ? pick_tma_clc_st<true>(st) : pick_tma_clc_st<false>(st);
#ifdef B200VA_TUNE_MATRIX
    if (store_mode == 1)  // st hint is meaningless for bulk stores: one instantiation
        return l2_hint ? vadd_tma<1, true, ST_PLAIN> : vadd_tma<1, false, ST_PLAIN>;
    return l2_hint ? pick_tma_st<0, true>(st) : pick_tma_st<0, false>(st);
#else
    // the static-split ring (store modes 0/1) lost to the CLC form everywhere: tune library only
    if (store_mode == 1 && !l2_hint) return vadd_tma<1, false, ST_PLAIN>;   // kept: the bulk-store (UBLKCP.G.S) form
    if (store_mode == 0 && !l2_hint && st == ST_NA) return vadd_tma<0, false, ST_NA>;
    return nullptr;
#endif
}

std::mutex g_attr_mu;

// Opt in to > 48 KiB dynamic shared memory once per (function, device).
int ensure_smem_optin(tma_fn fn, int device, int bytes)
{
    struct Key { tma_fn fn; int device; int bytes; };
    static Key seen[256];
    static int n_seen = 0;
    std::lock_guard<std::mutex> lk(g_attr_mu);
    for (int i = 0; i < n_seen; ++i)
        if (seen[i].fn == fn && seen[i].device == device) {
            if (seen[i].bytes >= bytes) return B200VA_OK;
            CU_TRY(cudaFuncSetAttribute(reinterpret_cast<const void*>(fn),
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
            seen[i].bytes = bytes;
            return B200VA_OK;
        }
    CU_TRY(cudaFuncSetAttribute(reinterpret_cast<const void*>(fn),
                                cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    if (n_seen < 256) seen[n_seen++] = Key{fn, device, bytes};
    return B200VA_OK;
}

// ----------------------------------------------------------------------- geometry
// Production choices per size class.  K_AUTO is always the 128-bit kernel; thread count / unroll /
// cache hints follow the footprint AND what the caller says about the data:
//
//  default (the same buffers may be launched again: the a1 loop; hot A/B in profiles/r01/{b,c}_ab_2p*.jsonl and
//  profiles/r02/b_hot_2p*.jsonl -- at these footprints the numbers are L2-assisted, not HBM figures)
//   n >= 2^25         HBM streaming         512 thr x1, stores skip L1            7.23 TB/s @2^28, 7.14 @2^26, 7.00 @2^25
//   2^23 < n < 2^25   footprint 1-3 x L2    128 thr x2, L2 evict-first loads      7.34 TB/s @2^24 (7.46 with early loads)
//   6 Mi <= n <= 2^23 footprint ~ L2        256 thr x2, stores skip L1            11.6 TB/s @2^23 (plain stores: 8.7); early: x4, 14.3
//   2^21 <= n < 6 Mi  L2-resident           256 thr x2, plain hints (L2 keeps it) 11.7 TB/s @2^22; early: x4, 13.2
//   n < 2^21          launch-bound          512 thr (>= 2^19) / 128 thr, x1
//
//  B200VA_F_COLD (operands not in L2: the stager's chunks, rotating buffers; profiles/r02/{a,g}_cold_2p*.jsonl, A/B on
//  >= 4 x L2 of rotating buffer sets).  The launch boundary is what costs here (~1.8 us: the previous grid's tail, then a
//  full DRAM round trip before the first store), and the always-legal L2 bulk prefetch ahead of griddepcontrol.wait
//  (early_loads = 2) recovers it without any promise from the caller:
//   n >= 12 Mi         512 thr x1   7.08 TB/s @2^24          (r01 hot-tuned class: 6.46; plain 512 x1: 6.81)
//   3 Mi <= n < 12 Mi  512 thr x2   6.95 @2^22, 7.06 @2^23   (5.75 / 6.26; plain 256/512 x1: 5.83 / 6.45)
//   n < 3 Mi           256 thr x1   4.49 @2^20, 5.87 @2^21   (3.50 / 4.62)
//  B200VA_F_COLD | B200VA_F_INPUTS_STABLE: from 3 Mi the prefetch form is already the best; below, register loads
//  ahead of the wait (early_loads = 1) are: 256 thr x4 6.91 TB/s @2^21, 128 thr x2 6.67 @2^20.
//  n >= 2^25 is never L2-resident, so it always takes the prefetch form (7.25 vs 7.20 TB/s @2^27, 7.22 vs 7.20 @2^28).
void default_tune(int variant, size_t n, b200va_tune_t* t, unsigned flags = 0)
{
    std::memset(t, 0, sizeof *t);
    const bool cold = (flags & B200VA_F_COLD) != 0, early = (flags & B200VA_F_INPUTS_STABLE) != 0;
    t->early_loads = early ? 1 : 0;      // vec kernels only; K0 / K2 ignore it
    switch (variant) {
        case B200VA_K0_SCALAR:
            t->kind = B200VA_K0_SCALAR;
            t->threads = 256;
            t->unroll = 1;
            return;
        case B200VA_K2_TMA:               // TMA ring + cluster-launch-control scheduler (profiles/r01/i_ab_*)
            t->kind = B200VA_K2_TMA;
            t->threads = n >= (size_t{1} << 25) ? 512 : 128;   // consumer threads (+32 producer)
            t->ctas_per_sm = 1;
            t->ld_hint = LD_PLAIN;
            t->st_hint = ST_NA;
            t->stages = n >= (size_t{1} << 25) ? 8 : 3;
            t->tile_bytes = 8192;
            t->store_mode = 2;
            return;
        case B200VA_K1_VEC128:
            t->kind = B200VA_K1_VEC128;
            t->threads = n < (size_t{1} << 19) ? 128 : 512;
            t->unroll = 1;
            t->ld_hint = LD_PLAIN;
            t->st_hint = ST_NA;
            return;
        case B200VA_K3_VEC256:
            t->kind = B200VA_K3_VEC256;
            t->threads = n < (size_t{1} << 26) ? 128 : 1024;
            t->unroll = 1;
            t->ld_hint = n < (size_t{1} << 26) ? LD_NA_EF : LD_PLAIN;
            t->st_hint = n < (size_t{1} << 26) ? ST_PLAIN : ST_NA;
            return;
        default:
            break;
    }
    // B200VA_K_AUTO
    t->kind = B200VA_K1_VEC128;
    t->unroll = 1;
    const size_t Mi = size_t{1} << 20;
    if (n >= 32 * Mi) {
        t->threads = 512; t->ld_hint = LD_PLAIN; t->st_hint = ST_NA;
        if (!early) t->early_loads = 2;
    } else if (cold) {
        t->ld_hint = LD_PLAIN; t->st_hint = ST_PLAIN;
        if (early && n < 3 * Mi) {                       // launch-latency dominated: register loads ahead of the wait
            if (n >= 3 * Mi / 2) { t->threads = 256; t->unroll = 4; }
            else if (n >= Mi / 2) { t->threads = 128; t->unroll = 2; }
            else t->threads = 128;
        } else {                                          // L2 bulk prefetch ahead of the wait
            t->early_loads = 2;
            if (n >= 12 * Mi) t->threads = 512;
            else if (n >= 3 * Mi) { t->threads = 512; t->unroll = 2; }
            else t->threads = n >= Mi / 2 ? 256 : 128;
        }
    } else if (n > 8 * Mi) {
        t->threads = 128; t->unroll = 2; t->ld_hint = LD_NA_EF; t->st_hint = ST_PLAIN;
    } else if (n >= 2 * Mi) {
        t->threads = 256; t->unroll = early ? 4 : 2; t->ld_hint = LD_PLAIN;
        t->st_hint = n >= 6 * Mi ? ST_NA : ST_PLAIN;            // from 6 Mi elements the output no longer fits next to the inputs
    } else if (n >= Mi / 2) {
        t->threads = 512; t->ld_hint = LD_PLAIN; t->st_hint = ST_PLAIN;
    } else {
        t->threads = 128; t->ld_hint = LD_PLAIN; t->st_hint = ST_PLAIN;
    }
}

inline bool is_pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }

int check_args(const float* dA, const float* dB, const float* dC, size_t n)
{
    if (n == 0) return B200VA_OK;
    if (!dA || !dB || !dC) return B200VA_ERR_INVALID;
    const uintptr_t a = reinterpret_cast<uintptr_t>(dA), b = reinterpret_cast<uintptr_t>(dB),
                    c = reinterpret_cast<uintptr_t>(dC);
    if ((a | b | c) & 3u) return B200VA_ERR_ALIGN;
    if (n > (size_t{1} << 40)) return B200VA_ERR_INVALID;
    const uintptr_t bytes = n * sizeof(float);
    auto partial = [&](uintptr_t x) { return x != c && x < c + bytes && c < x + bytes; };
    if (partial(a) || partial(b)) return B200VA_ERR_OVERLAP;
    return B200VA_OK;
}

// Launch geometry of a (validated) tune for a vector body of `nvec` vectors: the single
// place grid/block/smem are computed -- used by launch() and reported by b200va_geometry().
struct Geometry {
    unsigned grid = 1, block = 0;
    size_t smem = 0, ntiles = 0;
};

int plan_geometry(const b200va_tune_t& t, const b200va_devinfo_t* di, size_t n, size_t nvec, Geometry* g)
{
    if (t.kind == B200VA_K0_SCALAR) {
        const size_t blocks = (n + 255) / 256;
        if (blocks > 0x7fffffffull) return B200VA_ERR_INVALID;
        g->grid = static_cast<unsigned>(blocks ? blocks : 1);
        g->block = 256;
        return B200VA_OK;
    }
    if (t.kind == B200VA_K2_TMA) {
        if (t.threads < 32 || t.threads > 992 || (t.threads & 31)) return B200VA_ERR_VARIANT;
        if (t.stages < 2 || t.stages > 32) return B200VA_ERR_VARIANT;
        if (t.tile_bytes < 2048 || (t.tile_bytes & 2047)) return B200VA_ERR_VARIANT;
        if (t.st_hint < 0 || t.st_hint >= ST_HINTS) return B200VA_ERR_VARIANT;
        if (t.store_mode < 0 || t.store_mode > 2) return B200VA_ERR_VARIANT;
        // ring + full/empty barriers; the CLC form adds a barrier, a 16-B response and a tile slot per stage
        const long long smem = static_cast<long long>(t.stages) * 2 * t.tile_bytes +
                               (t.store_mode == 2 ? 44LL * t.stages + 16 : 16LL * t.stages);
        if (smem > di->max_smem_optin) return B200VA_ERR_VARIANT;
        g->smem = static_cast<size_t>(smem);
        g->ntiles = (nvec * 16u + t.tile_bytes - 1) / t.tile_bytes;
        size_t grid = static_cast<size_t>(di->sm_count) * (t.ctas_per_sm > 0 ? t.ctas_per_sm : 1);
        if (t.store_mode == 2) grid = g->ntiles;          // one CTA per tile; resident CTAs cancel the rest
        if (grid > 0x7fffffffull) return B200VA_ERR_INVALID;
        if (grid > g->ntiles) grid = g->ntiles;
        g->grid = static_cast<unsigned>(grid ? grid : 1);
        g->block = static_cast<unsigned>(t.threads + 32);     // + the producer warp
        return B200VA_OK;
    }
    if (t.kind != B200VA_K1_VEC128 && t.kind != B200VA_K3_VEC256) return B200VA_ERR_VARIANT;
    if (t.threads < 32 || t.threads > 1024 || (t.threads & 31)) return B200VA_ERR_VARIANT;
    if (!is_pow2(t.unroll) || t.unroll > 8) return B200VA_ERR_VARIANT;
    if (t.ld_hint < 0 || t.ld_hint >= LD_HINTS || t.st_hint < 0 || t.st_hint >= ST_HINTS) return B200VA_ERR_VARIANT;
    if (t.scheduler < 0 || t.scheduler > 1 || (t.scheduler == 1 && t.ctas_per_sm != 0)) return B200VA_ERR_VARIANT;
    const size_t tile_vecs = static_cast<size_t>(t.threads) * t.unroll;
    g->ntiles = (nvec + tile_vecs - 1) / tile_vecs;
    size_t grid = g->ntiles;
    if (t.scheduler == 1 && grid > 0x7fffffffull) return B200VA_ERR_INVALID;   // CLC: one CTA per tile, 32-bit tile index
    if (t.ctas_per_sm > 0) {
        const size_t cap = static_cast<size_t>(di->sm_count) * t.ctas_per_sm;
        if (grid > cap) grid = cap;
    }
    if (grid > 0x7fffffffull) grid = 0x7fffffffull;   // the kernel loops tile += gridDim.x
    g->grid = static_cast<unsigned>(grid ? grid : 1);
    g->block = static_cast<unsigned>(t.threads);
    return B200VA_OK;
}

// All hot-path launches go through here: programmatic stream serialization lets launch
// k+1 ramp up behind launch k's tail (the kernels call griddepcontrol.wait before their
// first global access, so stream order is unchanged).  B200VA_NO_PDL=1 disables it.
thread_local bool tl_pdl_off = false;   // set while re-capturing a graph without PDL edges

bool pdl_enabled()
{
    static const bool on = [] {
        const char* e = std::getenv("B200VA_NO_PDL");
        return !(e && e[0] == '1');
    }();
    return on && !tl_pdl_off;
}

template <class... KArgs, class... Args>
int launch_kernel(void (*fn)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t stream, Args... args)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, fn, static_cast<KArgs>(args)...);
    if (e != cudaSuccess) cudaGetLastError();   // a refused launch must not stay latched for the next caller
    return cuda_err(e);
}

// Largest CTA the kernel can be launched with (register-limited for the deep unrolls).
template <class Fn>
int check_block_size(Fn fn, unsigned block)
{
    thread_local const void* last_fn = nullptr;
    thread_local unsigned last_max = 0;
    const void* key = reinterpret_cast<const void*>(fn);
    if (key != last_fn) {
        cudaFuncAttributes fa;
        CU_TRY(cudaFuncGetAttributes(&fa, key));
        last_fn = key;
        last_max = static_cast<unsigned>(fa.maxThreadsPerBlock);
    }
    return block > last_max ? B200VA_ERR_VARIANT : B200VA_OK;
}

int launch(const float* dA, const float* dB, float* dC, size_t n, b200va_tune_t t, cudaStream_t stream)
{
    RC_TRY(check_args(dA, dB, dC, n));
    const b200va_devinfo_t* di = nullptr;
    RC_TRY(current_dev_info(&di));
    if (n == 0) return B200VA_OK;

    const uintptr_t a = reinterpret_cast<uintptr_t>(dA), b = reinterpret_cast<uintptr_t>(dB),
                    c = reinterpret_cast<uintptr_t>(dC);
    const bool aliased = (a == c) || (b == c);
    // .nc (non-coherent) loads require data that is read-only for the kernel's lifetime
    if (aliased && t.ld_hint == LD_NC_NA) t.ld_hint = LD_PLAIN;

    int vw = 0;
    if (t.kind == B200VA_K3_VEC256) vw = 8;
    else if (t.kind == B200VA_K1_VEC128 || t.kind == B200VA_K2_TMA) vw = 4;
    else if (t.kind != B200VA_K0_SCALAR && t.kind != B200VA_K4_SCALAR_MLP) return B200VA_ERR_VARIANT;

    // vector body needs A, B, C equally misaligned w.r.t. the vector width
    size_t head = 0;
    while (vw) {
        const uintptr_t mask = static_cast<uintptr_t>(vw) * 4u - 1u;
        if ((a & mask) == (b & mask) && (a & mask) == (c & mask)) {
            head = ((static_cast<uintptr_t>(vw) * 4u - (a & mask)) & mask) / 4u;
            break;
        }
        if (t.kind == B200VA_K2_TMA) { vw = 0; break; }
        vw = (vw == 8) ? 4 : 0;
    }
    Geometry g;
    if (t.kind == B200VA_K4_SCALAR_MLP || (vw == 0 && t.kind != B200VA_K0_SCALAR)) {
        // 4-byte kernel with U loads per array per thread in flight: explicit A/B variant, and the
        // path taken when A, B, C share no 16-byte phase (no vector body exists)
        const bool explicit_geo = t.kind == B200VA_K4_SCALAR_MLP;
        const unsigned threads = explicit_geo ? static_cast<unsigned>(t.threads) : 256u;
        const int U = explicit_geo ? t.unroll : 8;
        if (threads < 32 || threads > 1024 || (threads & 31u)) return B200VA_ERR_VARIANT;
        if (U != 4 && U != 8 && U != 16) return B200VA_ERR_VARIANT;
        const size_t per_cta = static_cast<size_t>(threads) * static_cast<size_t>(U);
        const size_t blocks = (n + per_cta - 1) / per_cta;
        if (blocks > 0x7fffffffull) return B200VA_ERR_INVALID;
        auto fn = U == 4 ? vadd_scalar_unrolled<4> : U == 8 ? vadd_scalar_unrolled<8> : vadd_scalar_unrolled<16>;
        if (threads > 256) RC_TRY(check_block_size(fn, threads));
        return launch_kernel(fn, static_cast<unsigned>(blocks), threads, 0, stream, dA, dB, dC, n);
    }
    if (vw == 0) {  // the scalar control
        b200va_tune_t k0{};
        k0.kind = B200VA_K0_SCALAR;
        RC_TRY(plan_geometry(k0, di, n, 0, &g));
        // the control keeps the sample's plain launch (no programmatic dependent launch)
        vadd_scalar<<<g.grid, g.block, 0, stream>>>(dA, dB, dC, n);
        return cuda_err(cudaGetLastError());
    }
    if (head > n) head = n;
    const size_t nvec = (n - head) / static_cast<size_t>(vw);
    RC_TRY(plan_geometry(t, di, n, nvec, &g));

    if (t.kind == B200VA_K2_TMA) {
        tma_fn fn = pick_tma(t.store_mode, t.ld_hint == LD_NA_EF, t.st_hint);
        if (!fn) return B200VA_ERR_VARIANT;
        RC_TRY(ensure_smem_optin(fn, di->device, static_cast<int>(g.smem)));
        return launch_kernel(fn, g.grid, g.block, g.smem, stream, dA, dB, dC, n, head, nvec,
                             static_cast<uint32_t>(t.tile_bytes), static_cast<uint32_t>(t.stages));
    }
    // early register loads (1) read A and B while the previous launch may still be running: never when C aliases
    // an input -- the always-legal L2 prefetch (2) takes their place
    const int early = (t.early_loads == 1 && aliased) ? 2 : t.early_loads;
    vec_fn fn = pick_vec(vw, t.unroll, t.ld_hint, t.st_hint, early, t.scheduler);
    if (!fn) return B200VA_ERR_VARIANT;
    if (g.block > 256) RC_TRY(check_block_size(fn, g.block));   // deep unrolls: the CTA size is register-limited
    return launch_kernel(fn, g.grid, g.block, 0, stream, dA, dB, dC, n, head, nvec, g.ntiles);
}

unsigned support_grid(const b200va_devinfo_t* di, size_t n, int threads)
{
    size_t want = (n + threads - 1) / threads;
    size_t cap = static_cast<size_t>(di->sm_count) * 16;
    if (want > cap) want = cap;
    if (want == 0) want = 1;
    return static_cast<unsigned>(want);
}

}  // namespace

// ----------------------------------------------------------------------- f4 dispatch
namespace {

template <int DT, int OP>
int launch_stream_typed(const void* dA, const void* dB, void* dC, size_t n, double scalar, cudaStream_t st)
{
    using S = typename dt_traits<DT>::scalar;
    constexpr size_t ES = dt_traits<DT>::size;
    constexpr bool binary = (OP == OP_ADD || OP == OP_TRIAD);
    const S s = static_cast<S>(scalar);
    const uintptr_t a = reinterpret_cast<uintptr_t>(dA), b = reinterpret_cast<uintptr_t>(dB),
                    c = reinterpret_cast<uintptr_t>(dC);
    const bool vec_ok = (a & 15u) == (c & 15u) && (!binary || (b & 15u) == (a & 15u));
    if (!vec_ok) {
        const size_t blocks = (n + 255) / 256;
        if (blocks > 0x7fffffffull) return B200VA_ERR_INVALID;
        stream_scalar<DT, OP><<<static_cast<unsigned>(blocks), 256, 0, st>>>(dA, dB, dC, n, s);
        return cuda_err(cudaGetLastError());
    }
    size_t head = ((16u - (a & 15u)) & 15u) / ES;
    if (head > n) head = n;
    const size_t nvec = (n - head) * ES / 16;
    // same footprint classes as the f32 add (default_tune), in 4-byte units
    const size_t m = n * ES / 4;
    unsigned threads = 128;
    int unroll = 1;
    bool skip_l1_stores = false;
    if (m >= (size_t{1} << 25)) {
        // three-array ops like the add: 512 x 1; two-array ops (copy, scale) want twice the bytes in
        // flight per thread: 1024 x 2 is 7.04 TB/s vs 6.41 (profiles/r01/r_stream_geometry.jsonl)
        threads = binary ? 512 : 1024;
        unroll = binary ? 1 : 2;
        skip_l1_stores = true;
    } else if (m > (size_t{1} << 23)) { threads = 128; unroll = 2; }
    else if (m >= (size_t{1} << 21)) { threads = 256; unroll = 2; }
    else if (m >= (size_t{1} << 19)) { threads = 512; }
#ifdef B200VA_TUNE_MATRIX
    // development knob for profiles/ (tune library only): B200VA_STREAM_GEOMETRY="threads,unroll,skip_l1_stores"
    static const struct Override { int threads = 0, unroll = 0, na = 0; } ov = [] {
        Override o;
        if (const char* e = std::getenv("B200VA_STREAM_GEOMETRY")) std::sscanf(e, "%d,%d,%d", &o.threads, &o.unroll, &o.na);
        return o;
    }();
    if (ov.threads >= 32 && ov.threads <= 1024 && (ov.threads & 31) == 0 && (ov.unroll == 1 || ov.unroll == 2 || ov.unroll == 4)) {
        threads = static_cast<unsigned>(ov.threads);
        unroll = ov.unroll;
        skip_l1_stores = ov.na != 0;
    }
#endif
    const size_t tile_vecs = static_cast<size_t>(threads) * unroll;
    size_t grid = (nvec + tile_vecs - 1) / tile_vecs;
    if (grid > 0x7fffffffull) grid = 0x7fffffffull;
    if (grid == 0) grid = 1;
    const size_t ntiles = (nvec + tile_vecs - 1) / tile_vecs;
    using fn_t = void (*)(const void*, const void*, void*, size_t, size_t, size_t, size_t, S, int);
    const int prefetch_first = m >= (size_t{1} << 25) ? 1 : 0;      // >= 128 MiB per array: never L2-resident
    fn_t fn = nullptr;
#ifdef B200VA_TUNE_MATRIX
    if (unroll == 4) fn = skip_l1_stores ? stream_vec<DT, OP, 4, LD_PLAIN, ST_NA> : stream_vec<DT, OP, 4, LD_PLAIN, ST_PLAIN>;
#endif
    if (!fn) {
        if (skip_l1_stores) fn = unroll == 2 ? stream_vec<DT, OP, 2, LD_PLAIN, ST_NA> : stream_vec<DT, OP, 1, LD_PLAIN, ST_NA>;
        else fn = unroll == 2 ? stream_vec<DT, OP, 2, LD_PLAIN, ST_PLAIN> : stream_vec<DT, OP, 1, LD_PLAIN, ST_PLAIN>;
    }
    return launch_kernel(fn, static_cast<unsigned>(grid), threads, 0, st, dA, dB, dC, n, head, nvec, ntiles, s, prefetch_first);
}

template <int DT>
int launch_stream_op(int op, const void* dA, const void* dB, void* dC, size_t n, double scalar, cudaStream_t st)
{
    switch (op) {
        case OP_COPY:  return launch_stream_typed<DT, OP_COPY>(dA, dB, dC, n, scalar, st);
        case OP_SCALE: return launch_stream_typed<DT, OP_SCALE>(dA, dB, dC, n, scalar, st);
        case OP_ADD:   return launch_stream_typed<DT, OP_ADD>(dA, dB, dC, n, scalar, st);
        case OP_TRIAD: return launch_stream_typed<DT, OP_TRIAD>(dA, dB, dC, n, scalar, st);
    }
    return B200VA_ERR_VARIANT;
}

// ----------------------------------------------------------------------- grouped dispatch
// Items per launch: the parameter block holds kGroupedCap items of 40 B (record + tile prefix),
// 32,032 B in all, under the 32,764-B limit of cudaLaunchKernelEx.
constexpr int kGroupedCap = 800;
static_assert(sizeof(GroupedParams<kGroupedCap>) + sizeof(double) + sizeof(int) <= 32764, "kernel parameter block too large");
// Production geometry (threads x unroll per tile) for every op and dtype.
constexpr unsigned kGroupedThreads = 256;
constexpr int kGroupedUnroll = 2;

// The checks of b200va_stream, for one item.
int check_stream_item(const b200va_item_t& it, bool binary, size_t es)
{
    if (it.n == 0) return B200VA_OK;
    if (!it.a || !it.c || (binary && !it.b)) return B200VA_ERR_INVALID;
    const uintptr_t a = reinterpret_cast<uintptr_t>(it.a), b = reinterpret_cast<uintptr_t>(it.b),
                    c = reinterpret_cast<uintptr_t>(it.c);
    if (((a | c | (binary ? b : 0)) & (es - 1)) != 0) return B200VA_ERR_ALIGN;
    if (it.n > (size_t{1} << 40)) return B200VA_ERR_INVALID;
    const uintptr_t bytes = it.n * es;
    auto partial = [&](uintptr_t x) { return x != c && x < c + bytes && c < x + bytes; };
    if (partial(a) || (binary && partial(b))) return B200VA_ERR_OVERLAP;
    return B200VA_OK;
}

// Packs the non-empty items into parameter blocks of CAP, computes each block's tile prefix and
// launches it; blocks go out in item order on `st`.
template <int DT, int OP, int UNROLL, int CAP>
int launch_grouped_blocks(const b200va_item_t* items, size_t count, double scalar, unsigned threads, cudaStream_t st)
{
    using S = typename dt_traits<DT>::scalar;
    constexpr int ES = dt_traits<DT>::size;
    constexpr bool binary = (OP == OP_ADD || OP == OP_TRIAD);
    const S s = static_cast<S>(scalar);
    const size_t tile_vecs = static_cast<size_t>(threads) * UNROLL;
    GroupedParams<CAP> p;
    size_t i = 0;
    while (i < count) {
        int k = 0;
        unsigned long long tiles = 0;
        size_t bytes = 0;
        for (; i < count && k < CAP; ++i) {
            const b200va_item_t& it = items[i];
            if (it.n == 0) continue;
            p.item[k] = GroupedItem{it.a, it.b, it.c, it.n};
            p.first_tile[k] = tiles;
            tiles += grouped_shape<ES, binary>(it.a, it.b, it.c, it.n, tile_vecs).ntiles;
            bytes += it.n * ES;
            ++k;
        }
        if (k == 0) break;
        p.count = k;
        p.total_tiles = tiles;
        const unsigned grid = static_cast<unsigned>(tiles > 0x7fffffffull ? 0x7fffffffull : tiles);   // the kernel loops tile += gridDim.x
        const int prefetch_first = bytes >= (size_t{1} << 27) ? 1 : 0;     // >= 128 MiB per array: never L2-resident
        RC_TRY(launch_kernel(stream_grouped<DT, OP, UNROLL, CAP>, grid, threads, 0, st, p, s, prefetch_first));
    }
    return B200VA_OK;
}

template <int DT, int OP>
int launch_grouped_typed(const b200va_item_t* items, size_t count, double scalar, cudaStream_t st)
{
#ifdef B200VA_TUNE_MATRIX
    // development knob for profiles/ (tune library only): B200VA_GROUPED_GEOMETRY="threads,unroll,capacity",
    // unroll 1 | 2 | 4, capacity 100 | 800
    static const struct Override { int threads = 0, unroll = 0, cap = 0; } ov = [] {
        Override o;
        if (const char* e = std::getenv("B200VA_GROUPED_GEOMETRY")) std::sscanf(e, "%d,%d,%d", &o.threads, &o.unroll, &o.cap);
        return o;
    }();
    if (ov.threads >= 32 && ov.threads <= 1024 && (ov.threads & 31) == 0 && (ov.cap == 100 || ov.cap == kGroupedCap)) {
        const unsigned t = static_cast<unsigned>(ov.threads);
        if (ov.cap == 100) {
            if (ov.unroll == 1) return launch_grouped_blocks<DT, OP, 1, 100>(items, count, scalar, t, st);
            if (ov.unroll == 2) return launch_grouped_blocks<DT, OP, 2, 100>(items, count, scalar, t, st);
            if (ov.unroll == 4) return launch_grouped_blocks<DT, OP, 4, 100>(items, count, scalar, t, st);
        } else {
            if (ov.unroll == 1) return launch_grouped_blocks<DT, OP, 1, kGroupedCap>(items, count, scalar, t, st);
            if (ov.unroll == 2) return launch_grouped_blocks<DT, OP, 2, kGroupedCap>(items, count, scalar, t, st);
            if (ov.unroll == 4) return launch_grouped_blocks<DT, OP, 4, kGroupedCap>(items, count, scalar, t, st);
        }
    }
#endif
    return launch_grouped_blocks<DT, OP, kGroupedUnroll, kGroupedCap>(items, count, scalar, kGroupedThreads, st);
}

template <int DT>
int launch_grouped_op(int op, const b200va_item_t* items, size_t count, double scalar, cudaStream_t st)
{
    switch (op) {
        case OP_COPY:  return launch_grouped_typed<DT, OP_COPY>(items, count, scalar, st);
        case OP_SCALE: return launch_grouped_typed<DT, OP_SCALE>(items, count, scalar, st);
        case OP_ADD:   return launch_grouped_typed<DT, OP_ADD>(items, count, scalar, st);
        case OP_TRIAD: return launch_grouped_typed<DT, OP_TRIAD>(items, count, scalar, st);
    }
    return B200VA_ERR_VARIANT;
}

}  // namespace

// =============================================================================== ABI
extern "C" {

int b200va_abi_version(void) { return B200VA_ABI_VERSION; }

const char* b200va_strerror(int code)
{
    switch (code) {
        case B200VA_OK:            return "success";
        case B200VA_ERR_INVALID:   return "invalid argument";
        case B200VA_ERR_ALIGN:     return "pointer not 4-byte aligned";
        case B200VA_ERR_OVERLAP:   return "output partially overlaps an input";
        case B200VA_ERR_VARIANT:   return "unknown kernel variant or unsupported geometry";
        case B200VA_ERR_NO_DEVICE: return "no sm_100 CUDA device";
        case B200VA_ERR_VERIFY:    return "result verification failed";
        case B200VA_ERR_NOMEM:     return "host allocation failed";
    }
    if (code <= B200VA_ERR_CUDA_BASE) return cudaGetErrorString(static_cast<cudaError_t>(-code - 1000));
    return "unknown error";
}

int b200va_query(int device, b200va_devinfo_t* out)
{
    if (!out) return B200VA_ERR_INVALID;
    const b200va_devinfo_t* di = nullptr;
    const int rc = dev_info(device, &di);
    if (!di || di->sm_count <= 0) return rc;
    *out = *di;
    cudaDeviceProp p;                       // name and memory size: only this (cold) call pays for them
    if (cudaGetDeviceProperties(&p, device) == cudaSuccess) {
        out->global_mem_bytes = p.totalGlobalMem;
        std::snprintf(out->name, sizeof out->name, "%s", p.name);
    }
    return rc;
}

int b200va_resolve(int variant, size_t n, b200va_tune_t* out)
{
    if (!out || variant < B200VA_K_AUTO || variant > B200VA_K3_VEC256) return B200VA_ERR_VARIANT;
    default_tune(variant, n, out);
    return B200VA_OK;
}

int b200va_resolve_ex(int variant, size_t n, unsigned flags, b200va_tune_t* out)
{
    if (!out || variant < B200VA_K_AUTO || variant > B200VA_K3_VEC256) return B200VA_ERR_VARIANT;
    if (flags & ~(B200VA_F_INPUTS_STABLE | B200VA_F_COLD)) return B200VA_ERR_INVALID;
    default_tune(variant, n, out, flags);
    return B200VA_OK;
}

int b200va_geometry(const b200va_tune_t* tune, size_t n, int device, unsigned* grid, unsigned* block,
                    unsigned* dyn_smem_bytes)
{
    if (!tune || !grid || !block) return B200VA_ERR_INVALID;
    const b200va_devinfo_t* di = nullptr;
    RC_TRY(dev_info(device, &di));
    Geometry g;
    const size_t vw = tune->kind == B200VA_K3_VEC256 ? 8 : 4;
    RC_TRY(plan_geometry(*tune, di, n, n / vw, &g));
    *grid = g.grid;
    *block = g.block;
    if (dyn_smem_bytes) *dyn_smem_bytes = static_cast<unsigned>(g.smem);
    return B200VA_OK;
}

int b200va_add_f32(const float* dA, const float* dB, float* dC, size_t n, int variant, void* stream)
{
    if (variant < B200VA_K_AUTO || variant > B200VA_K3_VEC256) return B200VA_ERR_VARIANT;
    b200va_tune_t t;
    default_tune(variant, n, &t);
    return launch(dA, dB, dC, n, t, static_cast<cudaStream_t>(stream));
}

int b200va_add_f32_ex(const float* dA, const float* dB, float* dC, size_t n, int variant, unsigned flags, void* stream)
{
    if (variant < B200VA_K_AUTO || variant > B200VA_K3_VEC256) return B200VA_ERR_VARIANT;
    if (flags & ~(B200VA_F_INPUTS_STABLE | B200VA_F_COLD)) return B200VA_ERR_INVALID;
    b200va_tune_t t;
    default_tune(variant, n, &t, flags);
    return launch(dA, dB, dC, n, t, static_cast<cudaStream_t>(stream));
}

int b200va_add_f32_tuned(const float* dA, const float* dB, float* dC, size_t n,
                         const b200va_tune_t* tune, void* stream)
{
    if (!tune) return B200VA_ERR_INVALID;
    b200va_tune_t t = *tune;
    b200va_tune_t d;
    default_tune(t.kind, n, &d);
    if (t.kind == B200VA_K_AUTO) t = d;
    if (t.kind == B200VA_K4_SCALAR_MLP) {
        if (t.threads == 0) t.threads = 256;
        if (t.unroll == 0) t.unroll = 8;
    }
    if (t.threads == 0) t.threads = d.threads;
    if (t.unroll == 0) t.unroll = d.unroll ? d.unroll : 1;
    if (t.stages == 0) t.stages = d.stages;
    if (t.tile_bytes == 0) t.tile_bytes = d.tile_bytes;
    if (t.early_loads < 0 || t.early_loads > 2 || (t.scheduler & ~1)) return B200VA_ERR_VARIANT;
    return launch(dA, dB, dC, n, t, static_cast<cudaStream_t>(stream));
}

// ---- a1: the launch loop --------------------------------------------------------------
struct b200va_loop {
    const float *dA = nullptr, *dB = nullptr;
    float* dC = nullptr;
    size_t n = 0;
    b200va_tune_t tune{};
    int batch = 1;
    int device = 0;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    bool pdl_edges = false;
};

static int capture_batch(b200va_loop* l, cudaStream_t cap)
{
    CU_TRY(cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
    int rc = B200VA_OK;
    // node 0 follows an unknown predecessor; nodes 1.. follow the same add (which writes only C),
    // so their loads may run ahead of the dependency (launch() drops the hint if C aliases A or B)
    b200va_tune_t follow = l->tune;
    follow.early_loads = 1;
    for (int i = 0; i < l->batch && rc == B200VA_OK; ++i) rc = launch(l->dA, l->dB, l->dC, l->n, i ? follow : l->tune, cap);
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(cap, &g);
    if (rc != B200VA_OK || e != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        return rc != B200VA_OK ? rc : cuda_err(e);
    }
    cudaGraphExec_t x = nullptr;
    const cudaError_t e2 = cudaGraphInstantiate(&x, g, 0);
    if (e2 != cudaSuccess) { cudaGraphDestroy(g); cudaGetLastError(); return cuda_err(e2); }
    l->graph = g;
    l->exec = x;
    return B200VA_OK;
}

int b200va_loop_destroy(b200va_loop_t* l)
{
    if (!l) return B200VA_OK;
    if (l->exec) cudaGraphExecDestroy(l->exec);
    if (l->graph) cudaGraphDestroy(l->graph);
    delete l;
    return B200VA_OK;
}

int b200va_loop_create(b200va_loop_t** out, const float* dA, const float* dB, float* dC, size_t n, int variant,
                       int graph_batch)
{
    if (!out || graph_batch < 0) return B200VA_ERR_INVALID;
    *out = nullptr;
    if (variant < B200VA_K_AUTO || variant > B200VA_K3_VEC256) return B200VA_ERR_VARIANT;
    RC_TRY(check_args(dA, dB, dC, n));
    b200va_loop* l = new (std::nothrow) b200va_loop;
    if (!l) return B200VA_ERR_NOMEM;
    l->dA = dA; l->dB = dB; l->dC = dC; l->n = n;
    l->batch = graph_batch > 1 ? graph_batch : 1;
    default_tune(variant, n, &l->tune);
    cudaError_t e = cudaGetDevice(&l->device);
    if (e != cudaSuccess) { delete l; return cuda_err(e); }
    if (l->batch > 1 && n > 0) {
        cudaStream_t cap = nullptr;
        e = cudaStreamCreateWithFlags(&cap, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete l; return cuda_err(e); }
        int rc = capture_batch(l, cap);
        l->pdl_edges = (rc == B200VA_OK) && pdl_enabled();
        if (rc != B200VA_OK && pdl_enabled()) {   // older drivers: capture without programmatic edges
            tl_pdl_off = true;
            rc = capture_batch(l, cap);
            tl_pdl_off = false;
        }
        cudaStreamDestroy(cap);
        if (rc != B200VA_OK) { delete l; return rc; }
    }
    *out = l;
    return B200VA_OK;
}

int b200va_loop_run(b200va_loop_t* l, int iters, void* stream)
{
    if (!l || iters < 0) return B200VA_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int left = iters;
    bool first = true;                       // the first launch of a run follows whatever the caller queued before
    if (l->exec) {
        for (; left >= l->batch; left -= l->batch) { CU_TRY(cudaGraphLaunch(l->exec, st)); first = false; }
    }
    b200va_tune_t follow = l->tune;
    follow.early_loads = 1;
    for (; left > 0; --left) { RC_TRY(launch(l->dA, l->dB, l->dC, l->n, first ? l->tune : follow, st)); first = false; }
    return B200VA_OK;
}

int b200va_add_f32_loop(const float* dA, const float* dB, float* dC, size_t n, int variant, int iters,
                        int graph_batch, void* stream)
{
    if (iters < 0 || graph_batch < 0) return B200VA_ERR_INVALID;
    if (variant < B200VA_K_AUTO || variant > B200VA_K3_VEC256) return B200VA_ERR_VARIANT;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (graph_batch <= 1 || iters < graph_batch) {
        b200va_tune_t t, follow;
        default_tune(variant, n, &t);
        follow = t;
        follow.early_loads = 1;
        for (int i = 0; i < iters; ++i) RC_TRY(launch(dA, dB, dC, n, i ? follow : t, st));
        return B200VA_OK;
    }
    b200va_loop_t* l = nullptr;
    RC_TRY(b200va_loop_create(&l, dA, dB, dC, n, variant, graph_batch));
    int rc = b200va_loop_run(l, iters, stream);
    // the executable graph must outlive its launches: the one-shot form drains the stream
    const cudaError_t e = cudaStreamSynchronize(st);
    b200va_loop_destroy(l);
    if (rc == B200VA_OK) rc = cuda_err(e);
    return rc;
}

// ------------------------------------------------------------------ a2: input recipes
int b200va_host_fill_rand_f32(float* hA, float* hB, size_t n)
{
    if (n && (!hA || !hB)) return B200VA_ERR_INVALID;
    srand(1);  // a fresh ./vectorAdd process never calls srand: glibc default seed is 1
    for (size_t i = 0; i < n; ++i) {
        hA[i] = rand() / (float)RAND_MAX;
        hB[i] = rand() / (float)RAND_MAX;
    }
    return B200VA_OK;
}

static inline uint64_t host_splitmix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

int b200va_host_fill_ctr_f32(float* h, size_t n, uint64_t seed, uint64_t first)
{
    if (n && !h) return B200VA_ERR_INVALID;
    const uint64_t base = seed * 0x9E3779B97F4A7C15ull + first;
    for (size_t i = 0; i < n; ++i)
        h[i] = static_cast<float>(static_cast<uint32_t>(host_splitmix64(base + i) >> 40)) * 0x1.0p-24f;
    return B200VA_OK;
}

int b200va_fill_ctr_f32(float* d, size_t n, uint64_t seed, uint64_t first, void* stream)
{
    if (n && !d) return B200VA_ERR_INVALID;
    const b200va_devinfo_t* di = nullptr;
    RC_TRY(current_dev_info(&di));
    if (n == 0) return B200VA_OK;
    const uint64_t base = seed * 0x9E3779B97F4A7C15ull + first;
    if ((reinterpret_cast<uintptr_t>(d) & 15u) == 0)      // the usual case: one STG.128 per four elements
        fill_ctr_vec<<<support_grid(di, (n + 3) / 4, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(d, n, base);
    else
        fill_ctr<<<support_grid(di, n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(d, n, base);
    return cuda_err(cudaGetLastError());
}

// ------------------------------------------------------------------ a6: verification
int b200va_host_verify_f32(const float* hA, const float* hB, const float* hC, size_t n, size_t* first_bad)
{
    if (n && (!hA || !hB || !hC)) return B200VA_ERR_INVALID;
    for (size_t i = 0; i < n; ++i) {
        const float want = hA[i] + hB[i];
        uint32_t uw, ug;
        std::memcpy(&uw, &want, 4);
        std::memcpy(&ug, &hC[i], 4);
        if (uw == ug) continue;
        const bool nw = (uw & 0x7fffffffu) > 0x7f800000u, ng = (ug & 0x7fffffffu) > 0x7f800000u;
        if (nw && ng) continue;
        if (first_bad) *first_bad = i;
        return B200VA_ERR_VERIFY;
    }
    return B200VA_OK;
}

int b200va_verify_f32(const float* dA, const float* dB, const float* dC, size_t n,
                      uint64_t* d_result, void* stream)
{
    if (!d_result || (n && (!dA || !dB || !dC))) return B200VA_ERR_INVALID;
    const b200va_devinfo_t* di = nullptr;
    RC_TRY(current_dev_info(&di));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    auto* res = reinterpret_cast<unsigned long long*>(d_result);
    reset_verify<<<1, 1, 0, st>>>(res);
    const bool aligned = ((reinterpret_cast<uintptr_t>(dA) | reinterpret_cast<uintptr_t>(dB) | reinterpret_cast<uintptr_t>(dC)) & 15u) == 0;
    if (n && aligned) verify_bits_vec<<<support_grid(di, (n + 3) / 4, 256), 256, 0, st>>>(dA, dB, dC, n, res);
    else if (n) verify_bits<<<support_grid(di, n, 256), 256, 0, st>>>(dA, dB, dC, n, res);
    return cuda_err(cudaGetLastError());
}

int b200va_digest_f32(const float* d, size_t n, uint64_t* d_out, void* stream)
{
    if (!d_out || (n && !d)) return B200VA_ERR_INVALID;
    const b200va_devinfo_t* di = nullptr;
    RC_TRY(current_dev_info(&di));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    auto* out = reinterpret_cast<unsigned long long*>(d_out);
    reset_digest<<<1, 1, 0, st>>>(out);
    if (n && (reinterpret_cast<uintptr_t>(d) & 15u) == 0) digest_bits_vec<<<support_grid(di, (n + 3) / 4, 256), 256, 0, st>>>(d, n, out);
    else if (n) digest_bits<<<support_grid(di, n, 256), 256, 0, st>>>(d, n, out);
    return cuda_err(cudaGetLastError());
}

// ------------------------------------------------------------------ f4: STREAM-style ops
int b200va_stream(int op, int dtype, const void* dA, const void* dB, void* dC, size_t n, double scalar, void* stream)
{
    if (op < 0 || op >= OP_COUNT || dtype < 0 || dtype >= DT_COUNT) return B200VA_ERR_VARIANT;
    const b200va_devinfo_t* di = nullptr;
    RC_TRY(current_dev_info(&di));
    if (n == 0) return B200VA_OK;
    const bool binary = (op == OP_ADD || op == OP_TRIAD);
    if (!dA || !dC || (binary && !dB)) return B200VA_ERR_INVALID;
    const size_t es = dtype == DT_F64 ? 8 : dtype == DT_F32 ? 4 : 2;
    const uintptr_t a = reinterpret_cast<uintptr_t>(dA), b = reinterpret_cast<uintptr_t>(dB),
                    c = reinterpret_cast<uintptr_t>(dC);
    if (((a | c | (binary ? b : 0)) & (es - 1)) != 0) return B200VA_ERR_ALIGN;
    if (n > (size_t{1} << 40)) return B200VA_ERR_INVALID;
    const uintptr_t bytes = n * es;
    auto partial = [&](uintptr_t x) { return x != c && x < c + bytes && c < x + bytes; };
    if (partial(a) || (binary && partial(b))) return B200VA_ERR_OVERLAP;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (dtype) {
        case DT_F32:  return launch_stream_op<DT_F32>(op, dA, dB, dC, n, scalar, st);
        case DT_F64:  return launch_stream_op<DT_F64>(op, dA, dB, dC, n, scalar, st);
        case DT_F16:  return launch_stream_op<DT_F16>(op, dA, dB, dC, n, scalar, st);
        case DT_BF16: return launch_stream_op<DT_BF16>(op, dA, dB, dC, n, scalar, st);
    }
    return B200VA_ERR_VARIANT;
}

int b200va_stream_grouped(int op, int dtype, const b200va_item_t* items, size_t count, double scalar, void* stream)
{
    if (op < 0 || op >= OP_COUNT || dtype < 0 || dtype >= DT_COUNT) return B200VA_ERR_VARIANT;
    const b200va_devinfo_t* di = nullptr;
    RC_TRY(current_dev_info(&di));
    if (count == 0) return B200VA_OK;
    if (!items) return B200VA_ERR_INVALID;
    const bool binary = (op == OP_ADD || op == OP_TRIAD);
    const size_t es = dtype == DT_F64 ? 8 : dtype == DT_F32 ? 4 : 2;
    for (size_t i = 0; i < count; ++i) RC_TRY(check_stream_item(items[i], binary, es));   // nothing is enqueued on a failure
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (dtype) {
        case DT_F32:  return launch_grouped_op<DT_F32>(op, items, count, scalar, st);
        case DT_F64:  return launch_grouped_op<DT_F64>(op, items, count, scalar, st);
        case DT_F16:  return launch_grouped_op<DT_F16>(op, items, count, scalar, st);
        case DT_BF16: return launch_grouped_op<DT_BF16>(op, items, count, scalar, st);
    }
    return B200VA_ERR_VARIANT;
}

// ------------------------------------------------------------------ ceiling probes
int b200va_probe_f32(int kind, const float* dA, const float* dB, float* dC, size_t n, void* stream)
{
    if (kind < B200VA_PROBE_READ2 || kind > B200VA_PROBE_COPY) return B200VA_ERR_VARIANT;
    const b200va_devinfo_t* di = nullptr;
    RC_TRY(current_dev_info(&di));
    const size_t nvec = n / 4;
    if (nvec == 0) return B200VA_OK;
    if (!dC || (kind != B200VA_PROBE_FILL && !dA) || (kind == B200VA_PROBE_READ2 && !dB)) return B200VA_ERR_INVALID;
    const uintptr_t bits = reinterpret_cast<uintptr_t>(dC) | (kind != B200VA_PROBE_FILL ? reinterpret_cast<uintptr_t>(dA) : 0) |
                           (kind == B200VA_PROBE_READ2 ? reinterpret_cast<uintptr_t>(dB) : 0);
    if (bits & 15u) return B200VA_ERR_ALIGN;
    const size_t blocks = (nvec + 511) / 512;
    if (blocks > 0x7fffffffull) return B200VA_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned grid = static_cast<unsigned>(blocks);
    switch (kind) {
        case B200VA_PROBE_READ2: return launch_kernel(probe_read2, grid, 512u, 0, st, dA, dB, dC, nvec);
        case B200VA_PROBE_FILL:  return launch_kernel(probe_fill, grid, 512u, 0, st, dC, nvec, 1.0f);
        default:                 return launch_kernel(probe_copy, grid, 512u, 0, st, dA, dC, nvec);
    }
}

// ------------------------------------------------------------------ shard arithmetic
int b200va_shard_range(size_t n, int world, int rank, size_t* begin, size_t* end)
{
    if (world < 1 || rank < 0 || rank >= world || !begin || !end) return B200VA_ERR_INVALID;
    size_t chunk = (n + static_cast<size_t>(world) - 1) / static_cast<size_t>(world);
    chunk = (chunk + 7) & ~size_t{7};  // shard starts stay 32-byte aligned (256-bit body)
    size_t b = static_cast<size_t>(rank) * chunk;
    if (b > n) b = n;
    size_t e = b + chunk;
    if (e > n) e = n;
    *begin = b;
    *end = e;
    return B200VA_OK;
}

// ------------------------------------------------------------------ host-buffer path
// Restores the calling thread's current device on every exit path of the entry points that
// take a `device` argument (include/b200va.h: "restore the caller's current device").
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
        if (prev != device) err = cudaSetDevice(device);
    }
    ~DeviceGuard()
    {
        int now = -1;
        if (prev >= 0 && cudaGetDevice(&now) == cudaSuccess && now != prev) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// Fork-join pool for the pageable path: T persistent workers, each copies one slice.
// Construction may throw (std::system_error from std::thread under a pids limit, bad_alloc):
// make_copy_pool() catches and degrades, nothing propagates through the C ABI.
class CopyPool {
public:
    explicit CopyPool(int threads) : n_(threads < 1 ? 1 : threads)
    {
        th_.reserve(static_cast<size_t>(n_));
        try {
            for (int i = 1; i < n_; ++i) th_.emplace_back([this, i] { worker(i); });
        } catch (...) {
            n_ = static_cast<int>(th_.size()) + 1;          // run with the workers that did start
        }
    }
    ~CopyPool()
    {
        { std::lock_guard<std::mutex> lk(m_); stop_ = true; ++gen_; }
        cv_.notify_all();
        for (auto& t : th_) t.join();
    }
    int size() const { return n_; }
    // dst[0..bytes) = src[0..bytes), split in 64-byte-aligned slices over the pool (caller = slice 0)
    void copy(void* dst, const void* src, size_t bytes)
    {
        if (bytes < (size_t{1} << 20) || n_ == 1) { std::memcpy(dst, src, bytes); return; }
        {
            std::lock_guard<std::mutex> lk(m_);
            dst_ = static_cast<unsigned char*>(dst); src_ = static_cast<const unsigned char*>(src); bytes_ = bytes;
            pending_ = n_ - 1;
            ++gen_;
        }
        cv_.notify_all();
        slice(0);
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [this] { return pending_ == 0; });
    }

private:
    void slice(int i)
    {
        size_t per = (bytes_ + static_cast<size_t>(n_) - 1) / static_cast<size_t>(n_);
        per = (per + 63) & ~size_t{63};
        const size_t lo = std::min(bytes_, per * static_cast<size_t>(i)), hi = std::min(bytes_, lo + per);
        if (hi > lo) std::memcpy(dst_ + lo, src_ + lo, hi - lo);
    }
    void worker(int i)
    {
        unsigned long seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return gen_ != seen; });
                seen = gen_;
                if (stop_) return;
            }
            if (i < n_) slice(i);
            std::lock_guard<std::mutex> lk(m_);
            if (--pending_ == 0) done_.notify_one();
        }
    }
    int n_;
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    unsigned long gen_ = 0;
    int pending_ = 0;
    bool stop_ = false;
    unsigned char* dst_ = nullptr;
    const unsigned char* src_ = nullptr;
    size_t bytes_ = 0;
};

// Copy threads: the CPUs this process may use (affinity mask, cgroup v2 bandwidth quota), at
// most 16; B200VA_COPY_THREADS overrides (clamped to 1..64).  Never throws: returns nullptr
// only if even a single-threaded pool cannot be allocated.
static CopyPool* make_copy_pool()
{
    unsigned hw = std::thread::hardware_concurrency();
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof set, &set) == 0 && CPU_COUNT(&set) > 0) hw = static_cast<unsigned>(CPU_COUNT(&set));
    if (FILE* f = std::fopen("/sys/fs/cgroup/cpu.max", "r")) {
        char q[64];
        double period = 0;
        if (std::fscanf(f, "%63s %lf", q, &period) == 2 && std::strcmp(q, "max") != 0 && period > 0)
            hw = std::min(hw, static_cast<unsigned>(std::max(1.0, std::atof(q) / period)));
        std::fclose(f);
    }
    unsigned want = std::max(1u, std::min(16u, hw));
    if (const char* e = std::getenv("B200VA_COPY_THREADS")) want = static_cast<unsigned>(std::min(64, std::max(1, std::atoi(e))));
    for (; want >= 1; want /= 2) {
        try {
            return new CopyPool(static_cast<int>(want));
        } catch (...) {
            // bad_alloc / system_error while building the pool: retry smaller
        }
        if (want == 1) break;
    }
    return nullptr;
}

struct HostRange { uintptr_t lo, hi; };     // [lo, hi) page-locked by this stager (mode 4)

struct b200va_stager {
    int device = 0;
    size_t chunk = 0;
    int depth = 0;
    float* d_buf = nullptr;            // depth * 3 * chunk floats
    cudaStream_t main = nullptr;
    cudaStream_t* slot = nullptr;
    cudaEvent_t* slot_done = nullptr;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
    // "lanes" pipeline (mode 2): one stream per direction + one for the kernel, events per slot
    cudaStream_t lane_h2d = nullptr, lane_k = nullptr, lane_d2h = nullptr;
    cudaEvent_t *ev_in = nullptr, *ev_sum = nullptr, *ev_out = nullptr;
    // pageable path (mode 3): pinned bounce chunks (depth * 3 * bounce_chunk floats) + copy threads, made on first use
    float* bounce = nullptr;
    size_t bounce_chunk = 0;
    CopyPool* pool = nullptr;
    // register-once path (mode 4): host ranges this stager page-locked
    std::vector<HostRange>* regs = nullptr;
    float last_ms = 0.f;
    int last_mode = -1;
};

// NUMA node a CUDA device hangs off (sysfs), or -1.  B200VA_NUMA_NODE overrides.
static int device_numa_node_of(int dev)
{
    if (const char* e = std::getenv("B200VA_NUMA_NODE")) return std::atoi(e);
    char bus[32] = {0}, path[128];
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, dev) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* c = bus; *c; ++c) *c = static_cast<char>(std::tolower(*c));
    std::snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    int node = -1;
    if (FILE* f = std::fopen(path, "r")) {
        if (std::fscanf(f, "%d", &node) != 1) node = -1;
        std::fclose(f);
    }
    return node;
}

static int device_numa_node()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return -1; }
    return device_numa_node_of(dev);
}

// Parses a sysfs cpulist ("0-31,64-95") into a cpu_set_t restricted to `allowed`.
static bool node_cpuset(int node, const cpu_set_t& allowed, cpu_set_t* out)
{
    char path[96], buf[4096];
    std::snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    FILE* f = std::fopen(path, "r");
    if (!f) return false;
    const bool ok = std::fgets(buf, sizeof buf, f) != nullptr;
    std::fclose(f);
    if (!ok) return false;
    CPU_ZERO(out);
    int count = 0;
    for (char* p = buf; *p && *p != '\n';) {
        char* end = nullptr;
        long lo = std::strtol(p, &end, 10), hi = lo;
        if (end == p) break;
        if (*end == '-') hi = std::strtol(end + 1, &end, 10);
        for (long c = lo; c <= hi && c < CPU_SETSIZE; ++c)
            if (CPU_ISSET(c, &allowed)) { CPU_SET(c, out); ++count; }
        p = (*end == ',') ? end + 1 : end;
    }
    return count > 0;
}

// Pinned, mapped host memory whose pages sit on the NUMA node local to the current GPU:
// the calling thread is moved onto that node's CPUs (and its memory policy set to prefer
// the node) for the duration of the allocation, so the first touch inside cudaHostAlloc
// lands there; a PCIe DMA then never crosses the inter-socket link.  Affinity and memory
// policy of the caller (e.g. numactl --interleave) are saved and put back.
int b200va_host_alloc_ex(void** out, size_t bytes, int write_combined)
{
    if (!out) return B200VA_ERR_INVALID;
    const int node = device_numa_node();
    cpu_set_t old_set, node_set;
    bool moved = false, policy = false;
    int old_mode = 0;
    unsigned long old_mask[16] = {0};                       // 1024 nodes
    constexpr unsigned long kMaxNode = sizeof old_mask * 8;
    if (node >= 0 && sched_getaffinity(0, sizeof old_set, &old_set) == 0 && node_cpuset(node, old_set, &node_set)) {
        moved = sched_setaffinity(0, sizeof node_set, &node_set) == 0;
        if (node < 64 && syscall(SYS_get_mempolicy, &old_mode, old_mask, kMaxNode, nullptr, 0ul) == 0) {
            unsigned long mask = 1ul << node;
            policy = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, &mask, 65ul) == 0;
        }
    }
    unsigned flags = cudaHostAllocPortable | cudaHostAllocMapped;
    if (write_combined) flags |= cudaHostAllocWriteCombined;   // H2D sources only: CPU reads of WC memory crawl
    const cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, flags);
    if (policy) {
        bool any = false;
        for (unsigned long w : old_mask) any = any || w != 0;
        if (syscall(SYS_set_mempolicy, old_mode, any ? old_mask : nullptr, any ? kMaxNode : 0ul) != 0)
            syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
    }
    if (moved) sched_setaffinity(0, sizeof old_set, &old_set);
    CU_TRY(e);
    return B200VA_OK;
}

int b200va_host_alloc(void** out, size_t bytes) { return b200va_host_alloc_ex(out, bytes, 0); }

// NUMA node the current CUDA device is attached to (sysfs), or -1.
int b200va_device_numa_node(void) { return device_numa_node(); }
int b200va_device_numa_node_of(int device) { return device_numa_node_of(device); }

// NUMA node holding the page at `p` (get_mempolicy(MPOL_F_NODE | MPOL_F_ADDR)), or -1.
int b200va_host_node_of(const void* p)
{
    int node = -1;
    if (!p) return -1;
    if (syscall(SYS_get_mempolicy, &node, nullptr, 0ul, const_cast<void*>(p), 3ul /* F_NODE|F_ADDR */) != 0) return -1;
    return node;
}

int b200va_host_free(void* p)
{
    if (!p) return B200VA_OK;
    CU_TRY(cudaFreeHost(p));
    return B200VA_OK;
}

static void stager_release_host(b200va_stager* s)
{
    if (!s->regs) return;
    for (const HostRange& r : *s->regs)
        if (cudaHostUnregister(reinterpret_cast<void*>(r.lo)) != cudaSuccess) cudaGetLastError();
    s->regs->clear();
}

int b200va_stager_release_host(b200va_stager_t* s)
{
    if (!s) return B200VA_ERR_INVALID;
    DeviceGuard g(s->device);
    stager_release_host(s);
    return B200VA_OK;
}

int b200va_stager_destroy(b200va_stager_t* s)
{
    if (!s) return B200VA_OK;
    DeviceGuard g(s->device);
    stager_release_host(s);
    delete s->regs;
    if (s->slot) {
        for (int i = 0; i < s->depth; ++i) {
            if (s->slot[i]) cudaStreamDestroy(s->slot[i]);
            if (s->slot_done && s->slot_done[i]) cudaEventDestroy(s->slot_done[i]);
        }
    }
    for (cudaStream_t st : {s->lane_h2d, s->lane_k, s->lane_d2h})
        if (st) cudaStreamDestroy(st);
    for (cudaEvent_t* arr : {s->ev_in, s->ev_sum, s->ev_out}) {
        if (!arr) continue;
        for (int i = 0; i < s->depth; ++i)
            if (arr[i]) cudaEventDestroy(arr[i]);
        delete[] arr;
    }
    if (s->main) cudaStreamDestroy(s->main);
    if (s->ev_start) cudaEventDestroy(s->ev_start);
    if (s->ev_stop) cudaEventDestroy(s->ev_stop);
    if (s->d_buf) cudaFree(s->d_buf);
    if (s->bounce) cudaFreeHost(s->bounce);
    delete s->pool;
    delete[] s->slot;
    delete[] s->slot_done;
    delete s;
    return B200VA_OK;
}

int b200va_stager_create(b200va_stager_t** out, int device, size_t chunk_elems, int depth)
{
    if (!out) return B200VA_ERR_INVALID;
    *out = nullptr;
    if (chunk_elems == 0) chunk_elems = size_t{1} << 25;   // 128 MiB per array per slot (tapered tail: profiles/r01/u_*, v_*)
    if (depth == 0) depth = 3;
    if (depth < 1 || depth > 16) return B200VA_ERR_INVALID;
    chunk_elems = (chunk_elems + 63) & ~size_t{63};        // slots stay 256-B aligned
    RC_TRY(dev_info(device, nullptr));
    DeviceGuard guard(device);
    CU_TRY(guard.err);
    b200va_stager* s = new (std::nothrow) b200va_stager;
    if (!s) return B200VA_ERR_NOMEM;
    s->device = device;
    s->chunk = chunk_elems;
    s->depth = depth;
    s->slot = new (std::nothrow) cudaStream_t[depth]();
    s->slot_done = new (std::nothrow) cudaEvent_t[depth]();
    s->regs = new (std::nothrow) std::vector<HostRange>();
    if (!s->slot || !s->slot_done || !s->regs) { b200va_stager_destroy(s); return B200VA_ERR_NOMEM; }
    cudaError_t e = cudaMalloc(&s->d_buf, static_cast<size_t>(depth) * 3 * chunk_elems * sizeof(float));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->main, cudaStreamNonBlocking);
    for (int i = 0; i < depth && e == cudaSuccess; ++i) {
        e = cudaStreamCreateWithFlags(&s->slot[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->slot_done[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev_start);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev_stop);
    s->ev_in = new (std::nothrow) cudaEvent_t[depth]();
    s->ev_sum = new (std::nothrow) cudaEvent_t[depth]();
    s->ev_out = new (std::nothrow) cudaEvent_t[depth]();
    if (!s->ev_in || !s->ev_sum || !s->ev_out) { b200va_stager_destroy(s); return B200VA_ERR_NOMEM; }
    for (cudaStream_t* st : {&s->lane_h2d, &s->lane_k, &s->lane_d2h})
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(st, cudaStreamNonBlocking);
    for (int i = 0; i < depth && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&s->ev_in[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_sum[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_out[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) { b200va_stager_destroy(s); return cuda_err(e); }
    *out = s;
    return B200VA_OK;
}

// ---- the pipelines (device already current; a non-OK return leaves work in flight: the caller drains)
static int stage_zero_copy(b200va_stager* s, const float* hA, const float* hB, float* hC, size_t n, int variant)
{
    // the kernel streams A and B from pinned host memory over PCIe and writes C back the same
    // way -- both link directions busy, no staging latency.
    const float *dA = nullptr, *dB = nullptr;
    float* dC = nullptr;
    if (n) {
        CU_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(const_cast<float**>(&dA)), const_cast<float*>(hA), 0));
        CU_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(const_cast<float**>(&dB)), const_cast<float*>(hB), 0));
        CU_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(&dC), hC, 0));
    }
    b200va_tune_t t;
    default_tune(variant == B200VA_K_AUTO ? B200VA_K1_VEC128 : variant, n, &t);
    return launch(dA, dB, dC, n, t, s->main);
}

static int stage_slots(b200va_stager* s, const float* hA, const float* hB, float* hC, size_t n, int variant)
{
    const size_t nchunks = (n + s->chunk - 1) / s->chunk;
    for (int i = 0; i < s->depth; ++i) CU_TRY(cudaStreamWaitEvent(s->slot[i], s->ev_start, 0));
    b200va_tune_t t;
    for (size_t k = 0; k < nchunks; ++k) {
        const int i = static_cast<int>(k % static_cast<size_t>(s->depth));
        const size_t off = k * s->chunk;
        const size_t m = (n - off < s->chunk) ? n - off : s->chunk;
        float* dA = s->d_buf + static_cast<size_t>(i) * 3 * s->chunk;
        float* dB = dA + s->chunk;
        float* dC = dB + s->chunk;
        CU_TRY(cudaMemcpyAsync(dA, hA + off, m * sizeof(float), cudaMemcpyHostToDevice, s->slot[i]));
        CU_TRY(cudaMemcpyAsync(dB, hB + off, m * sizeof(float), cudaMemcpyHostToDevice, s->slot[i]));
        default_tune(variant, m, &t, B200VA_F_COLD);      // a chunk fresh off the copy engine is never in L2
        RC_TRY(launch(dA, dB, dC, m, t, s->slot[i]));
        CU_TRY(cudaMemcpyAsync(hC + off, dC, m * sizeof(float), cudaMemcpyDeviceToHost, s->slot[i]));
    }
    for (int i = 0; i < s->depth; ++i) {
        CU_TRY(cudaEventRecord(s->slot_done[i], s->slot[i]));
        CU_TRY(cudaStreamWaitEvent(s->main, s->slot_done[i], 0));
    }
    return B200VA_OK;
}

// Fault injection for the error-path test (tests/test_gpu_host_path.py): with
// B200VA_TEST_FAIL_CHUNK=k in the environment the lanes pipeline fails ONCE per process, right
// after it has queued chunk k's H2D copies -- i.e. with DMA in flight on the caller's arrays.
static bool inject_fault_at_chunk(size_t k)
{
    static const long at = [] { const char* e = std::getenv("B200VA_TEST_FAIL_CHUNK"); return e ? std::atol(e) : -1L; }();
    static std::atomic<bool> fired{false};
    return at >= 0 && static_cast<long>(k) == at && !fired.exchange(true);
}

static int stage_lanes(b200va_stager* s, const float* hA, const float* hB, float* hC, size_t n, int variant)
{
    // lanes: every H2D copy queues on one stream, every add on a second, every D2H on a
    // third; slot reuse and data flow are event edges.  The H2D queue -- the bottleneck
    // direction -- never waits behind a kernel or a D2H of another chunk.
    for (cudaStream_t st : {s->lane_h2d, s->lane_k, s->lane_d2h}) CU_TRY(cudaStreamWaitEvent(st, s->ev_start, 0));
    b200va_tune_t t;
    // Full-size chunks, then a tapered tail (1/2, 1/4, ... down to ~1 Mi elements): what is left
    // after the last H2D byte has arrived is one small add and one small D2H, not a full chunk.
    const size_t taper_min = size_t{1} << 20;
    size_t off = 0;
    for (size_t k = 0; off < n; ++k) {
        const size_t left = n - off;
        size_t m = s->chunk;
        if (left <= s->chunk && s->depth > 1) {
            m = left / 2;
            m = (m + 63) & ~size_t{63};                      // chunk starts stay 256-byte aligned
            if (m < taper_min || m >= left) m = left;
        }
        if (m > left) m = left;
        const int i = static_cast<int>(k % static_cast<size_t>(s->depth));
        float* dA = s->d_buf + static_cast<size_t>(i) * 3 * s->chunk;
        float* dB = dA + s->chunk;
        float* dC = dB + s->chunk;
        if (k >= static_cast<size_t>(s->depth)) CU_TRY(cudaStreamWaitEvent(s->lane_h2d, s->ev_out[i], 0));  // slot drained
        CU_TRY(cudaMemcpyAsync(dA, hA + off, m * sizeof(float), cudaMemcpyHostToDevice, s->lane_h2d));
        CU_TRY(cudaMemcpyAsync(dB, hB + off, m * sizeof(float), cudaMemcpyHostToDevice, s->lane_h2d));
        CU_TRY(cudaEventRecord(s->ev_in[i], s->lane_h2d));
        if (inject_fault_at_chunk(k)) return B200VA_ERR_INVALID;   // test hook: fail with copies in flight
        CU_TRY(cudaStreamWaitEvent(s->lane_k, s->ev_in[i], 0));
        default_tune(variant, m, &t, B200VA_F_COLD);      // a chunk fresh off the copy engine is never in L2
        RC_TRY(launch(dA, dB, dC, m, t, s->lane_k));
        CU_TRY(cudaEventRecord(s->ev_sum[i], s->lane_k));
        CU_TRY(cudaStreamWaitEvent(s->lane_d2h, s->ev_sum[i], 0));
        CU_TRY(cudaMemcpyAsync(hC + off, dC, m * sizeof(float), cudaMemcpyDeviceToHost, s->lane_d2h));
        CU_TRY(cudaEventRecord(s->ev_out[i], s->lane_d2h));
        off += m;
    }
    CU_TRY(cudaEventRecord(s->slot_done[0], s->lane_d2h));   // the D2H lane finishes last
    CU_TRY(cudaStreamWaitEvent(s->main, s->slot_done[0], 0));
    return B200VA_OK;
}

static int stage_bounce(b200va_stager* s, const float* hA, const float* hB, float* hC, size_t n, int variant)
{
    // Pageable host arrays (plain malloc, what one ./vectorAdd process has): a cudaMemcpy from
    // pageable memory is staged by the driver on one thread at ~10 GB/s.  Here a pool of host
    // threads copies chunk k+1 into pinned bounce buffers and chunk k-2 out of them while the
    // copy engines and the add work on the chunks in between (lanes as in mode 2).
    const size_t bc = std::min(s->chunk, size_t{1} << 23);          // 32 MiB bounce chunks
    if (!s->pool) {
        s->pool = make_copy_pool();
        if (!s->pool) return B200VA_ERR_NOMEM;
    }
    if (!s->bounce || s->bounce_chunk != bc) {
        if (s->bounce) { cudaFreeHost(s->bounce); s->bounce = nullptr; }
        void* p = nullptr;
        RC_TRY(b200va_host_alloc(&p, static_cast<size_t>(s->depth) * 3 * bc * sizeof(float)));
        s->bounce = static_cast<float*>(p);
        s->bounce_chunk = bc;
    }
    for (cudaStream_t st : {s->lane_h2d, s->lane_k, s->lane_d2h}) CU_TRY(cudaStreamWaitEvent(st, s->ev_start, 0));
    const size_t nchunks = (n + bc - 1) / bc;
    const size_t depth = static_cast<size_t>(s->depth);
    b200va_tune_t t;
    auto span = [&](size_t k, size_t* off, size_t* m) { *off = k * bc; *m = std::min(bc, n - *off); };
    for (size_t k = 0; k < nchunks + depth - 1 || k < nchunks; ++k) {
        if (k < nchunks) {
            size_t off, m;
            span(k, &off, &m);
            const size_t i = k % depth;
            float* pA = s->bounce + i * 3 * bc;
            float* dA = s->d_buf + i * 3 * s->chunk;
            // slot i was drained (copied out) at iteration k-1 below, or never used
            s->pool->copy(pA, hA + off, m * sizeof(float));
            s->pool->copy(pA + bc, hB + off, m * sizeof(float));
            CU_TRY(cudaMemcpyAsync(dA, pA, m * sizeof(float), cudaMemcpyHostToDevice, s->lane_h2d));
            CU_TRY(cudaMemcpyAsync(dA + s->chunk, pA + bc, m * sizeof(float), cudaMemcpyHostToDevice, s->lane_h2d));
            CU_TRY(cudaEventRecord(s->ev_in[i], s->lane_h2d));
            CU_TRY(cudaStreamWaitEvent(s->lane_k, s->ev_in[i], 0));
            default_tune(variant, m, &t, B200VA_F_COLD);
            RC_TRY(launch(dA, dA + s->chunk, dA + 2 * s->chunk, m, t, s->lane_k));
            CU_TRY(cudaEventRecord(s->ev_sum[i], s->lane_k));
            CU_TRY(cudaStreamWaitEvent(s->lane_d2h, s->ev_sum[i], 0));
            CU_TRY(cudaMemcpyAsync(pA + 2 * bc, dA + 2 * s->chunk, m * sizeof(float), cudaMemcpyDeviceToHost, s->lane_d2h));
            CU_TRY(cudaEventRecord(s->ev_out[i], s->lane_d2h));
        }
        if (k + 1 >= depth) {                                       // retire chunk j = k - (depth - 1)
            const size_t j = k + 1 - depth;
            if (j < nchunks) {
                size_t off, m;
                span(j, &off, &m);
                const size_t i = j % depth;
                CU_TRY(cudaEventSynchronize(s->ev_out[i]));
                s->pool->copy(hC + off, s->bounce + i * 3 * bc + 2 * bc, m * sizeof(float));
            }
        }
    }
    CU_TRY(cudaEventRecord(s->slot_done[0], s->lane_d2h));
    CU_TRY(cudaStreamWaitEvent(s->main, s->slot_done[0], 0));
    return B200VA_OK;
}

static bool host_is_pinned(const void* p)
{
    cudaPointerAttributes at{};
    const bool ok = cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type != cudaMemoryTypeUnregistered;
    if (!ok) cudaGetLastError();
    return ok;
}

// Page-locks [p, p+bytes) in place unless the runtime already knows it (cudaHostAlloc'd,
// registered by the caller, or by this stager earlier).  Returns false if the range cannot be
// registered -- the caller then falls back to the bounce path.
static bool ensure_registered(b200va_stager* s, const void* p, size_t bytes)
{
    if (bytes == 0) return true;
    const uintptr_t lo = reinterpret_cast<uintptr_t>(p), hi = lo + bytes;
    for (const HostRange& r : *s->regs)
        if (r.lo <= lo && hi <= r.hi) return true;                  // cached
    if (host_is_pinned(p) && host_is_pinned(reinterpret_cast<const void*>(hi - 1))) return true;
    // a cached range that overlaps without containing the new one (the caller's buffer moved or grew): drop it
    for (size_t i = 0; i < s->regs->size();) {
        const HostRange r = (*s->regs)[i];
        if (r.lo < hi && lo < r.hi) {
            if (cudaHostUnregister(reinterpret_cast<void*>(r.lo)) != cudaSuccess) cudaGetLastError();
            s->regs->erase(s->regs->begin() + static_cast<long>(i));
        } else {
            ++i;
        }
    }
    const cudaError_t e = cudaHostRegister(const_cast<void*>(p), bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    try {
        s->regs->push_back(HostRange{lo, hi});
    } catch (...) {
        cudaHostUnregister(const_cast<void*>(p));
        return false;
    }
    return true;
}

static void stager_drain(b200va_stager* s)
{
    // after a failure in the middle of a pipeline: nothing may still be reading or writing the
    // caller's arrays (or the bounce ring) when the error code is returned
    for (int i = 0; i < s->depth; ++i)
        if (s->slot && s->slot[i]) cudaStreamSynchronize(s->slot[i]);
    for (cudaStream_t st : {s->lane_h2d, s->lane_k, s->lane_d2h, s->main})
        if (st) cudaStreamSynchronize(st);
    cudaGetLastError();
}

int b200va_stager_add_f32(b200va_stager_t* s, const float* hA, const float* hB, float* hC, size_t n,
                          int variant, int mode)
{
    if (!s || (n && (!hA || !hB || !hC))) return B200VA_ERR_INVALID;
    if (variant < B200VA_K_AUTO || variant > B200VA_K3_VEC256) return B200VA_ERR_VARIANT;
    if (mode < B200VA_STAGE_AUTO || mode > B200VA_STAGE_REGISTER) return B200VA_ERR_INVALID;
    DeviceGuard guard(s->device);
    CU_TRY(guard.err);
    const size_t bytes = n * sizeof(float);
    if (mode == B200VA_STAGE_AUTO) {
        const bool pinned = n == 0 || (host_is_pinned(hA) && host_is_pinned(hB) && host_is_pinned(hC));
        mode = pinned ? B200VA_STAGE_LANES : (3 * bytes >= (size_t{8} << 20) ? B200VA_STAGE_REGISTER : B200VA_STAGE_BOUNCE);
    }
    if (mode == B200VA_STAGE_REGISTER) {
        // page-lock the caller's arrays once (outside the timed pipeline: it is a one-off cost of the first call)
        const bool ok = ensure_registered(s, hA, bytes) && ensure_registered(s, hB, bytes) && ensure_registered(s, hC, bytes);
        if (!ok) mode = B200VA_STAGE_BOUNCE;
    }
    s->last_mode = mode;
    CU_TRY(cudaEventRecord(s->ev_start, s->main));
    int rc = B200VA_OK;
    switch (mode) {
        case B200VA_STAGE_ZEROCOPY: rc = stage_zero_copy(s, hA, hB, hC, n, variant); break;
        case B200VA_STAGE_SLOTS:    rc = stage_slots(s, hA, hB, hC, n, variant); break;
        case B200VA_STAGE_LANES:
        case B200VA_STAGE_REGISTER: rc = stage_lanes(s, hA, hB, hC, n, variant); break;
        case B200VA_STAGE_BOUNCE:   rc = stage_bounce(s, hA, hB, hC, n, variant); break;
    }
    if (rc == B200VA_OK) rc = cuda_err(cudaEventRecord(s->ev_stop, s->main));
    if (rc == B200VA_OK) rc = cuda_err(cudaStreamSynchronize(s->main));
    if (rc != B200VA_OK) { stager_drain(s); return rc; }
    CU_TRY(cudaEventElapsedTime(&s->last_ms, s->ev_start, s->ev_stop));
    return B200VA_OK;
}

int b200va_stager_last_ms(b200va_stager_t* s, float* ms)
{
    if (!s || !ms) return B200VA_ERR_INVALID;
    *ms = s->last_ms;
    return B200VA_OK;
}

int b200va_stager_last_mode(b200va_stager_t* s, int* mode)
{
    if (!s || !mode) return B200VA_ERR_INVALID;
    *mode = s->last_mode;
    return B200VA_OK;
}

int b200va_add_f32_host(const float* hA, const float* hB, float* hC, size_t n, int device, int variant)
{
    b200va_stager_t* s = nullptr;
    size_t chunk = size_t{1} << 25;
    if (n < chunk) chunk = n ? n : 1;
    RC_TRY(dev_info(device, nullptr));
    DeviceGuard guard(device);          // cudaPointerGetAttributes below needs a current device; restored on return
    CU_TRY(guard.err);
    // pinned/registered arrays go straight to the copy engines; pageable ones through the bounce pool
    // (one-shot: page-locking 3 arrays for a single pass costs more than bouncing them)
    const bool pageable = n && !(host_is_pinned(hA) && host_is_pinned(hB) && host_is_pinned(hC));
    // pinning the bounce ring costs ~0.35 ms/MiB, so keep it small (9 x 8 MiB)
    if (pageable && chunk > (size_t{1} << 21)) chunk = size_t{1} << 21;
    RC_TRY(b200va_stager_create(&s, device, chunk, n > chunk ? 3 : 1));
    const int rc = b200va_stager_add_f32(s, hA, hB, hC, n, variant, pageable ? B200VA_STAGE_BOUNCE : B200VA_STAGE_LANES);
    b200va_stager_destroy(s);
    return rc;
}

}  // extern "C"
