/*
 * b200va.h -- C ABI of libb200va.so: the B200 (sm_100a) vectorAdd hot path.
 *
 * The reference (ashrafgt/k8s-gpu-hpa) has NO library/plugin API for this path: the
 * kernel is statically linked into the `vectorAdd` executable inside the third-party
 * image k8s.gcr.io/cuda-vector-add:v0.1, and the reference only invokes it:
 *
 *     image:   "k8s.gcr.io/cuda-vector-add:v0.1"                     cuda-test-deployment.yaml:18
 *     command: for (( c=1; c<=5000; c++ )); do ./vectorAdd; done     cuda-test-deployment.yaml:19
 *     (same loop started by hand to raise utilisation)               README.md:113-116
 *
 * The outer drop-in boundary is therefore the `vectorAdd` executable
 * (k8s-gpu-hpa_b200/host/vectorAdd.cpp).  This header is the inner boundary the
 * executable -- and any other host language via cgo/JNI/ctypes -- binds: each entry
 * point below names the step of that process (SURVEY.md section 8(a), rows a1-a7) it
 * replaces.  See INTEGRATION.md for the binding stubs.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++ or torch types, no exceptions.
 *   - Functions return 0 (B200VA_OK) or a negative code; they never print or abort.
 *     CUDA runtime failures are returned as  -(1000 + cudaError_t).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *     Device entry points are asynchronous on that stream: no hidden synchronisation,
 *     no hidden allocation; the caller owns every buffer.
 *   - The current CUDA device of the calling thread is used (cudaSetDevice first);
 *     the library is re-entrant and keeps only immutable per-device attribute caches.
 *     Entry points that take a `device` argument (stager, b200va_add_f32_host, b200va_query)
 *     restore the caller's current device before returning, on every path.
 *   - Element type is IEEE-754 binary32; the add is add.rn.f32 without FTZ, so results
 *     are bit-identical to a scalar C loop on the same inputs (NaN payloads excepted:
 *     PTX returns the canonical NaN 0x7fffffff).
 */
#ifndef B200VA_H
#define B200VA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200VA_ABI_VERSION 2   /* 2: b200va_tune_t grew early_loads/scheduler; *_ex, stager modes 4/AUTO */

/* ---- status codes ------------------------------------------------------------- */
#define B200VA_OK               0
#define B200VA_ERR_INVALID     (-1)   /* NULL pointer with n > 0, bad argument            */
#define B200VA_ERR_ALIGN       (-2)   /* pointer not 4-byte aligned                       */
#define B200VA_ERR_OVERLAP     (-3)   /* C partially overlaps A or B (exact alias is ok)  */
#define B200VA_ERR_VARIANT     (-4)   /* unknown kernel variant / unsupported tune combo  */
#define B200VA_ERR_NO_DEVICE   (-5)   /* no CUDA device / not an sm_100 device            */
#define B200VA_ERR_VERIFY      (-6)   /* result verification failed (a6)                  */
#define B200VA_ERR_NOMEM       (-7)   /* host allocation failed                           */
#define B200VA_ERR_CUDA_BASE   (-1000) /* code = -(1000 + cudaError_t)                    */
/* Which combinations a library carries: libb200va.so ships the production set (what
 * B200VA_K_AUTO and the named variants resolve to, plus a few neighbours); the full
 * A/B matrix of b200va_tune_t lives in libb200va_tune.so (same ABI, development only).
 * A combination the loaded library does not carry returns B200VA_ERR_VARIANT. */

/* ---- kernel variants (argument `variant`) ---------------------------------------- */
#define B200VA_K_AUTO      0   /* the tuned production choice for this n                */
#define B200VA_K0_SCALAR   1   /* reference-shape control: 1 elem/thread, 256-thread CTAs,
                                  (n+255)/256 CTAs  (CUDA sample launch geometry, a5)   */
#define B200VA_K1_VEC128   2   /* 128-bit ld/st.global.v4.f32, unrolled, cache-hinted   */
#define B200VA_K2_TMA      3   /* cp.async.bulk (TMA) smem ring; tiles handed out by the
                                  cluster-launch-control scheduler (store_mode 2)        */
#define B200VA_K3_VEC256   4   /* 256-bit ld/st.global.v8.f32 (PTX 8.8, sm_100)         */
#define B200VA_K4_SCALAR_MLP 5 /* 32-bit accesses, `unroll` (4|8|16) independent loads per array
                                  per thread in flight: the mixed-misalignment path, also
                                  selectable through b200va_add_f32_tuned for A/B runs   */

/* Explicit geometry for A/B experiments (b200va_add_f32_tuned). Zero = default.      */
typedef struct b200va_tune {
    int kind;         /* B200VA_K0_SCALAR .. B200VA_K3_VEC256                           */
    int threads;      /* CTA size (vec kernels) or consumer threads (TMA kernel)        */
    int unroll;       /* vec: vectors per thread per tile: 1,2,4,8                      */
    int ctas_per_sm;  /* 0: one tile per CTA; >0: persistent grid = SMs * ctas_per_sm   */
    int ld_hint;      /* 0 plain, 1 L1::no_allocate, 2 .cs, 3 no_allocate+L2 evict_first, 4 .nc+no_allocate, 5 no_allocate+L2::256B */
    int st_hint;      /* 0 plain, 1 L1::no_allocate,   2 .cs, 3 no_allocate+L2 evict_first */
    int stages;       /* TMA: ring depth (2..16)                                        */
    int tile_bytes;   /* TMA: bytes per array per stage (multiple of 2048)              */
    int store_mode;   /* TMA: 0 = st.global from registers, 1 = bulk store from smem,
                         2 = register stores + cluster-launch-control tile scheduler    */
    int early_loads;  /* vec: what a CTA does about its first tile before the programmatic
                         dependency on the previous launch resolves:
                         1 = issue the loads themselves (only the stores wait).  Requires that
                             the previous launch on the stream does not write A or B; replaced
                             by 2 when C aliases A or B.  See b200va_add_f32_ex.
                         2 = bulk-prefetch the A and B tiles into L2 (cp.async.bulk.prefetch.L2);
                             loads and stores wait.  Always legal (L2 is the coherence point);
                             pays off on data that is not already in L2.                     */
    int scheduler;    /* vec: 0 = hardware block scheduler (one CTA per tile, or the static
                         persistent split of ctas_per_sm), 1 = cluster launch control:
                         resident CTAs cancel and take over not-yet-started ones (K1c)   */
} b200va_tune_t;

typedef struct b200va_devinfo {
    int device;
    int cc_major, cc_minor;
    int sm_count;
    int max_smem_optin;        /* bytes                                                 */
    int l2_bytes;
    size_t global_mem_bytes;
    char name[64];
} b200va_devinfo_t;

/* ---- library ----------------------------------------------------------------------- */
int         b200va_abi_version(void);
const char *b200va_strerror(int code);
/* Attributes of `device` (does not change the current device). */
int         b200va_query(int device, b200va_devinfo_t *out);
/* The geometry B200VA_K_AUTO (or a named variant) resolves to for n elements; the _ex form
 * takes the B200VA_F_* hints b200va_add_f32_ex takes. */
int         b200va_resolve(int variant, size_t n, b200va_tune_t *out);
int         b200va_resolve_ex(int variant, size_t n, unsigned flags, b200va_tune_t *out);

/* Launch geometry a tune resolves to on `device` for n elements with 32-byte-aligned
 * pointers (what "CUDA kernel launch with %d blocks of %d threads" prints, a5). */
int         b200va_geometry(const b200va_tune_t *tune, size_t n, int device,
                            unsigned *grid, unsigned *block, unsigned *dyn_smem_bytes);

/* ---- a4 + a5: the vectorAdd kernel and its launch geometry -------------------------
 * Replaces `vectorAdd<<<blocksPerGrid, threadsPerBlock>>>(d_A, d_B, d_C, numElements)`
 * of the image's binary (invoked at cuda-test-deployment.yaml:19).
 * dA, dB, dC: device pointers, 4-byte aligned; any n >= 0; dC may equal dA or dB. */
int b200va_add_f32(const float *dA, const float *dB, float *dC, size_t n,
                   int variant, void *stream);
int b200va_add_f32_tuned(const float *dA, const float *dB, float *dC, size_t n,
                         const b200va_tune_t *tune, void *stream);
/* Same as b200va_add_f32 with launch-ordering hints (`flags`, OR of B200VA_F_*).
 * B200VA_F_INPUTS_STABLE: the caller promises that the launch immediately preceding this
 * one on `stream` does not write A or B (e.g. it is another add into a different or the
 * same C).  The kernel then issues its loads while that launch is still draining and only
 * its stores wait for it (programmatic dependent launch), which removes most of the
 * ~2 us bubble between back-to-back launches.  Results and stream order of C are
 * unchanged; the flag is ignored when C aliases A or B. */
#define B200VA_F_INPUTS_STABLE 1u
/* B200VA_F_COLD: the operands are not L2-resident (fresh from a copy engine, or one of many
 * buffer sets touched in rotation): B200VA_K_AUTO then resolves to the geometry tuned on
 * rotating buffers instead of the one tuned for relaunching the same buffers -- in particular
 * the launch prefetches its first tiles into L2 while the previous launch is still draining
 * (early_loads = 2; no promise about the previous launch is needed for that).  A hint only;
 * vectors of 2^25 elements and more can never be L2-resident and are always treated as cold. */
#define B200VA_F_COLD          2u
int b200va_add_f32_ex(const float *dA, const float *dB, float *dC, size_t n,
                      int variant, unsigned flags, void *stream);

/* ---- a1: the launch loop, in-process -----------------------------------------------
 * Replaces the 5000-process bash loop (cuda-test-deployment.yaml:19): `iters`
 * back-to-back launches on `stream`; graph_batch > 1 captures that many launches into
 * one CUDA graph and replays it (launch-bound sizes).  Asynchronous, except that the
 * graph form (graph_batch > 1) drains the stream before returning; any capturable or
 * legacy stream is accepted (the capture happens on a private stream).
 * Launches 2..iters of a loop know their predecessor (the same add, which writes only C),
 * so unless C aliases A or B they run with early loads (see B200VA_F_INPUTS_STABLE). */
int b200va_add_f32_loop(const float *dA, const float *dB, float *dC, size_t n,
                        int variant, int iters, int graph_batch, void *stream);
/* Persistent form for a long-running load generator: the graph of `graph_batch` launches
 * is captured once; b200va_loop_run replays it floor(iters/graph_batch) times plus
 * iters%graph_batch direct launches, asynchronously on `stream`.  Destroy only after
 * the stream has drained. */
typedef struct b200va_loop b200va_loop_t;
int b200va_loop_create(b200va_loop_t **out, const float *dA, const float *dB, float *dC,
                       size_t n, int variant, int graph_batch);
int b200va_loop_run(b200va_loop_t *loop, int iters, void *stream);
int b200va_loop_destroy(b200va_loop_t *loop);

/* ---- a2: input recipes ---------------------------------------------------------------
 * Host: the sample's recipe  h_A[i] = rand()/(float)RAND_MAX; h_B[i] = ... interleaved,
 * never seeded.  Reseeds glibc to 1 so every call equals a fresh ./vectorAdd process. */
int b200va_host_fill_rand_f32(float *hA, float *hB, size_t n);
/* Counter generator for large n (index-addressable, shard-invariant):
 * x[i] = (float)(splitmix64(seed*0x9E3779B97F4A7C15 + first + i) >> 40) * 2^-24.       */
int b200va_host_fill_ctr_f32(float *h, size_t n, uint64_t seed, uint64_t first);
int b200va_fill_ctr_f32(float *d, size_t n, uint64_t seed, uint64_t first, void *stream);

/* ---- a6: verification ----------------------------------------------------------------
 * Host: the sample's check made strict: bitwise C[i] == A[i]+B[i] (NaNs as a class).
 * Returns B200VA_OK or B200VA_ERR_VERIFY with *first_bad = failing index.            */
int b200va_host_verify_f32(const float *hA, const float *hB, const float *hC, size_t n,
                           size_t *first_bad);
/* Device: recompute + bit-compare in HBM.  d_result[0] = mismatch count,
 * d_result[1] = first mismatching index (UINT64_MAX if none).  Asynchronous; the
 * caller zero-inits nothing (the call resets d_result on the stream first).          */
int b200va_verify_f32(const float *dA, const float *dB, const float *dC, size_t n,
                      uint64_t *d_result, void *stream);
/* Device digest of a vector's bit patterns: d_out[0] = sum of uint32 patterns mod 2^64,
 * d_out[1] = xor of them.  Order-independent, so shards combine by + and ^.          */
int b200va_digest_f32(const float *d, size_t n, uint64_t *d_out, void *stream);

/* ---- a3 + a4 + a6(copy) : host-buffer path -------------------------------------------
 * Replaces cudaMalloc x3 / cudaMemcpy H2D x2 / kernel / cudaMemcpy D2H of one
 * ./vectorAdd run, for host arrays of any size: a staged, double-direction pipeline
 * (H2D of chunk k+1, add of chunk k, D2H of chunk k-1 overlap on separate streams).
 * A stager owns its device staging buffers and streams; create one per device/thread. */
typedef struct b200va_stager b200va_stager_t;
/* mode 0: copy-engine pipeline through HBM staging buffers;
 * mode 1: zero-copy kernel reading/writing pinned host memory directly over PCIe
 *         (requires all three host buffers pinned/registered);
 * mode 2: "lanes" pipeline: one stream per direction plus one for the adds, event edges
 *         per slot, so the H2D queue never waits behind another chunk's kernel or D2H;
 * mode 3: pageable host arrays (plain malloc): host threads copy chunks through pinned
 *         bounce buffers around the lanes pipeline.  b200va_add_f32_host picks 2 or 3
 *         by asking the runtime whether the arrays are pinned.
 * mode 4: register-once: pageable arrays are page-locked in place (cudaHostRegister) the
 *         first time the stager sees them and the registration is cached by address range,
 *         so a long-lived loop over the same malloc'd arrays -- the reference process's
 *         shape -- runs the lanes pipeline at the pinned rate from the second call on.
 *         The first call pays the pinning (~0.3 ms/MiB).  Registered arrays must stay
 *         allocated until b200va_stager_release_host / b200va_stager_destroy.  Falls back
 *         to mode 3 if the registration is refused (RLIMIT_MEMLOCK, exotic mappings).
 * mode -1 (B200VA_STAGE_AUTO): mode 2 for pinned arrays, mode 4 for pageable arrays of at
 *         least 8 MiB in total, mode 3 below that. */
#define B200VA_STAGE_AUTO      (-1)
#define B200VA_STAGE_SLOTS       0
#define B200VA_STAGE_ZEROCOPY    1
#define B200VA_STAGE_LANES       2
#define B200VA_STAGE_BOUNCE      3
#define B200VA_STAGE_REGISTER    4
/* chunk_elems = 0 -> 32 Mi elements (128 MiB per array per slot), depth = 0 -> 3 slots.
 * The lanes pipeline tapers the last chunk (1/2, 1/4, ... ~1 Mi) so the D2H tail is short. */
int b200va_stager_create(b200va_stager_t **out, int device, size_t chunk_elems, int depth);
/* Synchronous.  On an error in the middle of the pipeline every stream of the stager is
 * drained before the call returns, so no copy is still touching the caller's arrays. */
int b200va_stager_add_f32(b200va_stager_t *s, const float *hA, const float *hB, float *hC,
                          size_t n, int variant, int mode);
/* Device-side time of the last b200va_stager_add_f32 call, milliseconds (events). */
int b200va_stager_last_ms(b200va_stager_t *s, float *ms);
/* The mode the last b200va_stager_add_f32 call actually ran (after AUTO / fallbacks). */
int b200va_stager_last_mode(b200va_stager_t *s, int *mode);
/* Unregister every host range the stager page-locked (mode 4); call before freeing them
 * if the stager outlives the arrays.  b200va_stager_destroy does this too. */
int b200va_stager_release_host(b200va_stager_t *s);
int b200va_stager_destroy(b200va_stager_t *s);
/* One-shot convenience: create, add, destroy (synchronous). */
int b200va_add_f32_host(const float *hA, const float *hB, float *hC, size_t n,
                        int device, int variant);
/* Pinned, mapped host memory for the pipeline (cudaHostAlloc / cudaFreeHost), placed on
 * the NUMA node of the current CUDA device.  write_combined != 0 adds
 * cudaHostAllocWriteCombined: meant for H2D *sources* the CPU only writes. */
int b200va_host_alloc(void **out, size_t bytes);
int b200va_host_alloc_ex(void **out, size_t bytes, int write_combined);
int b200va_host_free(void *p);
/* NUMA node that holds the page at p, or -1 if it cannot be determined. */
int b200va_host_node_of(const void *p);
/* NUMA node the current CUDA device is attached to, or -1. */
int b200va_device_numa_node(void);
/* Same for `device`, without making it current (no context is created). */
int b200va_device_numa_node_of(int device);

/* ---- generalised streaming element-wise core (SURVEY.md 8(f) row 4) -------------------
 * The tuned 128-bit streaming skeleton of the vectorAdd kernel over other element types
 * and STREAM operations.  Not part of the reference's surface (its only op is the f32
 * add, for which  b200va_stream(ADD, F32, ...)  is bit-identical to  b200va_add_f32).
 *   COPY  c = a            SCALE c = s*a          ADD c = a + b      TRIAD c = fma(s, b, a)
 * f32/f64: native IEEE arithmetic, round-to-nearest-even, no FTZ.  f16/bf16: operands
 * widened exactly to f32, op in f32 (s rounded to f32), result rounded to nearest-even.
 * dB is ignored (may be NULL) for COPY and SCALE.  Pointers aligned to the element size. */
#define B200VA_OP_COPY   0
#define B200VA_OP_SCALE  1
#define B200VA_OP_ADD    2
#define B200VA_OP_TRIAD  3
#define B200VA_DT_F32    0
#define B200VA_DT_F64    1
#define B200VA_DT_F16    2
#define B200VA_DT_BF16   3
int b200va_stream(int op, int dtype, const void *dA, const void *dB, void *dC, size_t n,
                  double scalar, void *stream);

/* Grouped form: one op and dtype over many independent vectors, in as few launches as the
 * kernel parameter block allows (800 items per launch; larger calls are split at item
 * boundaries into launches enqueued in order on `stream`).  Many small vectors then cost one
 * launch boundary instead of one each -- the torch._foreach_* / multi-tensor-apply shape.
 *   - Each item's result is bit-identical to  b200va_stream(op, dtype, a, b, c, n, scalar, stream).
 *   - Asynchronous on `stream`, current device; no hidden allocation or synchronisation, so the
 *     call can be captured into a CUDA graph.  `items` is host memory, read before the call
 *     returns: the caller may reuse the array at once.
 *   - Every item is checked before anything is enqueued, with the checks of b200va_stream
 *     (NULL with n > 0 or n > 2^40: ERR_INVALID; not aligned to the element size: ERR_ALIGN;
 *     C partially overlapping its own A or B: ERR_OVERLAP, exact aliasing is fine).  On a
 *     failure nothing is enqueued and the first failing item's code is returned.
 *   - count == 0 is a no-op; items == NULL with count > 0 is ERR_INVALID; an unknown op or
 *     dtype is ERR_VARIANT.  Items with n == 0 are skipped (their pointers may be NULL).
 *   - PRECONDITION, not checked: items are independent -- no item's C overlaps another item's
 *     A, B or C.  Items run concurrently in no defined order.  (Checking this needs a sort of
 *     the address ranges, tens of microseconds of host time per call: more than the GPU time
 *     of a small batch.) */
typedef struct b200va_item {
    const void *a;      /* input A (device)                                       */
    const void *b;      /* input B (device); ignored, may be NULL, for COPY/SCALE */
    void       *c;      /* output C (device)                                      */
    size_t      n;      /* elements; 0 = skipped (pointers may then be NULL)      */
} b200va_item_t;
int b200va_stream_grouped(int op, int dtype, const b200va_item_t *items, size_t count,
                          double scalar, void *stream);

/* ---- ceiling probes (measurement aids; not part of the reference's surface) -------------
 * The production launch geometry with one side of the add's traffic removed, so a harness can
 * measure on the spot what the HBM gives each kind of stream (bench.py reports the add as a
 * fraction of the READ2 rate).  n is rounded down to a multiple of 4; pointers 16-byte aligned.
 *   READ2  load A and B, store one float per CTA into C (8 B/element read)
 *   FILL   C = 1.0f, nothing is read                       (4 B/element written)
 *   COPY   C = A                                            (4 B read + 4 B written per element) */
#define B200VA_PROBE_READ2  0
#define B200VA_PROBE_FILL   1
#define B200VA_PROBE_COPY   2
int b200va_probe_f32(int kind, const float *dA, const float *dB, float *dC, size_t n, void *stream);

/* ---- shard arithmetic (8(e)): contiguous equal shards, starts on 16-byte multiples --- */
int b200va_shard_range(size_t n, int world, int rank, size_t *begin, size_t *end);

#ifdef __cplusplus
}
#endif
#endif /* B200VA_H */
