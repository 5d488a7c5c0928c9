// gort_abi.cu -- the extern "C" boundary of libgort_b200 (include/gort_b200.h): context, device
// scratch management, host-pointer wrappers (H2D -> kernels -> D2H) and the LUT text layout.
// No model arithmetic lives here; there is no CPU fallback.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <sched.h>
#include <vector>
#include "gort_internal.h"
#include "../data/gort_tables.h"

static char g_create_error[512] = "";

namespace gort {

int set_error(gort_ctx *ctx, int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(ctx ? ctx->err : g_create_error, 512, fmt, ap);
    va_end(ap);
    return code;
}

int check_cuda(gort_ctx *ctx, cudaError_t e, const char *what)
{
    if (e == cudaSuccess) return GORT_OK;
    return set_error(ctx, GORT_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

static void *grow(gort_ctx *ctx, void **p, size_t *cap, size_t bytes)
{
    if (bytes == 0) bytes = 8;
    if (*cap >= bytes) return *p;
    // the buffer may still be in use by work enqueued earlier (on the context's stream or on a
    // caller-supplied one); regrowth is rare, so wait for the whole device
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { set_error(ctx, GORT_ERR_CUDA, "device synchronize before regrowing a buffer: %s", cudaGetErrorString(e)); return NULL; }
    if (*p) {
        e = cudaFree(*p);
        if (e != cudaSuccess) { set_error(ctx, GORT_ERR_CUDA, "cudaFree while regrowing a buffer: %s", cudaGetErrorString(e)); return NULL; }
    }
    *p = NULL; *cap = 0;
    size_t want = bytes + bytes / 8;
    e = cudaMalloc(p, want);
    if (e != cudaSuccess) { e = cudaMalloc(p, bytes); want = bytes; }
    if (e != cudaSuccess) { *p = NULL; set_error(ctx, GORT_ERR_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e)); return NULL; }
    *cap = want;
    return *p;
}

void *scratch(gort_ctx *ctx, int slot, size_t bytes) { return grow(ctx, &ctx->scratch[slot], &ctx->scratch_cap[slot], bytes); }
void *workspace(gort_ctx *ctx, size_t bytes) { return grow(ctx, &ctx->work, &ctx->work_cap, bytes); }
void *rec_buffer(gort_ctx *ctx, int which, size_t bytes) { return grow(ctx, &ctx->rec_buf[which], &ctx->rec_cap[which], bytes); }

int order_after_previous(gort_ctx *ctx, cudaStream_t s)
{
    if (ctx->last_stream && ctx->last_stream != s) {
        cudaError_t e = cudaEventRecord(ctx->xstream_ev, ctx->last_stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(s, ctx->xstream_ev, 0);
        if (e != cudaSuccess) return check_cuda(ctx, e, "ordering calls across streams");
        ctx->last_was_wide = 0;
    }
    ctx->last_stream = s;
    return GORT_OK;
}

}  // namespace gort

using namespace gort;

#define TRY(x) do { int _r = (x); if (_r != GORT_OK) return _r; } while (0)
#define TRYCUDA(ctx, x, what) do { int _r = check_cuda(ctx, (x), what); if (_r != GORT_OK) return _r; } while (0)

extern "C" {

int gort_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int gort_create(int device, gort_ctx **out)
{
    if (!out) return set_error(NULL, GORT_ERR_INVALID, "gort_create: out is NULL");
    *out = NULL;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return set_error(NULL, GORT_ERR_CUDA, "gort_create: no CUDA device (%s); this library has no CPU path",
                         e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return set_error(NULL, GORT_ERR_INVALID, "gort_create: device %d out of range (0..%d)", device, n - 1);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return set_error(NULL, GORT_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
    gort_ctx *ctx = (gort_ctx *) calloc(1, sizeof(gort_ctx));
    if (!ctx) return set_error(NULL, GORT_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { set_error(NULL, GORT_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e)); free(ctx); return GORT_ERR_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { set_error(NULL, GORT_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); free(ctx); return GORT_ERR_CUDA; }
    int rc = GORT_OK;
    if (cudaMalloc((void **) &ctx->d_gauleg, sizeof(double) * 2 * GORT_NQUAD) != cudaSuccess ||
        cudaMalloc((void **) &ctx->d_prospect, sizeof(double) * 9 * GORT_PROSPECT_NW) != cudaSuccess ||
        cudaMalloc((void **) &ctx->d_soil, sizeof(double) * 4 * GORT_SOIL_NW) != cudaSuccess)
        rc = set_error(ctx, GORT_ERR_NOMEM, "cudaMalloc of constant tables failed");
    // BRDF pipeline flags: per-CTA epochs + the fault word, cleared here, before anything can poll them
    if (rc == GORT_OK && cudaMalloc((void **) &ctx->d_done, sizeof(unsigned long long) * (GORT_MAX_WIDE_CTAS + 1)) != cudaSuccess)
        rc = set_error(ctx, GORT_ERR_NOMEM, "cudaMalloc of the pipeline flags failed");
    if (rc == GORT_OK) rc = check_cuda(ctx, cudaMemsetAsync(ctx->d_done, 0, sizeof(unsigned long long) * (GORT_MAX_WIDE_CTAS + 1), ctx->stream), "pipeline flags");
    if (rc == GORT_OK) rc = check_cuda(ctx, cudaEventCreateWithFlags(&ctx->xstream_ev, cudaEventDisableTiming), "cudaEventCreate");
    ctx->dbg_timeline = getenv("GORT_TIMELINE") ? atoi(getenv("GORT_TIMELINE")) : 0;
    if (rc == GORT_OK) rc = launch_gauleg(ctx, ctx->stream, ctx->d_gauleg);
    if (rc == GORT_OK) rc = launch_tav_tables(ctx, ctx->stream, ctx->d_prospect);
    if (rc == GORT_OK) rc = upload_soil_tables(ctx, ctx->stream, ctx->d_soil);
    if (rc == GORT_OK) rc = check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "context initialisation");
    if (rc != GORT_OK) {
        strncpy(g_create_error, ctx->err, sizeof g_create_error - 1);
        gort_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return GORT_OK;
}

void gort_destroy(gort_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < GORT_NSCRATCH; i++) if (ctx->scratch[i]) cudaFree(ctx->scratch[i]);
    if (ctx->work) cudaFree(ctx->work);
    for (int i = 0; i < 2; i++) {
        if (ctx->rec_buf[i]) cudaFree(ctx->rec_buf[i]);
        if (ctx->d_flags[i]) cudaFree(ctx->d_flags[i]);
    }
    if (ctx->d_done) cudaFree(ctx->d_done);
    if (ctx->d_timeline) cudaFree(ctx->d_timeline);
    if (ctx->xstream_ev) cudaEventDestroy(ctx->xstream_ev);
    if (ctx->d_gauleg) cudaFree(ctx->d_gauleg);
    if (ctx->d_prospect) cudaFree(ctx->d_prospect);
    if (ctx->d_soil) cudaFree(ctx->d_soil);
    if (ctx->prof_ev) { for (int i = 0; i < 3 * ctx->prof_cap; i++) cudaEventDestroy(ctx->prof_ev[i]); free(ctx->prof_ev); }
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); for (int i = 0; i < 6; i++) if (ctx->fwd_ev[i]) cudaEventDestroy(ctx->fwd_ev[i]); cudaStreamDestroy(ctx->copy_stream); }
    if (ctx->copy_stream_out) { cudaStreamSynchronize(ctx->copy_stream_out); cudaStreamDestroy(ctx->copy_stream_out); }
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    free(ctx);
}

const char *gort_last_error(const gort_ctx *ctx) { return ctx ? ctx->err : g_create_error; }
void *gort_stream(gort_ctx *ctx) { return ctx ? (void *) ctx->stream : NULL; }
long gort_launch_count(const gort_ctx *ctx) { return ctx ? ctx->launches : 0; }

// the BRDF pipeline's in-kernel waits are bounded; one that expired (a broken predecessor) leaves a mark
static int check_pipeline_fault(gort_ctx *ctx)
{
    if (!ctx->d_done) return GORT_OK;
    unsigned long long f = 0;
    cudaError_t e = cudaMemcpy(&f, ctx->d_done + GORT_MAX_WIDE_CTAS, sizeof f, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return check_cuda(ctx, e, "pipeline fault word");
    if (f) {
        // reported once: clear the word so that later calls are judged on their own
        cudaMemset(ctx->d_done + GORT_MAX_WIDE_CTAS, 0, sizeof f);
        return set_error(ctx, GORT_ERR_CUDA, "BRDF pipeline: an in-kernel wait timed out in call %llu; the affected CTAs stored nothing for that call", f);
    }
    return GORT_OK;
}

int gort_synchronize(gort_ctx *ctx)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    // everything this context enqueued: each call waited for the one before it (order_after_previous), so the last
    // call's stream completes after all of them
    TRYCUDA(ctx, cudaStreamSynchronize(ctx->stream), "synchronize");
    if (ctx->last_stream && ctx->last_stream != ctx->stream) TRYCUDA(ctx, cudaStreamSynchronize(ctx->last_stream), "synchronize");
    ctx->last_stream = NULL;           // everything is complete: the caller may destroy its stream now
    ctx->last_was_wide = 0;
    return check_pipeline_fault(ctx);
}

int gort_set_overlap(gort_ctx *ctx, int enable)
{
    if (!ctx) return GORT_ERR_INVALID;
    ctx->overlap = enable ? 1 : 0;
    ctx->last_was_wide = 0;
    return GORT_OK;
}

void *gort_host_alloc(size_t bytes)
{
    void *p = NULL;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) return NULL;
    return p;
}

void gort_host_free(void *p) { if (p) cudaFreeHost(p); }

// ---- pinned buffers next to the GPU: probe which CPUs give the best device-to-host rate (see the header) ----
static void probe_host_placement(gort_ctx *ctx)
{
    ctx->near_probed = 1;
    ctx->near_ncpu = 0;
    snprintf(ctx->near_desc, sizeof ctx->near_desc, "not probed");
    cpu_set_t all;
    CPU_ZERO(&all);
    if (sched_getaffinity(0, sizeof all, &all) != 0) { snprintf(ctx->near_desc, sizeof ctx->near_desc, "sched_getaffinity failed"); return; }
    int cpus[1024], n = 0;
    for (int c = 0; c < CPU_SETSIZE && n < 1024; c++) if (CPU_ISSET(c, &all)) cpus[n++] = c;
    if (n < 4) { snprintf(ctx->near_desc, sizeof ctx->near_desc, "%d cpus: nothing to choose", n); return; }
    const size_t probe_bytes = (size_t) 32 << 20;
    if (order_after_previous(ctx, ctx->stream) != GORT_OK) { snprintf(ctx->near_desc, sizeof ctx->near_desc, "probe failed"); return; }
    void *d = workspace(ctx, probe_bytes);
    if (!d) return;
    const int n_groups = n >= 16 ? 8 : 4;
    cudaEvent_t e0, e1;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return;
    double best = 0.0, worst = 1e30;
    int best_g = -1;
    for (int gI = 0; gI < n_groups; gI++) {
        const int lo = (int) ((long) gI * n / n_groups), hi = (int) ((long) (gI + 1) * n / n_groups);
        cpu_set_t grp;
        CPU_ZERO(&grp);
        for (int k = lo; k < hi; k++) CPU_SET(cpus[k], &grp);
        if (sched_setaffinity(0, sizeof grp, &grp) != 0) continue;
        void *h = NULL;
        if (cudaMallocHost(&h, probe_bytes) != cudaSuccess) continue;
        memset(h, 0, probe_bytes);
        float ms_best = 1e30f;
        for (int rep = 0; rep < 4; rep++) {
            cudaEventRecord(e0, ctx->stream);
            cudaMemcpyAsync(h, d, probe_bytes, cudaMemcpyDeviceToHost, ctx->stream);
            cudaEventRecord(e1, ctx->stream);
            cudaEventSynchronize(e1);
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep && ms < ms_best) ms_best = ms;
        }
        cudaFreeHost(h);
        const double gbs = probe_bytes / (ms_best * 1e-3) / 1e9;
        if (gbs > best * 1.03) { best = gbs; best_g = gI; }       // ties go to the earlier group
        if (gbs < worst) worst = gbs;
    }
    sched_setaffinity(0, sizeof all, &all);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaGetLastError();
    if (best_g < 0) { snprintf(ctx->near_desc, sizeof ctx->near_desc, "probe failed"); return; }
    const int lo = (int) ((long) best_g * n / n_groups), hi = (int) ((long) (best_g + 1) * n / n_groups);
    for (int k = lo; k < hi; k++) ctx->near_cpu[ctx->near_ncpu++] = cpus[k];
    snprintf(ctx->near_desc, sizeof ctx->near_desc, "probed %d groups of %d cpus with 32 MB device-to-host copies: best %.1f GB/s from cpus %d-%d, worst %.1f GB/s",
             n_groups, n, best, cpus[lo], cpus[hi - 1], worst);
}

void *gort_host_alloc_on_cpus(size_t bytes, const int *cpus, int n_cpus)
{
    if (!cpus || n_cpus <= 0) return gort_host_alloc(bytes);
    cpu_set_t all, grp;
    CPU_ZERO(&all); CPU_ZERO(&grp);
    if (sched_getaffinity(0, sizeof all, &all) != 0) return gort_host_alloc(bytes);
    for (int k = 0; k < n_cpus; k++) if (cpus[k] >= 0 && cpus[k] < CPU_SETSIZE) CPU_SET(cpus[k], &grp);
    if (sched_setaffinity(0, sizeof grp, &grp) != 0) return gort_host_alloc(bytes);
    void *p = NULL;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) p = NULL;
    else memset(p, 0, bytes);                       // touch every page while still running on those CPUs
    sched_setaffinity(0, sizeof all, &all);
    return p;
}

void *gort_host_alloc_near(gort_ctx *ctx, size_t bytes)
{
    if (!ctx) return NULL;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return NULL;
    if (!ctx->near_probed) probe_host_placement(ctx);
    if (ctx->near_ncpu == 0) return gort_host_alloc(bytes);
    return gort_host_alloc_on_cpus(bytes, ctx->near_cpu, ctx->near_ncpu);
}

int gort_host_placement(gort_ctx *ctx, char *buf, size_t len)
{
    if (!ctx || !buf || len == 0) return GORT_ERR_INVALID;
    snprintf(buf, len, "%s", ctx->near_probed ? ctx->near_desc : "not probed yet");
    return GORT_OK;
}

static cudaStream_t pick(gort_ctx *ctx, void *stream) { return stream ? (cudaStream_t) stream : ctx->stream; }

static int h2d(gort_ctx *ctx, int slot, const double *h, size_t n, double **d)
{
    *d = NULL;
    if (!h || n == 0) return GORT_OK;
    double *p = (double *) scratch(ctx, slot, n * sizeof(double));
    if (!p) return GORT_ERR_NOMEM;
    TRYCUDA(ctx, cudaMemcpyAsync(p, h, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream), "host to device copy");
    *d = p;
    return GORT_OK;
}

static int dout(gort_ctx *ctx, int slot, const double *h, size_t n, double **d)
{
    *d = NULL;
    if (!h || n == 0) return GORT_OK;
    double *p = (double *) scratch(ctx, slot, n * sizeof(double));
    if (!p) return GORT_ERR_NOMEM;
    *d = p;
    return GORT_OK;
}

static int d2h(gort_ctx *ctx, double *h, const double *d, size_t n)
{
    if (!h || !d || n == 0) return GORT_OK;
    TRYCUDA(ctx, cudaMemcpyAsync(h, d, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream), "device to host copy");
    return GORT_OK;
}

// ---- gap probabilities --------------------------------------------------------------------------
int gort_lut_batch_dev(gort_ctx *ctx, void *stream, int n_sets, const double *structure, int method, double *lut)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!structure || !lut || n_sets <= 0) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_batch: bad arguments");
    if (method != GORT_LUT_FULL && method != GORT_LUT_Q08) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_batch: unknown method %d", method);
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_lut(ctx, s, n_sets, structure, method, lut);
}

int gort_lut_batch_scatter_dev(gort_ctx *ctx, void *stream, int n_sets, const double *structure, int method,
                               double *lut, int n_dst, double *const *dst, int multicast)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!structure || !lut || n_sets <= 0 || n_dst < 0 || n_dst > GORT_LUT_MAX_DST || (n_dst > 0 && !dst))
        return set_error(ctx, GORT_ERR_INVALID, "gort_lut_batch_scatter: bad arguments");
    for (int q = 0; q < n_dst; q++)
        if (!dst[q] || ((uintptr_t) dst[q] & 7)) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_batch_scatter: destination %d is null or misaligned", q);
    if (method != GORT_LUT_FULL && method != GORT_LUT_Q08) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_batch: unknown method %d", method);
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_lut_out(ctx, s, n_sets, structure, method, lut, n_dst, dst, multicast != 0);
}

int gort_lut_batch(gort_ctx *ctx, int n_sets, const double *structure, int method, double *lut)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!structure || !lut || n_sets <= 0) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_batch: bad arguments");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    double *d_st, *d_lut;
    TRY(h2d(ctx, 0, structure, (size_t) 6 * n_sets, &d_st));
    TRY(dout(ctx, 1, lut, (size_t) n_sets * GORT_LUT_STRIDE, &d_lut));
    TRY(gort_lut_batch_dev(ctx, NULL, n_sets, d_st, method, d_lut));
    TRY(d2h(ctx, lut, d_lut, (size_t) n_sets * GORT_LUT_STRIDE));
    return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_lut_batch");
}

int gort_lut_intermediates_batch_dev(gort_ctx *ctx, void *stream, int n_sets, const double *structure, double *vb,
                                     double *fb, double *t_open, double *dt_open, double *dk_open, double *k_open)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!structure || n_sets <= 0) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_intermediates_batch: bad arguments");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_lut_dead(ctx, s, n_sets, structure, vb, fb, t_open, dt_open, dk_open, k_open);
}

int gort_lut_intermediates_batch(gort_ctx *ctx, int n_sets, const double *structure, double *vb, double *fb,
                                 double *t_open, double *dt_open, double *dk_open, double *k_open)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!structure || n_sets <= 0) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_intermediates_batch: bad arguments");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    const size_t M = n_sets;
    double *d_st, *d[6];
    double *h[6] = {vb, fb, t_open, dt_open, dk_open, k_open};
    const size_t sz[6] = {M * 15, M * 15 * GORT_NTH, M * 225, M * 225, M * 15, M * 15};
    TRY(h2d(ctx, 0, structure, 6 * M, &d_st));
    for (int k = 0; k < 6; k++) TRY(dout(ctx, 1 + k, h[k], sz[k], &d[k]));
    TRY(gort_lut_intermediates_batch_dev(ctx, NULL, n_sets, d_st, d[0], d[1], d[2], d[3], d[4], d[5]));
    for (int k = 0; k < 6; k++) TRY(d2h(ctx, h[k], d[k], sz[k]));
    return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_lut_intermediates_batch");
}

// ---- spectra ------------------------------------------------------------------------------------
int gort_spectra_batch_dev(gort_ctx *ctx, void *stream, int n_sets, const double *leaf, const double *soil,
                           double user_leaf, double user_soil, int n_wl, const double *wavelength,
                           double *rleaf, double *tleaf, double *rsoil)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!wavelength || !rleaf || !tleaf || !rsoil) return set_error(ctx, GORT_ERR_INVALID, "gort_spectra_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_spectra(ctx, s, n_sets, leaf, soil, user_leaf, user_soil, n_wl, wavelength, rleaf, tleaf, rsoil);
}

int gort_spectra_batch(gort_ctx *ctx, int n_sets, const double *leaf, const double *soil,
                       double user_leaf, double user_soil, int n_wl, const double *wavelength,
                       double *rleaf, double *tleaf, double *rsoil)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!wavelength || !rleaf || !tleaf || !rsoil || n_sets <= 0 || n_wl <= 0)
        return set_error(ctx, GORT_ERR_INVALID, "gort_spectra_batch: bad arguments");
    for (int i = 0; i < n_wl; i++)
        if (wavelength[i] < GORT_WL_MIN || wavelength[i] > GORT_WL_MAX)
            return set_error(ctx, GORT_ERR_RANGE, "wavlength out of range (400-2500)");   /* sic, gortt.c:1300 */
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    double *d_leaf, *d_soil, *d_wl, *d_rl, *d_tl, *d_rs;
    size_t n = (size_t) n_sets * n_wl;
    TRY(h2d(ctx, 0, user_leaf < 0.0 ? leaf : NULL, (size_t) 7 * n_sets, &d_leaf));
    TRY(h2d(ctx, 1, user_soil < 0.0 ? soil : NULL, (size_t) 4 * n_sets, &d_soil));
    TRY(h2d(ctx, 2, wavelength, n_wl, &d_wl));
    TRY(dout(ctx, 3, rleaf, n, &d_rl));
    TRY(dout(ctx, 4, tleaf, n, &d_tl));
    TRY(dout(ctx, 5, rsoil, n, &d_rs));
    TRY(gort_spectra_batch_dev(ctx, NULL, n_sets, d_leaf, d_soil, user_leaf, user_soil, n_wl, d_wl, d_rl, d_tl, d_rs));
    TRY(d2h(ctx, rleaf, d_rl, n));
    TRY(d2h(ctx, tleaf, d_tl, n));
    TRY(d2h(ctx, rsoil, d_rs, n));
    return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_spectra_batch");
}

int gort_prospect_batch(gort_ctx *ctx, int n_sets, const double *leaf, double *refl, double *tran)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!leaf || !refl || !tran || n_sets <= 0) return set_error(ctx, GORT_ERR_INVALID, "gort_prospect_batch: bad arguments");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    double *d_leaf, *d_r, *d_t;
    size_t n = (size_t) n_sets * GORT_PROSPECT_NW;
    TRY(h2d(ctx, 0, leaf, (size_t) 7 * n_sets, &d_leaf));
    TRY(dout(ctx, 1, refl, n, &d_r));
    TRY(dout(ctx, 2, tran, n, &d_t));
    TRY(launch_prospect_full(ctx, ctx->stream, n_sets, d_leaf, d_r, d_t));
    TRY(d2h(ctx, refl, d_r, n));
    TRY(d2h(ctx, tran, d_t, n));
    return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_prospect_batch");
}

// ---- soil spectrum file (finishes gortt_read_soil_lut, gortt.c:1388-1451) --------------------------------
int gort_soil_table_read(const char *path, double *table, char *errbuf, size_t errlen)
{
    if (errbuf && errlen) errbuf[0] = '\0';
    if (!path || !table) return GORT_ERR_INVALID;
#define SOIL_FAIL(...) do { if (errbuf && errlen) snprintf(errbuf, errlen, __VA_ARGS__); if (fp) fclose(fp); free(line); return GORT_ERR_IO; } while (0)
    char *line = NULL; size_t cap = 0;
    FILE *fp = fopen(path, "r");
    if (!fp) SOIL_FAIL("cannot open file: %s", path);                                            /* :1399-1402 */
    for (int i = 0; i < GORT_SOIL_TABLE_NW; i++) table[i] = 0.0;
    int n = 0;
    double this_wl = 0, this_rs = 0, last_wl = 0, last_rs = 0;
    while (getline(&line, &cap, fp) >= 0) {                                                      /* :1404 (no line-length limit here) */
        n++;
        if (sscanf(line, "%lf %lf", &this_wl, &this_rs) != 2)
            SOIL_FAIL("error in soil file (%s), line %d", path, n + 1);                          /* :1407-1410, "n+1" sic */
        if (n == 1 && this_wl > 400)
            SOIL_FAIL("error in soil file (%s), first wavelength (%lf) should be <=400", path, this_wl);   /* :1412-1416 */
        if (n > 1) {
            for (int i = (int) ceil(last_wl); i <= floor(this_wl); i++) {                        /* :1420-1428 */
                int index = i - 400;
                if ((index >= 0) && (index <= 2100))
                    table[index] = last_rs + (i - last_wl) / (this_wl - last_wl) * (this_rs - last_rs);
            }
        }
        last_wl = this_wl;
        last_rs = this_rs;
    }
    if (last_wl < 2500)
        SOIL_FAIL("error in soil file (%s), last wavelength (%lf) should be >=2500", path, last_wl);       /* :1435-1438 */
#undef SOIL_FAIL
    fclose(fp);
    free(line);
    return GORT_OK;
}

int gort_soil_from_table_dev(gort_ctx *ctx, void *stream, const double *table, int n_sets, int n_wl,
                             const double *wavelength, double *rsoil)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!table || !wavelength || !rsoil || n_sets <= 0 || n_wl <= 0)
        return set_error(ctx, GORT_ERR_INVALID, "gort_soil_from_table: bad arguments");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_soil_table(ctx, s, table, n_sets, n_wl, wavelength, rsoil);
}

int gort_soil_from_table(gort_ctx *ctx, const double *table, int n_sets, int n_wl, const double *wavelength, double *rsoil)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!table || !wavelength || !rsoil || n_sets <= 0 || n_wl <= 0)
        return set_error(ctx, GORT_ERR_INVALID, "gort_soil_from_table: bad arguments");
    for (int i = 0; i < n_wl; i++)
        if (wavelength[i] < GORT_WL_MIN || wavelength[i] > GORT_WL_MAX)
            return set_error(ctx, GORT_ERR_RANGE, "wavlength out of range (400-2500)");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    double *d_tab, *d_wl, *d_rs;
    TRY(h2d(ctx, 0, table, GORT_SOIL_TABLE_NW, &d_tab));
    TRY(h2d(ctx, 1, wavelength, n_wl, &d_wl));
    TRY(dout(ctx, 2, rsoil, (size_t) n_sets * n_wl, &d_rs));
    TRY(gort_soil_from_table_dev(ctx, NULL, d_tab, n_sets, n_wl, d_wl, d_rs));
    TRY(d2h(ctx, rsoil, d_rs, (size_t) n_sets * n_wl));
    return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_soil_from_table");
}

// ---- BRDF / energy --------------------------------------------------------------------------------
static int check_shape(gort_ctx *ctx, const gort_shape *sh, const char *who)
{
    if (!sh) return set_error(ctx, GORT_ERR_INVALID, "%s: shape is NULL", who);
    if (sh->n_sets <= 0 || sh->n_geom <= 0 || sh->n_wl <= 0)
        return set_error(ctx, GORT_ERR_INVALID, "%s: n_sets, n_geom and n_wl must be positive", who);
    if ((long) sh->n_sets * sh->n_geom > 2000000000L)
        return set_error(ctx, GORT_ERR_INVALID, "%s: n_sets*n_geom too large", who);
    return GORT_OK;
}

int gort_brdf_batch_dev(gort_ctx *ctx, void *stream, const gort_shape *shape, const double *structure,
                        const double *lut, const double *angles, const double *rleaf, const double *tleaf,
                        const double *rsoil, double *rsurf, double *scomp, double *kprop)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_shape(ctx, shape, "gort_brdf_batch"));
    if (!structure || !lut || !angles || !rleaf || !tleaf || !rsoil || !rsurf)
        return set_error(ctx, GORT_ERR_INVALID, "gort_brdf_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_brdf(ctx, s, *shape, structure, lut, angles, rleaf, tleaf, rsoil, rsurf, scomp, kprop);
}

static int copy_rows(gort_ctx *ctx, cudaStream_t s, double *dst, size_t dst_pitch, const double *src, size_t src_pitch,
                     size_t width, int rows, cudaMemcpyKind kind, const char *what);

struct Staged { double *st, *lut, *ang, *rl, *tl, *rs; };

static int stage_inputs(gort_ctx *ctx, const gort_shape *sh, const double *structure, const double *lut,
                        const double *angles, const double *rleaf, const double *tleaf, const double *rsoil, Staged *d)
{
    size_t M = sh->n_sets, G = sh->n_geom, W = sh->n_wl;
    size_t na = sh->geom_per_set ? M * G : G;
    size_t ns = sh->spectra_per_set ? M * W : W;
    TRY(h2d(ctx, 0, structure, 6 * M, &d->st));
    TRY(h2d(ctx, 1, lut, M * GORT_LUT_STRIDE, &d->lut));
    TRY(h2d(ctx, 2, angles, 4 * na, &d->ang));
    TRY(h2d(ctx, 3, rleaf, ns, &d->rl));
    TRY(h2d(ctx, 4, tleaf, ns, &d->tl));
    TRY(h2d(ctx, 5, rsoil, ns, &d->rs));
    return GORT_OK;
}

int gort_brdf_batch(gort_ctx *ctx, const gort_shape *shape, const double *structure, const double *lut,
                    const double *angles, const double *rleaf, const double *tleaf, const double *rsoil,
                    double *rsurf, double *scomp, double *kprop)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_shape(ctx, shape, "gort_brdf_batch"));
    if (!structure || !lut || !angles || !rleaf || !tleaf || !rsoil || !rsurf)
        return set_error(ctx, GORT_ERR_INVALID, "gort_brdf_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    Staged d;
    TRY(stage_inputs(ctx, shape, structure, lut, angles, rleaf, tleaf, rsoil, &d));
    size_t nl = (size_t) shape->n_sets * shape->n_geom;
    // the device buffer uses the caller's row pitch: a dense host array comes back in ONE contiguous copy, a pitched
    // one row by row (2-D copy) so that its padding columns stay untouched
    const size_t W = shape->n_wl;
    const size_t hp = shape->out_pitch > 0 ? (size_t) shape->out_pitch : W;
    if (hp < W) return set_error(ctx, GORT_ERR_INVALID, "gort_brdf_batch: out_pitch smaller than n_wl");
    double *d_rsurf, *d_scomp, *d_kprop;
    TRY(dout(ctx, 6, rsurf, nl * hp, &d_rsurf));
    TRY(dout(ctx, 7, scomp, 4 * nl * hp, &d_scomp));
    TRY(dout(ctx, 8, kprop, 4 * nl, &d_kprop));
    TRY(launch_brdf(ctx, ctx->stream, *shape, d.st, d.lut, d.ang, d.rl, d.tl, d.rs, d_rsurf, d_scomp, d_kprop));
    if (hp == W) {
        TRY(d2h(ctx, rsurf, d_rsurf, nl * hp));
        TRY(d2h(ctx, scomp, d_scomp, 4 * nl * hp));
    } else {
        // pitched host rows: only the n_wl columns of every row are copied back -- the padding columns of the caller's
        // array are never touched, as the header promises (the device buffer's padding holds kernel scratch)
        TRY(copy_rows(ctx, ctx->stream, rsurf, hp, d_rsurf, hp, W, (int) nl, cudaMemcpyDeviceToHost, "device to host copy"));
        if (scomp) TRY(copy_rows(ctx, ctx->stream, scomp, 4 * hp, d_scomp, 4 * hp, 4 * W, (int) nl, cudaMemcpyDeviceToHost, "device to host copy"));
    }
    TRY(d2h(ctx, kprop, d_kprop, 4 * nl));
    TRY(check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_brdf_batch"));
    return check_pipeline_fault(ctx);
}

// ---- ensemble forward operator: LUT -> spectra -> BRDF, chunked, copies under kernels -------------------
static int copy_rows(gort_ctx *ctx, cudaStream_t s, double *dst, size_t dst_pitch, const double *src, size_t src_pitch,
                     size_t width, int rows, cudaMemcpyKind kind, const char *what)
{
    // `rows` rows of `width` doubles; pitches in doubles
    return check_cuda(ctx, cudaMemcpy2DAsync(dst, dst_pitch * sizeof(double), src, src_pitch * sizeof(double),
                                             width * sizeof(double), (size_t) rows, kind, s), what);
}

}  // extern "C"

// The chunked ensemble pipeline of gort_forward_batch, gort_forward_band_batch and gort_lai_tangent_batch: members in
// chunks on three streams -- the inputs of chunk i+1 go up (stream B) and the results of chunk i-1 come down (stream D)
// while chunk i's kernels run (stream A); two chunk buffers alternate.  kernels(A, c, bufs) enqueues one chunk's kernels
// on A.  out_pm[k] sizes the chunk buffer out[k] (doubles per member; 0: none).  After the kernels every copy with a
// host pointer takes its per_member doubles per member from out[src] (src < 0: the LUT records) to the host.  The caller
// has uploaded the grid's wavelengths and shared angles (slots 22 and up); the chunk buffers use scratch slots 0-21.
struct EnsBufs { double *st, *leaf, *soil, *ang, *lut, *rl, *tl, *rs, *out[3]; };
struct EnsCopy { double *host; int src; size_t per_member; };

template <class Kernels>
static int ensemble_chunks(gort_ctx *ctx, const gort_shape *shape, const double *structure, const double *leaf,
                           const double *soil, double user_leaf, double user_soil, const double *angles, size_t n_col,
                           const size_t out_pm[3], int n_copies, const EnsCopy *copies, const char *who, Kernels kernels)
{
    if (!ctx->copy_stream) {
        TRYCUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking), "cudaStreamCreate");
        TRYCUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream_out, cudaStreamNonBlocking), "cudaStreamCreate");
        for (int i = 0; i < 6; i++) TRYCUDA(ctx, cudaEventCreateWithFlags(&ctx->fwd_ev[i], cudaEventDisableTiming), "cudaEventCreate");
    }
    // three streams: the two copy directions have their own engines, and on ONE copy stream the inputs of chunk i+1 would
    // queue behind the results of chunk i, which wait for chunk i's kernels -- no copy would run under a kernel
    cudaStream_t A = ctx->stream, B = ctx->copy_stream, D = ctx->copy_stream_out;
    const size_t M = shape->n_sets, G = shape->n_geom;
    // chunk: at least 8 per batch when the batch is large, never above 16384 members, at least 1024
    size_t C = (M + 7) / 8;
    if (C > 16384) C = 16384;
    if (C < 1024) C = 1024;
    if (C > M) C = M;
    const bool per_set_geom = shape->geom_per_set != 0;
    EnsBufs buf[2];
    const size_t sz[11] = {6 * C, 7 * C, 4 * C, per_set_geom ? 4 * C * G : 8, C * GORT_LUT_STRIDE, C * n_col, C * n_col,
                           C * n_col, C * out_pm[0], C * out_pm[1], C * out_pm[2]};
    for (int b = 0; b < 2; b++) {
        double **p[11] = {&buf[b].st, &buf[b].leaf, &buf[b].soil, &buf[b].ang, &buf[b].lut, &buf[b].rl, &buf[b].tl,
                          &buf[b].rs, &buf[b].out[0], &buf[b].out[1], &buf[b].out[2]};
        for (int k = 0; k < 11; k++) {
            *p[k] = NULL;
            if (sz[k] == 0) continue;
            *p[k] = (double *) scratch(ctx, 11 * b + k, sz[k] * sizeof(double));
            if (!*p[k]) return GORT_ERR_NOMEM;
        }
    }
    // the kernels wait for the previous call; the input copies on B need not: they only fill this call's scratch slots,
    // which no other call reads while this one runs (every host-pointer call returns synchronised)
    TRY(order_after_previous(ctx, A));
    // events per buffer: [b] inputs ready (B), [2+b] kernels done (A), [4+b] outputs copied (D)
    int chunk_no = 0;
    for (size_t m0 = 0; m0 < M; m0 += C, chunk_no++) {
        const size_t c = M - m0 < C ? M - m0 : C;
        const int b = chunk_no & 1;
        const EnsBufs &d = buf[b];
        // -- stream B: inputs of this chunk (after the kernels that last read this buffer's inputs) --
        if (chunk_no >= 2) TRYCUDA(ctx, cudaStreamWaitEvent(B, ctx->fwd_ev[2 + b], 0), "cudaStreamWaitEvent");
        TRY(copy_rows(ctx, B, d.st, c, structure + m0, M, c, 6, cudaMemcpyHostToDevice, "forward: structure"));
        if (user_leaf < 0.0) TRY(copy_rows(ctx, B, d.leaf, c, leaf + m0, M, c, 7, cudaMemcpyHostToDevice, "forward: leaf"));
        if (user_soil < 0.0) TRY(copy_rows(ctx, B, d.soil, c, soil + m0, M, c, 4, cudaMemcpyHostToDevice, "forward: soil"));
        if (per_set_geom) TRY(copy_rows(ctx, B, d.ang, c * G, angles + m0 * G, M * G, c * G, 4, cudaMemcpyHostToDevice, "forward: angles"));
        TRYCUDA(ctx, cudaEventRecord(ctx->fwd_ev[b], B), "cudaEventRecord");
        // -- stream A: kernels (after the inputs are in, and after the previous outputs of this buffer have left) --
        TRYCUDA(ctx, cudaStreamWaitEvent(A, ctx->fwd_ev[b], 0), "cudaStreamWaitEvent");
        if (chunk_no >= 2) TRYCUDA(ctx, cudaStreamWaitEvent(A, ctx->fwd_ev[4 + b], 0), "cudaStreamWaitEvent");
        TRY(kernels(A, c, d));
        TRYCUDA(ctx, cudaEventRecord(ctx->fwd_ev[2 + b], A), "cudaEventRecord");
        // -- stream D: results of this chunk --
        TRYCUDA(ctx, cudaStreamWaitEvent(D, ctx->fwd_ev[2 + b], 0), "cudaStreamWaitEvent");
        for (int k = 0; k < n_copies; k++) {
            const EnsCopy &q = copies[k];
            if (!q.host) continue;
            TRYCUDA(ctx, cudaMemcpyAsync(q.host + m0 * q.per_member, q.src < 0 ? d.lut : d.out[q.src],
                                         c * q.per_member * sizeof(double), cudaMemcpyDeviceToHost, D), "forward: results");
        }
        TRYCUDA(ctx, cudaEventRecord(ctx->fwd_ev[4 + b], D), "cudaEventRecord");
    }
    TRYCUDA(ctx, cudaStreamSynchronize(D), who);
    TRYCUDA(ctx, cudaStreamSynchronize(B), who);
    TRYCUDA(ctx, cudaStreamSynchronize(A), who);
    note_other_work(ctx);
    return check_pipeline_fault(ctx);
}

extern "C" {

int gort_forward_batch(gort_ctx *ctx, const gort_shape *shape, int lut_method, const double *structure,
                       const double *leaf, const double *soil, double user_leaf, double user_soil,
                       const double *wavelength, const double *angles, double *rsurf, double *lut_out)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_shape(ctx, shape, "gort_forward_batch"));
    if (!structure || !wavelength || !angles || !rsurf || (user_leaf < 0.0 && !leaf) || (user_soil < 0.0 && !soil))
        return set_error(ctx, GORT_ERR_INVALID, "gort_forward_batch: NULL argument");
    if (lut_method != GORT_LUT_FULL && lut_method != GORT_LUT_Q08)
        return set_error(ctx, GORT_ERR_INVALID, "gort_forward_batch: unknown LUT method %d", lut_method);
    const size_t G = shape->n_geom, W = shape->n_wl;
    for (size_t i = 0; i < W; i++)
        if (wavelength[i] < GORT_WL_MIN || wavelength[i] > GORT_WL_MAX)
            return set_error(ctx, GORT_ERR_RANGE, "wavlength out of range (400-2500)");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    // slot 22 the wavelengths, 23 shared angles
    double *d_wl, *d_ang_shared = NULL;
    TRY(h2d(ctx, 22, wavelength, W, &d_wl));
    if (!shape->geom_per_set) TRY(h2d(ctx, 23, angles, 4 * G, &d_ang_shared));
    gort_shape sh = *shape;
    sh.spectra_per_set = 1;
    sh.out_pitch = 0;
    const size_t out_pm[3] = {G * W, 0, 0};
    const EnsCopy copies[2] = {{rsurf, 0, G * W}, {lut_out, -1, GORT_LUT_STRIDE}};
    return ensemble_chunks(ctx, shape, structure, leaf, soil, user_leaf, user_soil, angles, W, out_pm, 2, copies, "gort_forward_batch",
                           [&](cudaStream_t A, size_t c, const EnsBufs &d) {
        sh.n_sets = (int) c;
        TRY(launch_lut(ctx, A, (int) c, d.st, lut_method, d.lut));
        TRY(launch_spectra(ctx, A, (int) c, user_leaf < 0.0 ? d.leaf : NULL, user_soil < 0.0 ? d.soil : NULL, user_leaf, user_soil,
                           (int) W, d_wl, d.rl, d.tl, d.rs));
        return launch_brdf(ctx, A, sh, d.st, d.lut, sh.geom_per_set ? d.ang : d_ang_shared, d.rl, d.tl, d.rs, d.out[0], NULL, NULL);
    });
}

// ---- finite-difference Jacobian through the whole chain (SURVEY.md 8f row 4) -----------------------------
int gort_jacobian_batch(gort_ctx *ctx, const gort_shape *shape, int lut_method, int param, double rel_step,
                        const double *structure, const double *leaf, const double *soil, double user_leaf,
                        double user_soil, const double *wavelength, const double *angles, double *jac, double *rsurf)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_shape(ctx, shape, "gort_jacobian_batch"));
    if (!structure || !wavelength || !angles || !jac || (user_leaf < 0.0 && !leaf) || (user_soil < 0.0 && !soil))
        return set_error(ctx, GORT_ERR_INVALID, "gort_jacobian_batch: NULL argument");
    if (param < GORT_JAC_LAMBDA || param > GORT_JAC_LAI) return set_error(ctx, GORT_ERR_INVALID, "gort_jacobian_batch: unknown parameter %d", param);
    if (lut_method != GORT_LUT_FULL && lut_method != GORT_LUT_Q08)
        return set_error(ctx, GORT_ERR_INVALID, "gort_jacobian_batch: unknown LUT method %d", lut_method);
    const size_t M = shape->n_sets, G = shape->n_geom, W = shape->n_wl;
    for (size_t i = 0; i < W; i++)
        if (wavelength[i] < GORT_WL_MIN || wavelength[i] > GORT_WL_MAX)
            return set_error(ctx, GORT_ERR_RANGE, "wavlength out of range (400-2500)");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const double h = rel_step > 0.0 ? rel_step : 1e-4;
    const int row = param == GORT_JAC_LAI ? 5 : param;
    cudaStream_t A = ctx->stream;
    TRY(order_after_previous(ctx, A));
    // members in chunks that keep the three result buffers below ~768 MB
    size_t C = ((size_t) 256 << 20) / (G * W * sizeof(double));
    if (C < 1) C = 1;
    if (C > M) C = M;
    const bool per_set_geom = shape->geom_per_set != 0;
    double *d_wl, *d_ang_shared = NULL;
    TRY(h2d(ctx, 18, wavelength, W, &d_wl));
    if (!per_set_geom) TRY(h2d(ctx, 19, angles, 4 * G, &d_ang_shared));
    // slots: 0 structure, 1 leaf, 2 soil, 3 angles, 4 perturbed structure, 5 lut, 6-8 spectra, 9 f+, 10 f-, 11 f0 / jac
    const size_t sz[12] = {6 * C, 7 * C, 4 * C, per_set_geom ? 4 * C * G : 8, 6 * C, C * GORT_LUT_STRIDE, C * W, C * W, C * W,
                           C * G * W, C * G * W, C * G * W};
    double *d[12];
    for (int k = 0; k < 12; k++) {
        d[k] = (double *) scratch(ctx, k, sz[k] * sizeof(double));
        if (!d[k]) return GORT_ERR_NOMEM;
    }
    gort_shape sh = *shape;
    sh.spectra_per_set = 1;
    sh.out_pitch = 0;
    for (size_t m0 = 0; m0 < M; m0 += C) {
        const size_t c = M - m0 < C ? M - m0 : C;
        sh.n_sets = (int) c;
        TRY(copy_rows(ctx, A, d[0], c, structure + m0, M, c, 6, cudaMemcpyHostToDevice, "jacobian: structure"));
        if (user_leaf < 0.0) TRY(copy_rows(ctx, A, d[1], c, leaf + m0, M, c, 7, cudaMemcpyHostToDevice, "jacobian: leaf"));
        if (user_soil < 0.0) TRY(copy_rows(ctx, A, d[2], c, soil + m0, M, c, 4, cudaMemcpyHostToDevice, "jacobian: soil"));
        if (per_set_geom) TRY(copy_rows(ctx, A, d[3], c * G, angles + m0 * G, M * G, c * G, 4, cudaMemcpyHostToDevice, "jacobian: angles"));
        const double *d_ang = per_set_geom ? d[3] : d_ang_shared;
        TRY(launch_spectra(ctx, A, (int) c, user_leaf < 0.0 ? d[1] : NULL, user_soil < 0.0 ? d[2] : NULL, user_leaf, user_soil,
                           (int) W, d_wl, d[6], d[7], d[8]));
        for (int side = 0; side < 2; side++) {
            TRY(launch_jac_perturb(ctx, A, (int) c, row, side == 0 ? 1.0 + h : 1.0 - h, d[0], d[4]));
            TRY(launch_lut(ctx, A, (int) c, d[4], lut_method, d[5]));
            TRY(launch_brdf(ctx, A, sh, d[4], d[5], d_ang, d[6], d[7], d[8], d[9 + side], NULL, NULL));
        }
        if (rsurf) {
            TRY(launch_lut(ctx, A, (int) c, d[0], lut_method, d[5]));
            TRY(launch_brdf(ctx, A, sh, d[0], d[5], d_ang, d[6], d[7], d[8], d[11], NULL, NULL));
            TRYCUDA(ctx, cudaMemcpyAsync(rsurf + m0 * G * W, d[11], c * G * W * sizeof(double), cudaMemcpyDeviceToHost, A), "jacobian: rsurf");
        }
        TRY(launch_jac_diff(ctx, A, (int) c, (long) (G * W), row, param == GORT_JAC_LAI, h, d[0], d[9], d[10], d[11]));
        TRYCUDA(ctx, cudaMemcpyAsync(jac + m0 * G * W, d[11], c * G * W * sizeof(double), cudaMemcpyDeviceToHost, A), "jacobian: result");
    }
    TRYCUDA(ctx, cudaStreamSynchronize(A), "gort_jacobian_batch");
    return check_pipeline_fault(ctx);
}

// ---- exact favd / LAI tangent (forward mode) -----------------------------------------------------------------------
int gort_lut_tangent_batch_dev(gort_ctx *ctx, void *stream, int n_sets, const double *structure, int method, double *lut,
                               double *dlut)
{
    if (!ctx) return GORT_ERR_INVALID;
    if (!structure || !lut || !dlut || n_sets <= 0) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_tangent_batch: bad arguments");
    if (method != GORT_LUT_FULL && method != GORT_LUT_Q08) return set_error(ctx, GORT_ERR_INVALID, "gort_lut_tangent_batch: unknown method %d", method);
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_lut_tangent(ctx, s, n_sets, structure, method, lut, dlut);
}

int gort_brdf_tangent_batch_dev(gort_ctx *ctx, void *stream, const gort_shape *shape, const double *structure,
                                const double *lut, const double *dlut, const double *angles, const double *rleaf,
                                const double *tleaf, const double *rsoil, double *drsurf)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_shape(ctx, shape, "gort_brdf_tangent_batch"));
    if (!structure || !lut || !dlut || !angles || !rleaf || !tleaf || !rsoil || !drsurf)
        return set_error(ctx, GORT_ERR_INVALID, "gort_brdf_tangent_batch: NULL argument");
    if (shape->out_pitch != 0) return set_error(ctx, GORT_ERR_INVALID, "gort_brdf_tangent_batch: drsurf is dense (out_pitch must be 0)");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_brdf_tangent(ctx, s, *shape, structure, lut, dlut, angles, rleaf, tleaf, rsoil, drsurf, 0);
}

int gort_lai_tangent_batch(gort_ctx *ctx, const gort_shape *shape, int lut_method, int param, const double *structure,
                           const double *leaf, const double *soil, double user_leaf, double user_soil,
                           const double *wavelength, const double *angles, double *jac, double *rsurf)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_shape(ctx, shape, "gort_lai_tangent_batch"));
    if (!structure || !wavelength || !angles || !jac || (user_leaf < 0.0 && !leaf) || (user_soil < 0.0 && !soil))
        return set_error(ctx, GORT_ERR_INVALID, "gort_lai_tangent_batch: NULL argument");
    if (param != GORT_JAC_FAVD && param != GORT_JAC_LAI)
        return set_error(ctx, GORT_ERR_INVALID, "gort_lai_tangent_batch: parameter %d is not GORT_JAC_FAVD or GORT_JAC_LAI", param);
    if (lut_method != GORT_LUT_FULL && lut_method != GORT_LUT_Q08)
        return set_error(ctx, GORT_ERR_INVALID, "gort_lai_tangent_batch: unknown LUT method %d", lut_method);
    const size_t G = shape->n_geom, W = shape->n_wl;
    for (size_t i = 0; i < W; i++)
        if (wavelength[i] < GORT_WL_MIN || wavelength[i] > GORT_WL_MAX)
            return set_error(ctx, GORT_ERR_RANGE, "wavlength out of range (400-2500)");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    double *d_wl, *d_ang_shared = NULL;
    TRY(h2d(ctx, 22, wavelength, W, &d_wl));
    if (!shape->geom_per_set) TRY(h2d(ctx, 23, angles, 4 * G, &d_ang_shared));
    gort_shape sh = *shape;
    sh.spectra_per_set = 1;
    sh.out_pitch = 0;
    // chunk buffers: out[0] jac, out[1] rsurf, out[2] the LUT tangent
    const size_t out_pm[3] = {G * W, rsurf ? G * W : 0, GORT_LUT_STRIDE};
    const EnsCopy copies[2] = {{jac, 0, G * W}, {rsurf, 1, G * W}};
    return ensemble_chunks(ctx, shape, structure, leaf, soil, user_leaf, user_soil, angles, W, out_pm, 2, copies, "gort_lai_tangent_batch",
                           [&](cudaStream_t A, size_t c, const EnsBufs &d) {
        sh.n_sets = (int) c;
        const double *ang = sh.geom_per_set ? d.ang : d_ang_shared;
        TRY(launch_lut_tangent(ctx, A, (int) c, d.st, lut_method, d.lut, d.out[2]));
        TRY(launch_spectra(ctx, A, (int) c, user_leaf < 0.0 ? d.leaf : NULL, user_soil < 0.0 ? d.soil : NULL, user_leaf, user_soil,
                           (int) W, d_wl, d.rl, d.tl, d.rs));
        // rsurf from the existing BRDF kernels on this LUT: the bits of gort_forward_batch
        if (rsurf) TRY(launch_brdf(ctx, A, sh, d.st, d.lut, ang, d.rl, d.tl, d.rs, d.out[1], NULL, NULL));
        return launch_brdf_tangent(ctx, A, sh, d.st, d.lut, d.out[2], ang, d.rl, d.tl, d.rs, d.out[0], param == GORT_JAC_LAI);
    });
}

int gort_energy_batch_dev(gort_ctx *ctx, void *stream, const gort_shape *shape, const double *structure,
                          const double *lut, const double *angles, const double *rleaf, const double *tleaf,
                          const double *rsoil, double *albedo, double *favegt, double *fasoil)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_shape(ctx, shape, "gort_energy_batch"));
    if (!structure || !lut || !angles || !rleaf || !tleaf || !rsoil || !albedo || !favegt || !fasoil)
        return set_error(ctx, GORT_ERR_INVALID, "gort_energy_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_energy(ctx, s, *shape, structure, lut, angles, rleaf, tleaf, rsoil, albedo, favegt, fasoil);
}

int gort_energy_batch(gort_ctx *ctx, const gort_shape *shape, const double *structure, const double *lut,
                      const double *angles, const double *rleaf, const double *tleaf, const double *rsoil,
                      double *albedo, double *favegt, double *fasoil)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_shape(ctx, shape, "gort_energy_batch"));
    if (!structure || !lut || !angles || !rleaf || !tleaf || !rsoil || !albedo || !favegt || !fasoil)
        return set_error(ctx, GORT_ERR_INVALID, "gort_energy_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    Staged d;
    TRY(stage_inputs(ctx, shape, structure, lut, angles, rleaf, tleaf, rsoil, &d));
    size_t n = (size_t) shape->n_sets * shape->n_geom * shape->n_wl;
    double *d_a, *d_v, *d_s;
    TRY(dout(ctx, 6, albedo, n, &d_a));
    TRY(dout(ctx, 7, favegt, n, &d_v));
    TRY(dout(ctx, 8, fasoil, n, &d_s));
    TRY(launch_energy(ctx, ctx->stream, *shape, d.st, d.lut, d.ang, d.rl, d.tl, d.rs, d_a, d_v, d_s));
    TRY(d2h(ctx, albedo, d_a, n));
    TRY(d2h(ctx, favegt, d_v, n));
    TRY(d2h(ctx, fasoil, d_s, n));
    return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_energy_batch");
}

// ---- sensor bands ---------------------------------------------------------------------------------
// host_weights: the rows are on the host and are checked here (the _dev entry points cannot look at device weights)
static int check_bands(gort_ctx *ctx, const gort_shape *sh, int n_bands, const double *weights, bool host_weights,
                       const char *who)
{
    TRY(check_shape(ctx, sh, who));
    if (n_bands < 1 || n_bands > GORT_MAX_BANDS)
        return set_error(ctx, GORT_ERR_INVALID, "%s: n_bands %d outside 1..%d", who, n_bands, GORT_MAX_BANDS);
    if (!weights) return set_error(ctx, GORT_ERR_INVALID, "%s: weights is NULL", who);
    if (sh->out_pitch != 0) return set_error(ctx, GORT_ERR_INVALID, "%s: band outputs are dense (out_pitch must be 0)", who);
    if (!host_weights) return GORT_OK;
    const size_t W = sh->n_wl;
    for (int b = 0; b < n_bands; b++) {
        int positive = 0;
        for (size_t i = 0; i < W; i++) {
            const double w = weights[(size_t) b * W + i];
            if (!isfinite(w) || w < 0.0) return set_error(ctx, GORT_ERR_INVALID, "%s: weight [%d][%zu] is not finite and >= 0", who, b, i);
            positive |= w > 0.0;
        }
        if (!positive) return set_error(ctx, GORT_ERR_INVALID, "%s: band %d has no positive weight", who, b);
    }
    return GORT_OK;
}

int gort_brdf_band_batch_dev(gort_ctx *ctx, void *stream, const gort_shape *shape, int n_bands, const double *weights,
                             const double *structure, const double *lut, const double *angles, const double *rleaf,
                             const double *tleaf, const double *rsoil, double *rband)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_bands(ctx, shape, n_bands, weights, false, "gort_brdf_band_batch"));
    if (!structure || !lut || !angles || !rleaf || !tleaf || !rsoil || !rband)
        return set_error(ctx, GORT_ERR_INVALID, "gort_brdf_band_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_brdf_band(ctx, s, *shape, n_bands, weights, structure, lut, angles, rleaf, tleaf, rsoil, rband);
}

int gort_brdf_band_batch(gort_ctx *ctx, const gort_shape *shape, int n_bands, const double *weights,
                         const double *structure, const double *lut, const double *angles, const double *rleaf,
                         const double *tleaf, const double *rsoil, double *rband)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_bands(ctx, shape, n_bands, weights, true, "gort_brdf_band_batch"));
    if (!structure || !lut || !angles || !rleaf || !tleaf || !rsoil || !rband)
        return set_error(ctx, GORT_ERR_INVALID, "gort_brdf_band_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    Staged d;
    TRY(stage_inputs(ctx, shape, structure, lut, angles, rleaf, tleaf, rsoil, &d));
    const size_t n = (size_t) shape->n_sets * shape->n_geom * n_bands;
    double *d_w, *d_out;
    TRY(h2d(ctx, 6, weights, (size_t) n_bands * shape->n_wl, &d_w));
    TRY(dout(ctx, 7, rband, n, &d_out));
    TRY(launch_brdf_band(ctx, ctx->stream, *shape, n_bands, d_w, d.st, d.lut, d.ang, d.rl, d.tl, d.rs, d_out));
    TRY(d2h(ctx, rband, d_out, n));
    TRY(check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_brdf_band_batch"));
    return check_pipeline_fault(ctx);
}

int gort_energy_band_batch_dev(gort_ctx *ctx, void *stream, const gort_shape *shape, int n_bands, const double *weights,
                               const double *structure, const double *lut, const double *angles, const double *rleaf,
                               const double *tleaf, const double *rsoil, double *albedo, double *favegt, double *fasoil)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_bands(ctx, shape, n_bands, weights, false, "gort_energy_band_batch"));
    if (!structure || !lut || !angles || !rleaf || !tleaf || !rsoil || !albedo || !favegt || !fasoil)
        return set_error(ctx, GORT_ERR_INVALID, "gort_energy_band_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    const cudaStream_t s = pick(ctx, stream);
    TRY(order_after_previous(ctx, s));
    return launch_energy_band(ctx, s, *shape, n_bands, weights, structure, lut, angles, rleaf, tleaf, rsoil, albedo, favegt, fasoil);
}

int gort_energy_band_batch(gort_ctx *ctx, const gort_shape *shape, int n_bands, const double *weights,
                           const double *structure, const double *lut, const double *angles, const double *rleaf,
                           const double *tleaf, const double *rsoil, double *albedo, double *favegt, double *fasoil)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_bands(ctx, shape, n_bands, weights, true, "gort_energy_band_batch"));
    if (!structure || !lut || !angles || !rleaf || !tleaf || !rsoil || !albedo || !favegt || !fasoil)
        return set_error(ctx, GORT_ERR_INVALID, "gort_energy_band_batch: NULL argument");
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    Staged d;
    TRY(stage_inputs(ctx, shape, structure, lut, angles, rleaf, tleaf, rsoil, &d));
    const size_t n = (size_t) shape->n_sets * shape->n_geom * n_bands;
    double *d_w, *d_a, *d_v, *d_s;
    TRY(h2d(ctx, 6, weights, (size_t) n_bands * shape->n_wl, &d_w));
    TRY(dout(ctx, 7, albedo, n, &d_a));
    TRY(dout(ctx, 8, favegt, n, &d_v));
    TRY(dout(ctx, 9, fasoil, n, &d_s));
    TRY(launch_energy_band(ctx, ctx->stream, *shape, n_bands, d_w, d.st, d.lut, d.ang, d.rl, d.tl, d.rs, d_a, d_v, d_s));
    TRY(d2h(ctx, albedo, d_a, n));
    TRY(d2h(ctx, favegt, d_v, n));
    TRY(d2h(ctx, fasoil, d_s, n));
    return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_energy_band_batch");
}

// gort_forward_batch with band outputs: the same chunked three-stream pipeline, with the spectra computed on the union U
// of the bands' supports only (the host compacts wavelengths and weight columns to U before the loop)
int gort_forward_band_batch(gort_ctx *ctx, const gort_shape *shape, int lut_method, const double *structure,
                            const double *leaf, const double *soil, double user_leaf, double user_soil,
                            const double *wavelength, int n_bands, const double *weights,
                            const double *angles, double *rband, double *lut_out)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRY(check_bands(ctx, shape, n_bands, weights, true, "gort_forward_band_batch"));
    if (!structure || !wavelength || !angles || !rband || (user_leaf < 0.0 && !leaf) || (user_soil < 0.0 && !soil))
        return set_error(ctx, GORT_ERR_INVALID, "gort_forward_band_batch: NULL argument");
    if (lut_method != GORT_LUT_FULL && lut_method != GORT_LUT_Q08)
        return set_error(ctx, GORT_ERR_INVALID, "gort_forward_band_batch: unknown LUT method %d", lut_method);
    const size_t G = shape->n_geom, W = shape->n_wl, B = n_bands;
    for (size_t i = 0; i < W; i++)
        if (wavelength[i] < GORT_WL_MIN || wavelength[i] > GORT_WL_MAX)
            return set_error(ctx, GORT_ERR_RANGE, "wavlength out of range (400-2500)");
    // union of the supports, in grid order
    std::vector<size_t> cols;
    for (size_t i = 0; i < W; i++) {
        bool any = false;
        for (size_t b = 0; b < B; b++) any |= weights[b * W + i] > 0.0;
        if (any) cols.push_back(i);
    }
    const size_t U = cols.size();
    std::vector<double> wl_u(U), w_u(B * U);
    for (size_t k = 0; k < U; k++) {
        wl_u[k] = wavelength[cols[k]];
        for (size_t b = 0; b < B; b++) w_u[b * U + k] = weights[b * W + cols[k]];
    }
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    // slot 22 the union's wavelengths, 23 shared angles, 24 the union's weights
    double *d_wl, *d_ang_shared = NULL, *d_w;
    TRY(h2d(ctx, 22, wl_u.data(), U, &d_wl));
    if (!shape->geom_per_set) TRY(h2d(ctx, 23, angles, 4 * G, &d_ang_shared));
    TRY(h2d(ctx, 24, w_u.data(), B * U, &d_w));
    gort_shape sh = *shape;
    sh.n_wl = (int) U;
    sh.spectra_per_set = 1;
    const size_t out_pm[3] = {G * B, 0, 0};
    const EnsCopy copies[2] = {{rband, 0, G * B}, {lut_out, -1, GORT_LUT_STRIDE}};
    // streams, chunking and events as gort_forward_batch
    return ensemble_chunks(ctx, shape, structure, leaf, soil, user_leaf, user_soil, angles, U, out_pm, 2, copies, "gort_forward_band_batch",
                           [&](cudaStream_t A, size_t c, const EnsBufs &d) {
        sh.n_sets = (int) c;
        TRY(launch_lut(ctx, A, (int) c, d.st, lut_method, d.lut));
        TRY(launch_spectra(ctx, A, (int) c, user_leaf < 0.0 ? d.leaf : NULL, user_soil < 0.0 ? d.soil : NULL, user_leaf, user_soil,
                           (int) U, d_wl, d.rl, d.tl, d.rs));
        return launch_brdf_band(ctx, A, sh, n_bands, d_w, d.st, d.lut, sh.geom_per_set ? d.ang : d_ang_shared,
                                d.rl, d.tl, d.rs, d.out[0]);
    });
}

int gort_gauleg(gort_ctx *ctx, double *abscissa, double *weights)
{
    if (!ctx || !abscissa || !weights) return GORT_ERR_INVALID;
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    TRYCUDA(ctx, cudaMemcpyAsync(abscissa, ctx->d_gauleg, sizeof(double) * GORT_NQUAD, cudaMemcpyDeviceToHost, ctx->stream), "gauleg copy");
    TRYCUDA(ctx, cudaMemcpyAsync(weights, ctx->d_gauleg + GORT_NQUAD, sizeof(double) * GORT_NQUAD, cudaMemcpyDeviceToHost, ctx->stream), "gauleg copy");
    return check_cuda(ctx, cudaStreamSynchronize(ctx->stream), "gort_gauleg");
}

int gort_dfma_peak(gort_ctx *ctx, double *tflops)
{
    if (!ctx || !tflops) return GORT_ERR_INVALID;
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    TRY(order_after_previous(ctx, ctx->stream));
    return launch_dfma_peak(ctx, ctx->stream, tflops);
}

int gort_kernel_stamps_enable(gort_ctx *ctx, int enable)
{
    if (!ctx) return GORT_ERR_INVALID;
    ctx->stamps_on = enable ? 1 : 0;
    return GORT_OK;
}

int gort_kernel_stamps(gort_ctx *ctx, double *span_us, double *startup_us, double *store_us, int *n_cta)
{
    if (!ctx) return GORT_ERR_INVALID;
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    return read_kernel_stamps(ctx, span_us, startup_us, store_us, n_cta);
}

int gort_profile_begin(gort_ctx *ctx, int max_steps)
{
    if (!ctx || max_steps <= 0) return GORT_ERR_INVALID;
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    if (ctx->prof_ev) { for (int i = 0; i < 3 * ctx->prof_cap; i++) cudaEventDestroy(ctx->prof_ev[i]); free(ctx->prof_ev); ctx->prof_ev = NULL; }
    ctx->prof_ev = (cudaEvent_t *) calloc((size_t) 3 * max_steps, sizeof(cudaEvent_t));
    if (!ctx->prof_ev) return set_error(ctx, GORT_ERR_NOMEM, "out of host memory");
    for (int i = 0; i < 3 * max_steps; i++) TRYCUDA(ctx, cudaEventCreate(&ctx->prof_ev[i]), "cudaEventCreate");
    ctx->prof_cap = max_steps;
    ctx->prof_n = 0;
    return GORT_OK;
}

int gort_profile_end(gort_ctx *ctx, double *geom_ms, double *rsurf_ms, int *n_steps)
{
    if (!ctx || !ctx->prof_ev) return GORT_ERR_INVALID;
    TRYCUDA(ctx, cudaSetDevice(ctx->device), "cudaSetDevice");
    double g = 0, r = 0;
    int n = ctx->prof_n;
    for (int i = 0; i < n; i++) {
        float a = 0, b = 0;
        TRYCUDA(ctx, cudaEventSynchronize(ctx->prof_ev[3 * i + 2]), "cudaEventSynchronize");
        TRYCUDA(ctx, cudaEventElapsedTime(&a, ctx->prof_ev[3 * i], ctx->prof_ev[3 * i + 1]), "cudaEventElapsedTime");
        TRYCUDA(ctx, cudaEventElapsedTime(&b, ctx->prof_ev[3 * i + 1], ctx->prof_ev[3 * i + 2]), "cudaEventElapsedTime");
        g += a; r += b;
    }
    for (int i = 0; i < 3 * ctx->prof_cap; i++) cudaEventDestroy(ctx->prof_ev[i]);
    free(ctx->prof_ev);
    ctx->prof_ev = NULL; ctx->prof_cap = 0; ctx->prof_n = 0;
    if (geom_ms) *geom_ms = n ? g / n : 0.0;
    if (rsurf_ms) *rsurf_ms = n ? r / n : 0.0;
    if (n_steps) *n_steps = n;
    return GORT_OK;
}

// ---- LUT text layout, gortt.c:123-146 -------------------------------------------------------------
long gort_lut_write_text(const double *lut, void *fp)
{
    if (!lut || !fp) return -GORT_ERR_INVALID;
    FILE *f = (FILE *) fp;
    long n = 0;
    for (int j = 0; j < GORT_LUT_FILE_ROWS; j++) {
        int k = fprintf(f, "%d %0.40f %0.40f\n", j, lut[j], lut[GORT_NTH + j]);
        if (k < 0) return -GORT_ERR_IO;
        n += k;
    }
    int k = fprintf(f, "-1 %0.40f %0.40f\n", lut[2 * GORT_NTH], lut[2 * GORT_NTH + 1]);
    if (k < 0) return -GORT_ERR_IO;
    return n + k;
}

int gort_lut_read_text(const char *path, double *lut)
{
    if (!path || !lut) return GORT_ERR_INVALID;
    FILE *f = fopen(path, "r");
    if (!f) return GORT_ERR_IO;
    int j, rows = 0;
    double x1, x2;
    while (fscanf(f, "%d %lf %lf", &j, &x1, &x2) == 3) {
        rows++;
        if (j >= 0) {
            if (j < GORT_NTH) { lut[j] = x1; lut[GORT_NTH + j] = x2; }   /* the reference has no bound */
        } else {
            lut[2 * GORT_NTH] = x1;
            lut[2 * GORT_NTH + 1] = x2;
        }
    }
    fclose(f);
    return rows > 0 ? GORT_OK : GORT_ERR_IO;      /* nothing parsable: not a LUT file */
}

}  // extern "C"
