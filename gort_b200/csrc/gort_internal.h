// gort_internal.h -- host-side internals of libgort_b200 (context, scratch buffers, launch
// prototypes).  Not part of the public ABI (include/gort_b200.h is).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include "../../include/gort_b200.h"

#define GORT_NSCRATCH 32
#define GORT_MAX_WIDE_CTAS 8192
#define GORT_BAND_SLOT (GORT_NSCRATCH - 1)   // scratch slot of the band supports (gort_*_band_batch[_dev])

struct gort_ctx {
    int device;
    cudaStream_t stream;
    cudaStream_t copy_stream;          // gort_forward_batch: inputs of the next chunk under the kernels of this one
    cudaStream_t copy_stream_out;      // gort_forward_batch: results of the previous chunk under the kernels of this one
    cudaEvent_t fwd_ev[6];             // its per-buffer events: inputs ready, kernels done, outputs copied (x2)
    char err[512];
    long launches;
    int sm_count;
    // grow-only device scratch used by the host-pointer entry points
    void *scratch[GORT_NSCRATCH];
    size_t scratch_cap[GORT_NSCRATCH];
    // grow-only device scratch used internally by _dev entry points (geometry records)
    void *work;
    size_t work_cap;
    // device constants built at creation
    double *d_gauleg;      // [2][32] abscissa, weights          (gauleg, gortt_albedo.c:142-198)
    double *d_prospect;    // [9][2101] refractive,k_Cab,k_Car,k_Anth,k_Brown,k_Cw,k_Cm, tav90, tav40
    double *d_soil;        // [4][421] Price EOF vectors
    // BRDF pipeline state (gort_brdf.cu).  Line records and their ready flags are double-buffered by call parity, so
    // that -- in overlap mode (gort_set_overlap) -- the geometry kernel of call i+1 can run under the store phase of call i
    void *rec_buf[2];                  // line records
    size_t rec_cap[2];
    unsigned long long *d_flags[2];    // [flag_cap] per buffer, one per 32-line tile; value = BRDF call number published
    size_t flag_cap[2];
    int rec_idx;
    unsigned long long *d_done;        // [GORT_MAX_WIDE_CTAS] per-CTA epoch of the last per-wavelength launch it finished; [+1] fault word
    unsigned long long epoch;          // per-wavelength launches so far
    unsigned long long call_no;        // BRDF calls so far
    unsigned long long last_sig[7];    // grid shape and output identity of the previous per-wavelength launch
    cudaStream_t last_stream;          // stream of the previous call (must stay alive until the next call or gort_synchronize)
    int last_was_wide;                 // the previous operation this context enqueued was a per-wavelength kernel
    int overlap;                       // gort_set_overlap: consecutive same-shape BRDF calls may overlap on the GPU
    const char *last_out_lo[3], *last_out_hi[3];   // byte ranges of the previous call's rsurf / scomp / kprop
    cudaEvent_t xstream_ev;            // orders calls issued on different streams (order_after_previous)
    struct { int key_lpt, key_scomp, key_tmab, key_threads; int occ; } wide_plan[8];
    int n_wide_plan;
    int geom_carveout_set, lut_attr_set, lut_tan_attr_set, band_attr_set;
    // development switch, read once from the environment by gort_create: GORT_TIMELINE=<call number>
    int dbg_timeline;
    unsigned long long *d_timeline;
    int timeline_calls;
    int stamps_on, stamps_ncta, stamps_half;       // gort_kernel_stamps
    cudaStream_t stamps_stream;
    // pinned-buffer placement (gort_host_alloc_near): probed once
    int near_probed, near_ncpu;
    int near_cpu[1024];
    char near_desc[512];
    // optional per-kernel event timing of the BRDF path (gort_profile_begin/end)
    cudaEvent_t *prof_ev;  // [3 * prof_cap]
    int prof_cap, prof_n;
};

namespace gort {

int set_error(gort_ctx *ctx, int code, const char *fmt, ...);
int check_cuda(gort_ctx *ctx, cudaError_t e, const char *what);
// returns device pointer with at least `bytes` capacity in scratch slot `slot`
void *scratch(gort_ctx *ctx, int slot, size_t bytes);
void *workspace(gort_ctx *ctx, size_t bytes);
void *rec_buffer(gort_ctx *ctx, int which, size_t bytes);
// any non-BRDF work this context enqueues ends the "previous operation was a per-wavelength kernel" state
inline void note_other_work(gort_ctx *ctx) { ctx->last_was_wide = 0; }
// every entry point calls this before it enqueues anything on `s`: consecutive calls on one context run one after the
// other whatever streams they use (they share the workspace, the record buffers and the pipeline flags)
int order_after_previous(gort_ctx *ctx, cudaStream_t s);

// kernels (device pointers, async on `s`)
int launch_brdf(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const double *structure,
                const double *lut, const double *angles, const double *rleaf, const double *tleaf,
                const double *rsoil, double *rsurf, double *scomp, double *kprop);
// the BRDF pipeline's record buffer and flags for a new call, and the geometry kernel that fills them (gort_brdf.cu)
int next_records(gort_ctx *ctx, cudaStream_t s, long L, double **rec, unsigned long long **flags);
int launch_geom(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const double *structure, const double *lut,
                const double *angles, double *rec, double *kprop, unsigned long long *flags, bool pdl);
// favd tangent of rsurf, drsurf [M][G][W] dense; lai != 0 scales it by d favd / d LAI (gort_tangent.cu)
int launch_brdf_tangent(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const double *structure, const double *lut,
                        const double *dlut, const double *angles, const double *rleaf, const double *tleaf,
                        const double *rsoil, double *drsurf, int lai);
int launch_energy(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const double *structure,
                  const double *lut, const double *angles, const double *rleaf, const double *tleaf,
                  const double *rsoil, double *albedo, double *favegt, double *fasoil);
// sensor bands: weights [n_bands][sh.n_wl] (device), outputs [M][G][n_bands]
int launch_brdf_band(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, int n_bands, const double *weights,
                     const double *structure, const double *lut, const double *angles, const double *rleaf,
                     const double *tleaf, const double *rsoil, double *rband);
int launch_energy_band(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, int n_bands, const double *weights,
                       const double *structure, const double *lut, const double *angles, const double *rleaf,
                       const double *tleaf, const double *rsoil, double *albedo, double *favegt, double *fasoil);
int launch_lut(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, int method, double *lut);
int launch_lut_out(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, int method, double *lut,
                   int n_dst, double *const *dst, int multicast);
// the same records and dlut [n_sets][GORT_LUT_STRIDE] = their favd tangent (gort_lut_tangent_batch_dev)
int launch_lut_tangent(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, int method, double *lut,
                       double *dlut);
int launch_lut_dead(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, double *vb, double *fb,
                    double *t_open, double *dt_open, double *dk_open, double *k_open);
int launch_spectra(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *leaf, const double *soil,
                   double user_leaf, double user_soil, int n_wl, const double *wl,
                   double *rleaf, double *tleaf, double *rsoil);
int launch_soil_table(gort_ctx *ctx, cudaStream_t s, const double *table, int n_sets, int n_wl, const double *wl, double *rsoil);
int launch_prospect_full(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *leaf, double *refl, double *tran);
int launch_jac_perturb(gort_ctx *ctx, cudaStream_t s, int n_sets, int row, double factor, const double *st_in, double *st_out);
int launch_jac_diff(gort_ctx *ctx, cudaStream_t s, int n_sets, long per_set, int row, int lai, double h, const double *st,
                    const double *fp, const double *fm, double *jac);
int read_kernel_stamps(gort_ctx *ctx, double *span_us, double *startup_us, double *store_us, int *n_cta);
int launch_gauleg(gort_ctx *ctx, cudaStream_t s, double *d_out /*[2][32]*/);
int launch_tav_tables(gort_ctx *ctx, cudaStream_t s, double *d_prospect);
int upload_soil_tables(gort_ctx *ctx, cudaStream_t s, double *d_soil);
int launch_dfma_peak(gort_ctx *ctx, cudaStream_t s, double *tflops);

}  // namespace gort
