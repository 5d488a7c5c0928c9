/* gort_b200.h -- C ABI of the B200-native GORT forward operator.
 *
 * The reference (tquaife/gort) has no plugin / FFI interface: its hot path sits behind the C
 * prototypes of include/gortt.h:216-277, called only from main() (gortt.c:108-120, :224-227,
 * :294-295, :322) with three mutable structs.  This header is the batched, re-entrant
 * replacement for exactly those prototypes.  Each entry point names the reference interface
 * it replaces.  Plain C types only: pointers, sizes, POD structs.
 *
 * Conventions
 *   - All arrays are FP64, structure-of-arrays, row-major, last index fastest.
 *   - "structure" is [6][n_sets]: rows lambda, r, b, h1, h2, favd  (gortt_parameters fields set
 *     by gortt.c:67-72 / gortt_cl_parser gortt.c:1026-1131).
 *   - "angles" is [4][n_lines]: rows vza, vaa, sza, saa in DEGREES, i.e. the columns of the
 *     reference's angles.dat (gortt.c:234, :1148).
 *   - a LUT record is GORT_LUT_STRIDE doubles: p_n0[0][0..90], epgap[0][0..90], k_open[0],
 *     k_openep[0] -- the only gap-probability results the BRDF reads (gortt.c:124-126,
 *     :896-910, :492-525).  The "-W"/"-P" text file holds rows 0..89 and the k_open pair.
 *   - Functions without a _dev suffix take HOST pointers: they copy inputs to the GPU, run the
 *     CUDA kernels and copy results back before returning.  _dev functions take DEVICE
 *     pointers, enqueue on `stream` (a cudaStream_t passed as void*, NULL = the context's own
 *     stream) and return without synchronising.
 *   - Every function returns GORT_OK or an error code; gort_last_error() gives the message.
 *     The reference convention (print to stderr, exit(EXIT_FAILURE)) is kept by the gortt CLI,
 *     not by the library.
 *   - There is no CPU fallback: without a CUDA device gort_create() fails.
 *   - Consecutive calls on one context run one after the other, whatever streams they use: a call on another stream
 *     than the previous call's waits for the work enqueued on that stream (the calls share the context's device
 *     scratch), and gort_synchronize() waits for every call.  So the previous call's stream must stay alive until the
 *     next call or gort_synchronize(); the Python binding's callers pass streams of a pool that never destroys them,
 *     so they meet this.  To run work concurrently, use two contexts.
 *   - gort_set_overlap(ctx, 1) (off by default) lets CONSECUTIVE gort_brdf_batch_dev calls of the same shape into the
 *     same output buffers overlap on the GPU: the geometry kernel of call i+1 runs under the store phase of call i;
 *     the stores of call i+1 to a region start only after call i's stores to that region are complete, so the
 *     results are exactly those of running the calls one after the other.  The library uses the overlap only when
 *     the previous operation THIS CONTEXT enqueued was such a call and no input (or kprop) of call i+1 lies inside an
 *     output buffer of call i.  The caller's side of the contract: between two such calls nothing else is enqueued
 *     on the stream that writes an input of the second call (kernels the library cannot see would otherwise be
 *     overtaken); copies, other gort_* calls and stream switches are seen and order the calls completely.
 *   - The in-kernel waits of the pipeline are bounded (2 s); should one ever expire, the affected CTAs store nothing
 *     and gort_synchronize() and the host-pointer entry points return GORT_ERR_CUDA with the number of the call.
 */
#ifndef GORT_B200_H
#define GORT_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GORT_NTH 91                         /* gortt.c:714 with dth = 1 degree */
#define GORT_NLAYERS 15                     /* gortt.c:78 */
#define GORT_LUT_STRIDE (2 * GORT_NTH + 2)  /* 184 doubles per parameter set */
#define GORT_LUT_FILE_ROWS 90               /* gortt.c:124 */
#define GORT_NQUAD 32                       /* gortt.c:93 npoints */
#define GORT_WL_MIN 400.0                   /* gortt.c:1299, :1350 */
#define GORT_WL_MAX 2500.0

enum {
    GORT_OK = 0,
    GORT_ERR_INVALID = 1,   /* bad argument */
    GORT_ERR_CUDA = 2,      /* CUDA runtime / launch failure, or no device */
    GORT_ERR_RANGE = 3,     /* wavelength outside 400-2500 nm (gortt.c:1299-1302, :1350-1353) */
    GORT_ERR_NOMEM = 4,
    GORT_ERR_IO = 5
};

enum { GORT_LUT_FULL = 0, GORT_LUT_Q08 = 1 };   /* gortt.c:116-120 */

typedef struct gort_ctx gort_ctx;

/* Run-time options of the BRDF path that the reference keeps in gortt_parameters:
 * -beta (gortt.c:1039, gortt_brdf.c:157) and -diffuse (gortt.c:1041, :290-291). */
typedef struct {
    int use_beta;
    double beta;
    int use_fd;
    double fd;      /* already 1 - arg, as the reference stores it */
} gort_options;

/* Shape of one batched BRDF / energy call. */
typedef struct {
    int n_sets;            /* M canopy parameter sets */
    int n_geom;            /* G input lines per set */
    int n_wl;              /* W wavelengths */
    int geom_per_set;      /* 0: angles is [4][G], shared by all sets; 1: [4][M*G], set-major */
    int spectra_per_set;   /* 0: rleaf/tleaf/rsoil are [W]; 1: [M][W] */
    gort_options opt;
    int out_pitch;         /* row stride, in doubles, of rsurf (and, x4, of scomp); 0 = n_wl (dense).
                              A multiple of 16 keeps every row 128-byte aligned in HBM; the padding columns
                              [n_wl, min(out_pitch, round_up(n_wl, 16))) then belong to the call and receive
                              copies of column n_wl-1, so that no row ends in a partially written line (the
                              same store stream runs 1.12x faster; an odd stride such as 2101 costs 1.5x).
                              Columns beyond that are never touched. */
} gort_shape;

/* ---- context ---------------------------------------------------------------------------- */
int gort_create(int device, gort_ctx **out);
void gort_destroy(gort_ctx *ctx);
const char *gort_last_error(const gort_ctx *ctx);      /* ctx may be NULL: creation errors */
void *gort_stream(gort_ctx *ctx);                       /* the context's cudaStream_t */
int gort_synchronize(gort_ctx *ctx);
/* allow consecutive same-shape gort_brdf_batch_dev calls to overlap (see the conventions above); default 0 */
int gort_set_overlap(gort_ctx *ctx, int enable);
int gort_device_count(void);
/* pinned host memory for fast H2D/D2H through the host-pointer entry points */
void *gort_host_alloc(size_t bytes);
void gort_host_free(void *p);
/* Where pinned pages land decides the PCIe rate of the host-pointer entry points once several GPUs copy at the same
 * time.  Measured on a 2-GPU box whose VM reports a single NUMA node (neither sysfs nor `nvidia-smi topo` reveals
 * anything there): two ranks copying 196 MB each get 57 GB/s per GPU into buffers pinned from CPUs 0-5 and 34.5 GB/s
 * from the other 18; one rank alone gets 57 GB/s either way.
 *   gort_host_alloc_on_cpus  pins the buffer (and touches every page) while the calling thread runs on the given
 *                            CPUs, then restores the thread's affinity: the primitive a multi-process job uses after
 *                            probing placements with all its ranks copying at once (bench.py does exactly that).
 *   gort_host_alloc_near     a single-context probe: for up to 8 groups of the CPUs this thread may run on it pins a
 *                            32 MB buffer from that group and times one device-to-host copy; the best group (ties:
 *                            the lowest CPUs) is remembered in the context and used for every later buffer.  It can
 *                            only see differences that a single copy stream exposes.
 *   gort_host_placement      describes what the probe found. */
void *gort_host_alloc_on_cpus(size_t bytes, const int *cpus, int n_cpus);
void *gort_host_alloc_near(gort_ctx *ctx, size_t bytes);
int gort_host_placement(gort_ctx *ctx, char *buf, size_t len);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
long gort_launch_count(const gort_ctx *ctx);

/* ---- gap probabilities: replaces gortt_init_params + gortt_gap_probabilities /
 *      gortt_gap_probabilities_Q08 (include/gortt.h:217,251; gortt.c:108-120) ------------- */
int gort_lut_batch(gort_ctx *ctx, int n_sets, const double *structure, int method, double *lut);
int gort_lut_batch_dev(gort_ctx *ctx, void *stream, int n_sets, const double *structure,
                       int method, double *lut);
/* The same records, and copies of them stored by the producing kernels into further tables: the multi-GPU assembly of a
 * LUT grid (BASELINE config 5) without a collective after the kernels.  Every rank owns a block of parameter sets and
 * holds a full table; `lut` is this rank's block inside its own table, dst[0..n_dst) (a HOST array of device
 * addresses, n_dst <= GORT_LUT_MAX_DST) are the addresses of the same block inside the other ranks' tables, mapped into
 * this process (CUDA peer / symmetric memory over NVLink), or -- multicast != 0 -- NVSwitch multicast addresses of it,
 * each written once and delivered to every GPU bound to the multicast object.  The stores are ordinary posted writes
 * issued by the kernels that produce the rows (they run underneath the arithmetic of the other CTAs); they are
 * complete when the work enqueued by this call is.  The caller synchronises the ranks around the call (nobody may
 * still read the old contents; everybody must have finished before the table is read) -- gort_b200/parallel.py does
 * it with the symmetric-memory barrier.  No reference counterpart (the reference computes one record per process,
 * gortt.c:108-120). */
#define GORT_LUT_MAX_DST 16
int gort_lut_batch_scatter_dev(gort_ctx *ctx, void *stream, int n_sets, const double *structure, int method,
                               double *lut, int n_dst, double *const *dst, int multicast);

/* ---- the intermediates of gortt_gap_probabilities that never reach the BRDF or albedo path (SURVEY.md 8f row 1):
 *      gortt_calc_vb / gortt_calc_fb / gortt_calc_t_open (gortt_pn_kopen.c:925-1078) and the dk_open / k_open[h] rows of
 *      gortt_calc_kopen (:351-375), for callers of the reference's unfinished LiDAR / energy extensions and for
 *      "same work as the reference" timings (gortt_calc_t_open is ~90 % of the reference's LUT time).
 *      Outputs per set, any of which may be NULL: vb [M][15], fb [M][15][91], t_open [M][15][15], dt_open [M][15][15],
 *      dk_open [M][15], k_open [M][15].  A set on which the reference would exit ("Significant negative volume",
 *      :964-967) gets NaN in vb.  GORT_LUT_FULL only. */
int gort_lut_intermediates_batch(gort_ctx *ctx, int n_sets, const double *structure, double *vb, double *fb,
                                 double *t_open, double *dt_open, double *dk_open, double *k_open);
int gort_lut_intermediates_batch_dev(gort_ctx *ctx, void *stream, int n_sets, const double *structure, double *vb,
                                     double *fb, double *t_open, double *dt_open, double *dk_open, double *k_open);

/* ---- spectra: replaces gortt_price_soil + gortt_prospect_interface + prospect_DB_
 *      (include/gortt.h:289-292; gortt.c:224-227).
 *      leaf is [7][M] rows N,Cab,Car,Anth,Cbrown,Cw,Cm; soil is [4][M] rows rsl1..4.
 *      user_leaf >= 0 is "-alb_leaf" (gortt.c:1355-1357), user_soil >= 0 is "-alb_soil"
 *      (gortt.c:1305-1307); pass a negative value for "not set".
 *      Outputs are [M][W]. ------------------------------------------------------------------ */
int gort_spectra_batch(gort_ctx *ctx, int n_sets, const double *leaf, const double *soil,
                       double user_leaf, double user_soil, int n_wl, const double *wavelength,
                       double *rleaf, double *tleaf, double *rsoil);
int gort_spectra_batch_dev(gort_ctx *ctx, void *stream, int n_sets, const double *leaf,
                           const double *soil, double user_leaf, double user_soil, int n_wl,
                           const double *wavelength, double *rleaf, double *tleaf, double *rsoil);
/* the full 2101-band PROSPECT-D output of prospect_DB_ (prospect_DB.f90:72): refl, tran [M][2101] */
int gort_prospect_batch(gort_ctx *ctx, int n_sets, const double *leaf, double *refl, double *tran);

/* ---- soil spectrum from a file ("-soil_spectra file", gortt.c:1056-1060).  The reference's reader
 *      gortt_read_soil_lut (gortt.c:1388-1451) is unfinished: it builds the 1-nm table, prints it and exits, and the
 *      lookup gortt_get_rsoil_lut it was meant to feed is declared (include/gortt.h:296) but never defined.  These two
 *      calls finish the feature with the documented file format (gortt.c:1377-1387).
 *      gort_soil_table_read: text file, one "wavelength_nm albedo" pair per line, ascending, first wavelength <= 400,
 *      last >= 2500, arbitrary sampling -> table[GORT_SOIL_TABLE_NW] on the 1-nm grid 400..2500 by the reference's own
 *      interpolation loop (gortt.c:1420-1428).  Host-side parsing only.  On error returns GORT_ERR_IO and writes the
 *      reference's message (without the "gortt: " prefix) into errbuf.
 *      gort_soil_from_table[_dev]: rsoil [M][W] at arbitrary wavelengths from such a table (shared by all M sets):
 *      linear interpolation between the two neighbouring 1-nm rows, indices and fraction formed as
 *      gortt_price_soil forms them for its 5-nm tables (gortt.c:1311-1314: upper = 1 + (wl-400)/1, lower = (wl-400)/1,
 *      FP64 fraction); wavelengths outside 400-2500 are GORT_ERR_RANGE (NaN from the _dev form). */
#define GORT_SOIL_TABLE_NW 2101
int gort_soil_table_read(const char *path, double *table, char *errbuf, size_t errlen);
int gort_soil_from_table(gort_ctx *ctx, const double *table, int n_sets, int n_wl, const double *wavelength,
                         double *rsoil);
int gort_soil_from_table_dev(gort_ctx *ctx, void *stream, const double *table, int n_sets, int n_wl,
                             const double *wavelength, double *rsoil);

/* ---- BRDF: replaces the per-line block of main (gortt.c:240-295):
 *      angle normalisation, gortt_prime_theta, fd, gortt_set_zenith_dependant_probabilities,
 *      gortt_rsurf (include/gortt.h:216-219).
 *      rsurf [M][G][pitch] (pitch = shape.out_pitch, default W); scomp (optional, may be NULL)
 *      [M][G][pitch][4] = C,G,T,Z (gortt.c:562-565), 32-byte aligned (each quadruple is stored as one vector;
 *      any other address is GORT_ERR_INVALID and nothing is enqueued);
 *      kprop (optional) [M][G][4] = Kc,Kg,Kt,Kz (gortt.c:570-573). -------------------------- */
int gort_brdf_batch(gort_ctx *ctx, const gort_shape *shape, const double *structure,
                    const double *lut, const double *angles,
                    const double *rleaf, const double *tleaf, const double *rsoil,
                    double *rsurf, double *scomp, double *kprop);
int gort_brdf_batch_dev(gort_ctx *ctx, void *stream, const gort_shape *shape,
                        const double *structure, const double *lut, const double *angles,
                        const double *rleaf, const double *tleaf, const double *rsoil,
                        double *rsurf, double *scomp, double *kprop);

/* ---- forward operator for an ensemble: replaces the body of main for M members at once (gortt.c:108-120 gap
 *      probabilities, :224-227 spectra, :232-329 the per-line block) with everything but the inputs and rsurf staying
 *      on the GPU: the data-assimilation use case (BASELINE.json config 4).  Host pointers.
 *      structure [6][M]; leaf [7][M] / soil [4][M] (NULL when user_leaf / user_soil >= 0); wavelength [W];
 *      angles [4][G] or [4][M][G] per shape->geom_per_set; shape->spectra_per_set is ignored (spectra are per member).
 *      rsurf [M][G][W] dense; lut_out (optional, may be NULL) receives the LUT records [M][GORT_LUT_STRIDE].
 *      Members are processed in chunks on two streams: the copies of one chunk run under the kernels of the next. */
int gort_forward_batch(gort_ctx *ctx, const gort_shape *shape, int lut_method, const double *structure,
                       const double *leaf, const double *soil, double user_leaf, double user_soil,
                       const double *wavelength, const double *angles, double *rsurf, double *lut_out);

/* ---- Jacobian of the BRDF with respect to one canopy parameter (SURVEY.md 8f row 4, for variational data
 *      assimilation; the reference has no derivative code -- its only hook is the LAI -> favd mapping of
 *      gortt.c:1127-1131, favd = 3 LAI / (4 lambda pi r^2 b)).
 *      Central differences through the whole chain on the GPU: for every member the chosen structure row is scaled by
 *      (1 +- rel_step), gap probabilities and BRDF are evaluated for both (the spectra once), and a difference kernel
 *      forms  d rsurf / d p = (f(p (1 + h)) - f(p (1 - h))) / (2 h p);  only the Jacobian (and, if asked for, the
 *      unperturbed rsurf) travels back.  Host pointers; arguments as gort_forward_batch.
 *      param: GORT_JAC_LAMBDA .. GORT_JAC_FAVD = the structure row itself; GORT_JAC_LAI = leaf area index at fixed crown
 *      geometry, i.e. d/d favd times favd / LAI.  rel_step <= 0 selects 1e-4 (truncation ~1e-8 relative, rounding
 *      ~1e-12 / h).  The chain is smooth in lambda and favd (LAI); in r, b, h1, h2 it is only piecewise smooth -- the
 *      path-length histogram of gortt_get_pd_s bins on the crown shape ((int)(s/ds + 0.5), gortt_pn_kopen.c:134-139) --
 *      so those derivatives carry jumps of the size of a bin flip divided by the step.
 *      jac [M][G][W]; rsurf (optional, may be NULL) [M][G][W]. */
enum { GORT_JAC_LAMBDA = 0, GORT_JAC_R = 1, GORT_JAC_B = 2, GORT_JAC_H1 = 3, GORT_JAC_H2 = 4, GORT_JAC_FAVD = 5, GORT_JAC_LAI = 6 };
int gort_jacobian_batch(gort_ctx *ctx, const gort_shape *shape, int lut_method, int param, double rel_step,
                        const double *structure, const double *leaf, const double *soil, double user_leaf,
                        double user_soil, const double *wavelength, const double *angles, double *jac, double *rsurf);

/* ---- energy balance: replaces gortt_energy / gortt_albedo / gauleg (include/gortt.h:273-275;
 *      gortt.c:208-209, :322).  One result per input line (only sza/saa of the line matter):
 *      albedo, favegt, fasoil are [M][G][W]. ---------------------------------------------- */
int gort_energy_batch(gort_ctx *ctx, const gort_shape *shape, const double *structure,
                      const double *lut, const double *angles,
                      const double *rleaf, const double *tleaf, const double *rsoil,
                      double *albedo, double *favegt, double *fasoil);
int gort_energy_batch_dev(gort_ctx *ctx, void *stream, const gort_shape *shape,
                          const double *structure, const double *lut, const double *angles,
                          const double *rleaf, const double *tleaf, const double *rsoil,
                          double *albedo, double *favegt, double *fasoil);
/* the 32-point Gauss-Legendre rule the energy path uses (gauleg, gortt_albedo.c:142-198) */
int gort_gauleg(gort_ctx *ctx, double *abscissa, double *weights);

/* ---- LUT text layout ("-W" / "-P", gortt.c:123-146) -- host-side formatting only --------- */
/* writes 90 rows "%d %0.40f %0.40f\n" and the "-1" row for one LUT record; returns bytes
 * written or a negative GORT_ERR_*.  fp is a FILE*. */
long gort_lut_write_text(const double *lut, void *fp);
/* fscanf("%d %lf %lf") loop into a LUT record that the caller has pre-filled (the reference
 * reads over whatever gortt_init_params left: zeros) */
int gort_lut_read_text(const char *path, double *lut);

/* ---- measurement helpers --------------------------------------------------------------- */
/* FP64 FMA peak of this device, measured with a register-resident DFMA loop (TFLOP/s) */
int gort_dfma_peak(gort_ctx *ctx, double *tflops);
/* Per-kernel device timing of the BRDF path with CUDA events recorded on the launching stream.
 * gort_profile_begin arms up to max_steps BRDF calls; each armed gort_brdf_batch[_dev] records
 * events around its geometry kernel and its per-wavelength kernel.  gort_profile_end synchronises,
 * disarms and returns the mean milliseconds per call of each kernel over the recorded calls. */
int gort_profile_begin(gort_ctx *ctx, int max_steps);
int gort_profile_end(gort_ctx *ctx, double *geom_ms, double *rsurf_ms, int *n_steps);

/* In-kernel view of the per-wavelength kernel (W >= 64): with stamps enabled every CTA of the kernel records
 * %globaltimer at its phase boundaries (a store of 8 bytes per phase by one thread: no measurable cost); while stamps are
 * enabled BRDF calls run in plain stream order (no overlap between kernels or calls), so that a launch is separable.
 * gort_kernel_stamps synchronises the launching stream and returns, for the most recent such launch: the span from the
 * first CTA's first instruction to the last CTA's last completed store, and the per-CTA means of the start-up (entry to
 * first store) and store phases, in microseconds.  CUDA events around a launch additionally contain the launch and
 * completion latency outside any CTA; the difference is what a roofline fraction taken from event times cannot show. */
int gort_kernel_stamps_enable(gort_ctx *ctx, int enable);
int gort_kernel_stamps(gort_ctx *ctx, double *span_us, double *startup_us, double *store_us, int *n_cta);

#ifdef __cplusplus
}
#endif
#endif /* GORT_B200_H */
