// gort_brdf.cu -- BRDF and energy-balance kernels (sm_100a, FP64, no tensor cores: nothing here
// is a dense contraction).
//
//   geom_kernel          everything gortt_rsurf does before its wavelength loop (gortt.c:240-291, :424-449,
//                        gortt_brdf.c:7-238, :638-702) -> packed 128-byte line record in HBM.  32 lines x 5 role
//                        warps per CTA (latency-bound: few lines); geom_lines_kernel is the one-thread-per-line
//                        form for batches that fill the GPU (ensembles).  Both publish per-tile ready flags.
//   rsurf_wide_kernel    W >= 64 (gort_rsurf_wide.cuh): one CTA per (wavelength chunk, contiguous line range);
//                        (set, lambda) terms in shared memory, (sun, lambda) terms in registers, 5 FMAs and one
//                        coalesced store per evaluation; pipelined with geom_kernel and across calls.
//   rsurf_flat_kernel    W < 64 (band sets): one thread per (line, band).
//   energy_zenith_kernel / energy_kernel   hemispherical quadrature for albedo / fAPAR (gortt_albedo.c): the
//                        quadrature collapses onto five weighted sums of node coefficients.
//   gauleg_kernel, dfma_kernel            Gauss-Legendre nodes; FP64 FMA microbenchmark.
#include <stdio.h>
#include <stdlib.h>
#include "gort_device.cuh"
#include "gort_internal.h"
#include "gort_rsurf_wide.cuh"
#include "gort_rsurf_rows.cuh"

namespace gort {

// ------------------------------------------------------------------------------------------------
// geom_kernel: one CTA = 32 lines x 5 role warps.  A line's record is ~4200 dependent SASS instructions
// when one thread computes it (45 FP64 libm calls); with a few hundred warps on 592 SM sub-partitions the
// kernel is pure latency (18.6 us for 11 664 lines, ncu profiles/r1d).  The roles below have no data
// dependence on each other, so five warps compute them side by side and warp 0 combines them:
//   warp 0  pass at the actual relative azimuth (overlap, Kg, f, F)       gortt_brdf.c:7-100, :171-238
//   warp 1  pass at raa = 0                                              gortt_brdf.c:143-146
//   warp 2  pass at raa = pi                                             gortt_brdf.c:147-150
//   warp 3  exp terms of Kz / K'g / t0 and the mutual-shadowing beta     gortt.c:439-449, gortt_brdf.c:223-232
//   warp 4  zenith interpolation of the LUT and the Kuusk hotspot        gortt.c:872-915, gortt_brdf.c:638-702
#define GEOM_ROLES 5
// The first `n_tiles` CTAs of a geometry kernel do not compute line records: they fill the (set, lambda) table the
// full-spectrum per-wavelength kernel loads (gort_rsurf_rows.cuh) and publish one flag per tile.  n_tiles = 0: none.
struct TableJob {
    int n_tiles, n_wl, spectra_per_set, ncolt;
    const double *rleaf, *tleaf, *rsoil;
    double *table;
    unsigned long long *flags;          // one per tile
};

__global__ void __launch_bounds__(32 * GEOM_ROLES)
geom_kernel(int n_sets, int n_geom, int geom_per_set, gort_options opt,
            const double* __restrict__ structure, const double* __restrict__ lut,
            const double* __restrict__ angles, double* __restrict__ rec, double* __restrict__ kprop,
            unsigned long long* __restrict__ tile_flags, unsigned long long call_no, const TableJob tj)
{
    // let the dependent per-wavelength kernel start its prologue while this grid runs: it never waits for this
    // grid's completion, it acquires the per-tile flags published below
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if ((int) blockIdx.x < tj.n_tiles) {
        leaf_table_tile(blockIdx.x, n_sets, tj.n_wl, tj.spectra_per_set, tj.ncolt, structure, lut, tj.rleaf, tj.tleaf,
                        tj.rsoil, tj.table, tj.flags, call_no);
        return;
    }
    const unsigned gblock = blockIdx.x - tj.n_tiles;
    __shared__ double ex[12][32];
    const long L = (long) n_sets * n_geom;
    const int lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    const long line_raw = (long) gblock * 32 + lane;
    const long line = min(line_raw, L - 1);
    const int m = (int) (line / n_geom);
    const long a = geom_per_set ? line : (line - (long) m * n_geom);
    const long na = geom_per_set ? L : n_geom;
    const Canopy c = canopy_load(structure, n_sets, m, lut);
    const Line g = line_from_degrees(angles[0 * na + a], angles[1 * na + a], angles[2 * na + a], angles[3 * na + a]);
    // roles 0-2 run ONE copy of the pass code with their own relative azimuth (three inlined copies of the
    // libm-heavy pass made the kernel instruction-fetch bound: stall_no_instruction was its top stall).
    // The raa-independent crown terms (2 exp, acos) come from role 3 through shared memory: named barrier 1
    // joins warps 0-3 half-way, so those terms leave the critical path of the passes.
    Primed P;
    Pass pa = {0.0, 0.0, 0.0};
    if (role < 4) P = primed_trig(c, g.vza, g.sza);
    if (role < 3) {
        double raa = g.raa, cr = 1.0, sr = 0.0;
        if (role == 0) sincos(g.raa, &sr, &cr);
        else if (role == 1) raa = 0.0;
        else { raa = GORT_PI; cr = -1.0; sr = GORT_SIN_PI; }
        const PassA a1 = kc_pass_a(c, P, cr, sr);
        asm volatile("bar.sync 1, 128;" ::: "memory");
        CrownLite s;
        s.Mv = ex[9][lane]; s.theta_Mi = ex[10][lane]; s.Gamma_v = ex[11][lane];
        const bool vgs = fabs(g.vza) > fabs(g.sza);
        pa = kc_pass_b(P, a1, s, vgs, raa, cr);
        if (role > 0) ex[role - 1][lane] = pa.f * pa.F;
    } else if (role == 3) {
        const CrownLite s = crown_lite(c, P.t);
        ex[9][lane] = s.Mv; ex[10][lane] = s.theta_Mi; ex[11][lane] = s.Gamma_v;
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const Tail tl = tail_terms(c, P, opt);
        ex[2][lane] = tl.e_v; ex[3][lane] = tl.e_s; ex[4][lane] = tl.t0; ex[5][lane] = tl.beta;
    } else {
        double sr, cr;
        sincos(g.raa, &sr, &cr);
        const Hot h = hotspot(c, lut + (size_t) m * GORT_LUT_STRIDE, g.vza, g.sza, cr);
        ex[6][lane] = h.kuusk; ex[7][lane] = h.pn0_s; ex[8][lane] = h.pe_s;
    }
    __syncthreads();
    if (role != 0) return;
    if (line_raw < L) {
    Tail tl; Hot h;
    tl.e_v = ex[2][lane]; tl.e_s = ex[3][lane]; tl.t0 = ex[4][lane]; tl.beta = ex[5][lane];
    h.kuusk = ex[6][lane]; h.pn0_s = ex[7][lane]; h.pe_s = ex[8][lane];
    const double fd = opt.use_fd ? opt.fd : cos(g.sza) / (cos(g.sza) + 0.09);       // gortt.c:290-291
    const GeomRec r = geom_combine(c, P, pa, ex[0][lane], ex[1][lane], tl, h, g.raa, fd);
    // flags bit0: the sun of this line differs from the previous line's (every sun-dependent term is a
    // function of |sza| and the set only); bit1: first line of a parameter set
    int flags = 0;
    if (line % n_geom == 0) flags = 3;
    else if (fabs(angles[2 * na + a]) != fabs(angles[2 * na + a - 1])) flags = 1;
    double2* o = reinterpret_cast<double2*>(rec + (size_t) line * GORT_REC_STRIDE);
    o[0] = make_double2(r.cA, r.Kc);   o[1] = make_double2(r.cG, r.cZ);
    o[2] = make_double2(r.Kt, __longlong_as_double((long long) flags));
    o[3] = make_double2(r.q, r.fd);
    o[4] = make_double2(r.mus, r.t0);  o[5] = make_double2(r.tp0, r.pe_s);
    o[6] = make_double2(r.Kpg, r.Kpz); o[7] = make_double2(r.Kg, r.Kz);
    if (kprop) {
        kprop[4 * line + 0] = r.Kc; kprop[4 * line + 1] = r.Kg;
        kprop[4 * line + 2] = r.Kt; kprop[4 * line + 3] = r.Kz;
    }
    }
    // publish this tile: the per-wavelength kernel waits on these flags, not on the completion of this grid (a
    // grid launched as a programmatic dependent is not complete before its predecessors in the stream are)
    __syncwarp();
    if (lane == 0) {
        __threadfence();
        asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(tile_flags + gblock), "l"(call_no) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// geom_lines_kernel: the same record, one thread per line.  With hundreds of thousands of lines (ensembles: 10^5
// members x 16 geometries) the GPU is full and throughput counts, not the latency of one line; the role split of
// geom_kernel repeats the primed trig and the crown terms in four warps (1.8x the instructions), so large batches
// take this kernel instead.  Same device functions in the same order: same bits.
__global__ void __launch_bounds__(128, 6)
geom_lines_kernel(int n_sets, int n_geom, int geom_per_set, gort_options opt,
                  const double* __restrict__ structure, const double* __restrict__ lut,
                  const double* __restrict__ angles, double* __restrict__ rec, double* __restrict__ kprop,
                  unsigned long long* __restrict__ tile_flags, unsigned long long call_no, const TableJob tj)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if ((int) blockIdx.x < tj.n_tiles) {
        leaf_table_tile(blockIdx.x, n_sets, tj.n_wl, tj.spectra_per_set, tj.ncolt, structure, lut, tj.rleaf, tj.tleaf,
                        tj.rsoil, tj.table, tj.flags, call_no);
        return;
    }
    const long L = (long) n_sets * n_geom;
    const long line = (long) (blockIdx.x - tj.n_tiles) * blockDim.x + threadIdx.x;
    if (line < L) {
        const int m = (int) (line / n_geom);
        const long a = geom_per_set ? line : (line - (long) m * n_geom);
        const long na = geom_per_set ? L : n_geom;
        const Canopy c = canopy_load(structure, n_sets, m, lut);
        const Line g = line_from_degrees(angles[0 * na + a], angles[1 * na + a], angles[2 * na + a], angles[3 * na + a]);
        const double fd = opt.use_fd ? opt.fd : cos(g.sza) / (cos(g.sza) + 0.09);       // gortt.c:290-291
        const GeomRec r = geom_record(c, lut + (size_t) m * GORT_LUT_STRIDE, opt, g.vza, g.sza, g.raa, fd);
        int flags = 0;
        if (line % n_geom == 0) flags = 3;
        else if (fabs(angles[2 * na + a]) != fabs(angles[2 * na + a - 1])) flags = 1;
        double2* o = reinterpret_cast<double2*>(rec + (size_t) line * GORT_REC_STRIDE);
        o[0] = make_double2(r.cA, r.Kc);   o[1] = make_double2(r.cG, r.cZ);
        o[2] = make_double2(r.Kt, __longlong_as_double((long long) flags));
        o[3] = make_double2(r.q, r.fd);
        o[4] = make_double2(r.mus, r.t0);  o[5] = make_double2(r.tp0, r.pe_s);
        o[6] = make_double2(r.Kpg, r.Kpz); o[7] = make_double2(r.Kg, r.Kz);
        if (kprop) {
            kprop[4 * line + 0] = r.Kc; kprop[4 * line + 1] = r.Kg;
            kprop[4 * line + 2] = r.Kt; kprop[4 * line + 3] = r.Kz;
        }
    }
    // a warp is one 32-line tile
    __syncwarp();
    if ((threadIdx.x & 31) == 0 && (line >> 5) <= ((L - 1) >> 5)) {
        __threadfence();
        asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(tile_flags + (line >> 5)), "l"(call_no) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
rsurf_flat_kernel(int n_sets, int n_geom, int n_wl, int spectra_per_set, long pitch,
                  const double* __restrict__ structure, const double* __restrict__ lut,
                  const double* __restrict__ rec,
                  const double* __restrict__ rleaf, const double* __restrict__ tleaf,
                  const double* __restrict__ rsoil,
                  double* __restrict__ rsurf, double* __restrict__ scomp)
{
    const long L = (long) n_sets * n_geom;
    const long total = L * n_wl;
    long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const long line = e / n_wl;
    const int w = (int) (e - line * n_wl);
    const int m = (int) (line / n_geom);
    Canopy c = canopy_load(structure, n_sets, m, lut);
    const size_t sb = (spectra_per_set ? (size_t) m * n_wl : 0) + w;
    LeafTerms Lf = leaf_terms(c, rleaf[sb], tleaf[sb], rsoil[sb]);
    const double2* rr = reinterpret_cast<const double2*>(rec + (size_t) line * GORT_REC_STRIDE);
    // (cA,Kc) (cG,cZ) (Kt,flags) (q,fd) | (mus,t0) (tp0,pe_s) (K'g,K'z) (Kg,Kz)
    const double2 v0 = rr[0], v2 = rr[2], v3 = rr[3], s0v = rr[4], s1v = rr[5], v6 = rr[6], v7 = rr[7];
    const double fd = v3.y;
    SunTerms S = sun_terms(c, Lf, fd, s0v.x, s0v.y, s1v.x, s1v.y);
    double C;
    double r = view_rsurf(c, Lf, S, fd, v3.x, v0.y, v7.x, v2.x, v7.y, v6.x, v6.y, C);
    const size_t o = (size_t) line * pitch + w;
    rsurf[o] = r;
    if (scomp) *reinterpret_cast<double4*>(scomp + 4 * o) = make_double4(C, S.G, S.T, S.Z);
}

// Development aid: with GORT_TIMELINE=<call number> in the environment of gort_create, every per-wavelength CTA records
// %globaltimer stamps at its phase boundaries; after the given call the stamps of that call and the one before it are
// summarised on stderr.
static unsigned long long *timeline_half(gort_ctx *ctx, unsigned long long epoch)
{
    if (!ctx->dbg_timeline && !ctx->stamps_on) return NULL;
    if (!ctx->d_timeline && cudaMalloc((void **) &ctx->d_timeline, 2 * 64 * GORT_MAX_WIDE_CTAS) != cudaSuccess) return NULL;
    return ctx->d_timeline + (epoch & 1) * 8 * GORT_MAX_WIDE_CTAS;
}

static void timeline_report(gort_ctx *ctx, cudaStream_t s, int ncta, int half, const char *kernel)
{
    if (!ctx->dbg_timeline || ++ctx->timeline_calls != ctx->dbg_timeline) return;
    cudaStreamSynchronize(s);
    unsigned long long *h = (unsigned long long *) malloc(64 * (size_t) ncta), *prev = (unsigned long long *) malloc(64 * (size_t) ncta);
    if (!h || !prev) { free(h); free(prev); return; }
    cudaMemcpy(h, ctx->d_timeline + half * 8 * GORT_MAX_WIDE_CTAS, 64 * (size_t) ncta, cudaMemcpyDeviceToHost);
    cudaMemcpy(prev, ctx->d_timeline + (half ^ 1) * 8 * GORT_MAX_WIDE_CTAS, 64 * (size_t) ncta, cudaMemcpyDeviceToHost);
    unsigned long long t0 = ~0ull;
    for (int i = 0; i < ncta; i++) if (h[i * 8] < t0) t0 = h[i * 8];
    const char *nm[6] = {"entry", "leaf table done", "geometry complete", "first sun terms", "gate passed", "end"};
    fprintf(stderr, "%s timeline, call %d, %d CTAs, us since the first CTA entry of this call\n", kernel, ctx->dbg_timeline, ncta);
    {
        double mn = 1e30, mx = -1e30, sm = 0;
        for (int i = 0; i < ncta; i++) { double v = (double) ((long long) (prev[i * 8 + 5] - t0)) * 1e-3; if (v < mn) mn = v; if (v > mx) mx = v; sm += v; }
        fprintf(stderr, "  %-20s min %8.2f avg %8.2f max %8.2f\n", "previous call: end", mn, sm / ncta, mx);
    }
    for (int k = 0; k < 6; k++) {
        double mn = 1e30, mx = -1e30, sm = 0;
        for (int i = 0; i < ncta; i++) { double v = (double) ((long long) (h[i * 8 + k] - t0)) * 1e-3; if (v < mn) mn = v; if (v > mx) mx = v; sm += v; }
        fprintf(stderr, "  %-20s min %8.2f avg %8.2f max %8.2f\n", nm[k], mn, sm / ncta, mx);
    }
    double gw = 0, st = 0, run = 0;
    for (int i = 0; i < ncta; i++) { gw += (h[i * 8 + 4] - h[i * 8 + 3]) * 1e-3; st += (h[i * 8 + 3] - h[i * 8]) * 1e-3; run += (h[i * 8 + 5] - h[i * 8 + 4]) * 1e-3; }
    fprintf(stderr, "  per CTA: start-up %.2f us, gate wait %.2f us, store phase %.2f us\n", st / ncta, gw / ncta, run / ncta);
    free(h); free(prev);
}

// gort_kernel_stamps: in-kernel %globaltimer view of the most recent per-wavelength launch
int read_kernel_stamps(gort_ctx *ctx, double *span_us, double *startup_us, double *store_us, int *n_cta)
{
    if (!ctx->d_timeline || ctx->stamps_ncta <= 0) return set_error(ctx, GORT_ERR_INVALID, "gort_kernel_stamps: no stamped launch yet");
    cudaError_t e = cudaStreamSynchronize(ctx->stamps_stream);
    if (e != cudaSuccess) return check_cuda(ctx, e, "gort_kernel_stamps");
    const int n = ctx->stamps_ncta;
    unsigned long long *h = (unsigned long long *) malloc(64 * (size_t) n);
    if (!h) return set_error(ctx, GORT_ERR_NOMEM, "out of host memory");
    e = cudaMemcpy(h, ctx->d_timeline + ctx->stamps_half * 8 * GORT_MAX_WIDE_CTAS, 64 * (size_t) n, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { free(h); return check_cuda(ctx, e, "gort_kernel_stamps"); }
    unsigned long long first = ~0ull, last = 0;
    double st = 0, run = 0;
    for (int i = 0; i < n; i++) {
        if (h[i * 8] < first) first = h[i * 8];
        if (h[i * 8 + 5] > last) last = h[i * 8 + 5];
        st += (double) (h[i * 8 + 4] - h[i * 8]) * 1e-3;          // entry -> gate passed (first store follows)
        run += (double) (h[i * 8 + 5] - h[i * 8 + 4]) * 1e-3;     // gate passed -> all stores complete
    }
    free(h);
    if (span_us) *span_us = (double) (last - first) * 1e-3;
    if (startup_us) *startup_us = st / n;
    if (store_us) *store_us = run / n;
    if (n_cta) *n_cta = n;
    return GORT_OK;
}

// what launch_brdf hands to the per-wavelength launchers
struct BrdfPlan {
    long L;
    const double *rec;
    unsigned long long *flags;      // this call's flag array: geometry tiles, then table tiles
    bool pdl;                       // launch as a programmatic dependent of the geometry kernel
    bool gate;                      // overlap mode: wait per CTA for the previous launch's CTA of the same index
    const double *table;            // per-call (set, lambda) table for the wide kernel's TMA variants, or NULL
    int tab_ncol;
    long tab_flag_base;
};

// chunking of the wide kernel for a given variant: as few wavelength chunks as possible with <= pick threads per CTA
static void wide_chunking(int n_col, int lpt, int pick, int *n_chunks, int *threads)
{
    *n_chunks = (n_col + lpt * pick - 1) / (lpt * pick);
    int t = (n_col + *n_chunks * lpt - 1) / (*n_chunks * lpt);
    *threads = ((t + 31) / 32) * 32;
}

template <int LPT, bool SCOMP, int MINB, int TMAB, bool TAB = false>
static int launch_wide(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const BrdfPlan &pl, const double *structure,
                       const double *lut, const double *rleaf, const double *tleaf,
                       const double *rsoil, double *rsurf, double *scomp)
{
    const long L = pl.L;
    // columns written per row: the spectrum, plus -- when the caller's pitch leaves room -- the padding up to
    // the end of the row's last 128-byte line (16 doubles), so that no row ends in a partially written line
    const long pitch_ = sh.out_pitch > 0 ? sh.out_pitch : sh.n_wl;
    const int n_col = (int) (pitch_ % 16 == 0 ? ((long) (sh.n_wl + 15) / 16 * 16 < pitch_ ? (long) (sh.n_wl + 15) / 16 * 16 : pitch_) : sh.n_wl);
    // wavelength chunks: as few as possible with <= WIDE_PICK_THREADS threads per CTA, lanes spread evenly
    // block size cap: with the TMA row ring two CTAs must still fit an SM's shared memory
    const int pick = TMAB > 0 ? WIDE_PICK_THREADS_TMA : WIDE_PICK_THREADS;
    int n_chunks, threads;
    wide_chunking(n_col, LPT, pick, &n_chunks, &threads);
    WideArgs a;
    a.table = TAB ? pl.table : NULL; a.tab_ncol = pl.tab_ncol; a.tab_flag_base = pl.tab_flag_base;
    a.n_sets = sh.n_sets; a.n_geom = sh.n_geom; a.n_wl = sh.n_wl; a.spectra_per_set = sh.spectra_per_set;
    a.chunk = LPT * threads;
    a.n_col = n_col;
    a.pdl = pl.pdl ? 1 : 0;
    a.pitch = pitch_;
    a.structure = structure; a.lut = lut; a.rec = pl.rec; a.rleaf = rleaf; a.tleaf = tleaf; a.rsoil = rsoil;
    a.rsurf = rsurf; a.scomp = scomp;
    a.done = ctx->d_done; a.fault = ctx->d_done + GORT_MAX_WIDE_CTAS;
    a.tile_flags = pl.flags; a.call_no = ctx->call_no;
    constexpr int STAGE = WIDE_STAGE_LINES;
    constexpr int RINGW = SCOMP ? 5 : 1;                  // doubles per evaluation in the output ring
    const size_t smem = sizeof(double2) * 8 * STAGE + sizeof(unsigned) * 4
                      + sizeof(double) * (WIDE_NLEAF + 2 * TMAB * RINGW) * (size_t) a.chunk;
    auto kern = rsurf_wide_kernel<LPT, SCOMP, MINB, TMAB, TAB>;
    // occupancy of this (variant, block size) is looked up once per context
    int occ = 0;
    for (int i = 0; i < ctx->n_wide_plan; i++) {
        auto &wp = ctx->wide_plan[i];
        if (wp.key_lpt == LPT && wp.key_scomp == (int) SCOMP + 2 * TMAB + 16 * (int) TAB && wp.key_minb == MINB && wp.key_threads == threads) occ = wp.occ;
    }
    if (occ == 0) {
        // allow the largest chunk any block size can ask for, so that the attribute never shrinks
        const size_t smem_max = sizeof(double2) * 8 * STAGE + sizeof(unsigned) * 4
                              + sizeof(double) * (WIDE_NLEAF + 2 * TMAB * RINGW) * (size_t) LPT * (TMAB > 0 ? WIDE_PICK_THREADS_TMA : WIDE_MAX_THREADS);
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem_max);
        if (e != cudaSuccess) return check_cuda(ctx, e, "rsurf_wide_kernel shared memory");
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem);
        if (e != cudaSuccess || occ < 1) occ = 1;
        if (ctx->n_wide_plan < 8) {
            auto &wp = ctx->wide_plan[ctx->n_wide_plan++];
            wp.key_lpt = LPT; wp.key_scomp = (int) SCOMP + 2 * TMAB + 16 * (int) TAB; wp.key_minb = MINB; wp.key_threads = threads; wp.key_wl = sh.n_wl; wp.occ = occ;
        }
    }
    // one resident wave: grid.y contiguous line ranges so that n_chunks * grid.y ~ SMs * occupancy
    long nby = ((long) ctx->sm_count * occ) / n_chunks;
    if (nby < 1) nby = 1;
    if (nby > L) nby = L;
    a.lines_per_cta = (L + nby - 1) / nby;
    nby = (L + a.lines_per_cta - 1) / a.lines_per_cta;
    if ((long) n_chunks * nby > GORT_MAX_WIDE_CTAS) return set_error(ctx, GORT_ERR_INVALID, "gort_brdf: grid of %ld CTAs exceeds the pipeline's flag table", (long) n_chunks * nby);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned) n_chunks, (unsigned) nby);
    cfg.blockDim = dim3((unsigned) threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pl.pdl ? 1 : 0;
    // per-CTA gate: CTA k waits for CTA k of the previous launch when that launch had the same kernel, shape and
    // outputs (then CTA k wrote exactly the region this CTA k is about to write, and the grid is identical because
    // it is a function of the shape only).  launch_brdf lets a call overlap the previous one only in that case;
    // otherwise stream order serialises the two and there is nothing to wait for.
    a.epoch = ++ctx->epoch;
    a.tl = timeline_half(ctx, a.epoch);
    a.wait_target = pl.gate ? a.epoch - 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a);
    if (a.tl) { ctx->stamps_ncta = n_chunks * (int) nby; ctx->stamps_half = (int) (a.epoch & 1); ctx->stamps_stream = s; }
    if (a.tl) timeline_report(ctx, s, n_chunks * (int) nby, (int) (a.epoch & 1), "rsurf_wide_kernel");
    return check_cuda(ctx, e, "rsurf_wide_kernel launch");
}

// ---- full-spectrum kernel (gort_rsurf_rows.cuh) -------------------------------------------------------------------
struct RowsShape { bool ok; int n_col, ncolt, threads, tiles_per_set; size_t smem, tab_doubles; long lines_per_cta, grid; };

static RowsShape rows_shape(const gort_ctx *ctx, const gort_shape &sh, long L, const double *rsurf, const double *scomp)
{
    RowsShape r = {};
    const long pitch = sh.out_pitch > 0 ? sh.out_pitch : sh.n_wl;
    // EXPERIMENTAL, off unless GORT_ROWS=1: measured on C2 the kernel is correct (same bits as the chunked kernel) but
    // slower -- 50 us isolated against 43.6 us: with its 153 KB table a single CTA fits an SM, so nothing overlaps its
    // start-up (table load 3.6 us) and the (sun, lambda) terms of every new run (2 us each); see DESIGN.md 4.1
    if (scomp || !ctx->dbg_rows_on || ctx->dbg_no_tma || pitch % 16 != 0 || ((size_t) rsurf & 15) != 0) return r;
    const long padded = (long) (sh.n_wl + 15) / 16 * 16;
    r.n_col = (int) (padded < pitch ? padded : pitch);
    r.threads = ((r.n_col + 3) / 4 + 31) / 32 * 32;
    r.ncolt = 4 * r.threads;
    if (r.threads > ROWS_MAX_THREADS || r.threads < 256) return r;      // 1024 .. 2176 columns
    if (L < 2L * ctx->sm_count) return r;                               // few lines: the chunked kernel spreads them better
    r.tab_doubles = (size_t) sh.n_sets * ROWS_NLEAF * r.ncolt;
    if (r.tab_doubles * sizeof(double) > ((size_t) 1 << 30)) return r;
    r.tiles_per_set = r.ncolt / ROWS_TAB_TILE;
    r.smem = sizeof(double) * (size_t) (ROWS_NLEAF + ROWS_NBUF) * r.ncolt + 128 * (size_t) ROWS_STAGE_LINES + 8 * (1 + 2 * ROWS_NBUF);
    long nct = ctx->sm_count < L ? ctx->sm_count : L;
    r.lines_per_cta = (L + nct - 1) / nct;
    r.grid = (L + r.lines_per_cta - 1) / r.lines_per_cta;
    r.ok = true;
    return r;
}

static int launch_rows(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const BrdfPlan &pl, const RowsShape &rs,
                       const double *lut, const double *table, long tab_flag_base, double *rsurf)
{
    if (!ctx->rows_attr_set) {
        const size_t smem_max = sizeof(double) * (size_t) (ROWS_NLEAF + ROWS_NBUF) * 4 * ROWS_MAX_THREADS + 128 * (size_t) ROWS_STAGE_LINES + 8 * (1 + 2 * ROWS_NBUF);
        cudaError_t e = cudaFuncSetAttribute(rsurf_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem_max);
        if (e != cudaSuccess) return check_cuda(ctx, e, "rsurf_rows_kernel shared memory");
        ctx->rows_attr_set = 1;
    }
    RowsArgs a;
    a.n_sets = sh.n_sets; a.n_geom = sh.n_geom; a.n_wl = sh.n_wl; a.spectra_per_set = sh.spectra_per_set;
    a.n_col = rs.n_col; a.ncolt = rs.ncolt;
    a.pdl = pl.pdl ? 1 : 0;
    a.dbg = ctx->dbg_rows;
    a.flags = pl.flags; a.tab_flag_base = tab_flag_base; a.call_no = ctx->call_no;
    a.fault = ctx->d_done + GORT_MAX_WIDE_CTAS; a.done = ctx->d_done;
    a.pitch = sh.out_pitch > 0 ? sh.out_pitch : sh.n_wl;
    a.lines_per_cta = rs.lines_per_cta;
    a.lut = lut; a.rec = pl.rec; a.table = table; a.rsurf = rsurf;
    a.epoch = ++ctx->epoch;
    a.tl = timeline_half(ctx, a.epoch);
    a.wait_target = pl.gate ? a.epoch - 1 : 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned) rs.grid);
    cfg.blockDim = dim3((unsigned) rs.threads + 32);      // compute warps + the store warp
    cfg.dynamicSmemBytes = rs.smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pl.pdl ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, rsurf_rows_kernel, a);
    if (a.tl) timeline_report(ctx, s, (int) rs.grid, (int) (a.epoch & 1), "rsurf_rows_kernel");
    return check_cuda(ctx, e, "rsurf_rows_kernel launch");
}

static bool ranges_overlap(const void *p, const char *lo, const char *hi)
{
    return p && lo && (const char *) p >= lo && (const char *) p < hi;
}

// grow-only flag array of one record buffer; new entries are zeroed ON THE LAUNCH STREAM, ahead of the kernels that
// publish and poll them
static int ensure_flags(gort_ctx *ctx, cudaStream_t s, int which, size_t n)
{
    if (n <= ctx->flag_cap[which]) return GORT_OK;
    cudaError_t e = cudaDeviceSynchronize();                      // the old array may still be polled by enqueued work
    if (e != cudaSuccess) return check_cuda(ctx, e, "pipeline flags: synchronize");
    if (ctx->d_flags[which]) { e = cudaFree(ctx->d_flags[which]); if (e != cudaSuccess) return check_cuda(ctx, e, "pipeline flags: cudaFree"); }
    ctx->d_flags[which] = NULL; ctx->flag_cap[which] = 0;
    const size_t want = n + n / 4 + 1024;
    e = cudaMalloc((void **) &ctx->d_flags[which], sizeof(unsigned long long) * want);
    if (e != cudaSuccess) return set_error(ctx, GORT_ERR_NOMEM, "cudaMalloc of the pipeline flags failed: %s", cudaGetErrorString(e));
    e = cudaMemsetAsync(ctx->d_flags[which], 0, sizeof(unsigned long long) * want, s);
    if (e != cudaSuccess) return check_cuda(ctx, e, "pipeline flags: cudaMemsetAsync");
    ctx->flag_cap[which] = want;
    return GORT_OK;
}

int launch_brdf(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const double *structure,
                const double *lut, const double *angles, const double *rleaf, const double *tleaf,
                const double *rsoil, double *rsurf, double *scomp, double *kprop)
{
    if (sh.n_sets <= 0 || sh.n_geom <= 0 || sh.n_wl <= 0)
        return set_error(ctx, GORT_ERR_INVALID, "gort_brdf: n_sets, n_geom and n_wl must be positive");
    const long L = (long) sh.n_sets * sh.n_geom;
    const long pitch = sh.out_pitch > 0 ? sh.out_pitch : sh.n_wl;
    if (pitch < sh.n_wl) return set_error(ctx, GORT_ERR_INVALID, "gort_brdf: out_pitch smaller than n_wl");
    // every path stores a { C, G, T, Z } quadruple as one vector: double4 in rsurf_flat_kernel, double2 pairs or bulk
    // copies in the wide kernel
    if (((size_t) scomp & 31) != 0) return set_error(ctx, GORT_ERR_INVALID, "gort_brdf: scomp must be 32-byte aligned");
    const bool use_pdl = !ctx->dbg_no_pdl;
    // a call on another stream than the previous one has been ordered after it by the entry point (order_after_previous),
    // which also ended the previous call's claim to overlap
    ctx->call_no++;
    // line records, the (set, lambda) table and the ready flags are double-buffered by call parity: this call's
    // geometry kernel may run while the previous call's per-wavelength kernel still reads its own
    ctx->rec_idx ^= 1;
    const int bi = ctx->rec_idx;
    const RowsShape rs = sh.n_wl >= 64 ? rows_shape(ctx, sh, L, rsurf, scomp) : RowsShape{};
    const size_t geom_tiles = (size_t) ((L + 31) / 32);
    // EXPERIMENTAL, off unless GORT_WIDE_TABLE=1: the wide kernel's TMA variants can take their (set, lambda) table from the
    // geometry kernel's spare CTAs instead of computing it per CTA.  Measured on C2: 45.1 us per launch against 43.8 us,
    // 41.1 us per overlapped step against 36.6 us -- the per-CTA computation runs under the previous CTA's stores for free,
    // the table copy competes with them for L2 (DESIGN.md 4.1)
    int wt_ncol = 0;
    if (ctx->dbg_table_on && !rs.ok && sh.n_wl >= 64 && !ctx->dbg_no_tma && pitch % 16 == 0 && ((size_t) rsurf & 15) == 0 && ((size_t) scomp & 15) == 0) {
        const long padded = (long) (sh.n_wl + 15) / 16 * 16;
        const int n_col = (int) (padded < pitch ? padded : pitch);
        int nc, thr;
        wide_chunking(n_col, scomp ? 2 : 4, WIDE_PICK_THREADS_TMA, &nc, &thr);
        const int chunk = (scomp ? 2 : 4) * thr;
        if (chunk % 128 == 0 && (size_t) sh.n_sets * WIDE_NLEAF * nc * chunk * sizeof(double) <= ((size_t) 256 << 20)) wt_ncol = nc * chunk;
    }
    const int tab_ncol = rs.ok ? rs.ncolt : wt_ncol;
    const size_t tab_tiles = tab_ncol ? (size_t) sh.n_sets * (tab_ncol / ROWS_TAB_TILE) : 0;
    {
        int rc = ensure_flags(ctx, s, bi, geom_tiles + tab_tiles);
        if (rc != GORT_OK) return rc;
    }
    double *rec = (double *) rec_buffer(ctx, bi, sizeof(double) * GORT_REC_STRIDE * (size_t) L);
    if (!rec) return GORT_ERR_NOMEM;
    double *table = NULL;
    if (tab_ncol) {
        table = (double *) tab_buffer(ctx, bi, sizeof(double) * (size_t) sh.n_sets * ROWS_NLEAF * tab_ncol);
        if (!table) return GORT_ERR_NOMEM;
    }
    cudaEvent_t *ev = (ctx->prof_ev && ctx->prof_n < ctx->prof_cap) ? ctx->prof_ev + 3 * ctx->prof_n : NULL;
    if (ev) { cudaError_t e = cudaEventRecord(ev[0], s); if (e != cudaSuccess) return check_cuda(ctx, e, "cudaEventRecord"); }
    // Cross-call overlap (gort_set_overlap, off by default): if the previous operation this context put on the stream
    // was a per-wavelength kernel of the same kind, shape and outputs (it releases its dependents once it is past its
    // start-up), this call's geometry kernel is launched as a programmatic dependent that never waits: it reads only
    // this call's inputs and writes only the other record / table / flag buffers and kprop.  Not done if an input of
    // this call aliases an output of the previous call, or kprop aliases anything the previous call still reads or
    // writes.  The caller's side of the contract (nothing else enqueued on the stream in between that writes an
    // input of this call) is stated in include/gort_b200.h.
    bool alias = false;
    {
        const void *in[7] = {structure, lut, angles, rleaf, tleaf, rsoil, kprop};
        for (int k = 0; k < 7; k++) for (int r = 0; r < 3; r++) alias |= ranges_overlap(in[k], ctx->last_out_lo[r], ctx->last_out_hi[r]);
    }
    const unsigned long long sig[8] = {(unsigned long long) sh.n_sets, (unsigned long long) sh.n_geom, (unsigned long long) sh.n_wl,
                                       (unsigned long long) pitch, (unsigned long long) (size_t) rsurf, (unsigned long long) (size_t) scomp,
                                       (unsigned long long) (rs.ok ? 1 : 0), (unsigned long long) (size_t) kprop};
    bool same = ctx->last_was_wide != 0;
    for (int k = 0; k < 8; k++) same &= sig[k] == ctx->last_sig[k];
    for (int k = 0; k < 8; k++) ctx->last_sig[k] = sig[k];
    const bool early_geom = ctx->overlap && use_pdl && !ev && !ctx->stamps_on && same && !alias && sh.n_wl >= 64;
    {
        // the per-wavelength kernel that follows needs a large shared-memory carve-out; an SM only changes its
        // carve-out when idle, so ask for the same one here or the dependent kernel's CTAs could not join this
        // kernel's CTAs on an SM (measured: without it they entered only as geom_kernel's CTAs left)
        if (!ctx->geom_carveout_set) {            // per device, so per context
            cudaError_t e = cudaFuncSetAttribute(geom_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(geom_lines_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            if (e != cudaSuccess) return check_cuda(ctx, e, "geometry kernel carve-out");
            ctx->geom_carveout_set = 1;
        }
        TableJob tj = {};
        if (tab_ncol) {
            tj.n_tiles = (int) tab_tiles; tj.n_wl = sh.n_wl; tj.spectra_per_set = sh.spectra_per_set; tj.ncolt = tab_ncol;
            tj.rleaf = rleaf; tj.tleaf = tleaf; tj.rsoil = rsoil; tj.table = table;
            tj.flags = ctx->d_flags[bi] + geom_tiles;
        }
        cudaLaunchConfig_t cfg = {};
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = early_geom ? 1 : 0;
        // enough lines to fill the GPU several times over: one thread per line (see geom_lines_kernel)
        const bool by_line = L >= 64L * 4 * ctx->sm_count;
        cudaError_t e;
        if (by_line) {
            cfg.gridDim = dim3((unsigned) ((L + 127) / 128 + tab_tiles));
            cfg.blockDim = dim3(128);
            e = cudaLaunchKernelEx(&cfg, geom_lines_kernel, sh.n_sets, sh.n_geom, sh.geom_per_set, sh.opt,
                                   structure, lut, angles, rec, kprop, ctx->d_flags[bi], ctx->call_no, tj);
        } else {
            cfg.gridDim = dim3((unsigned) ((L + 31) / 32 + tab_tiles));
            cfg.blockDim = dim3(32 * GEOM_ROLES);
            e = cudaLaunchKernelEx(&cfg, geom_kernel, sh.n_sets, sh.n_geom, sh.geom_per_set, sh.opt,
                                   structure, lut, angles, rec, kprop, ctx->d_flags[bi], ctx->call_no, tj);
        }
        if (e != cudaSuccess) return check_cuda(ctx, e, "geom_kernel launch");
        ctx->launches++;
    }
    if (ev) { cudaError_t e = cudaEventRecord(ev[1], s); if (e != cudaSuccess) return check_cuda(ctx, e, "cudaEventRecord"); }
    if (sh.n_wl >= 64) {
        // programmatic dependent launch: the kernel's prologue overlaps geom_kernel.  Off while per-kernel events
        // are being recorded (an event between the two launches would time the overlap)
        BrdfPlan pl;
        pl.L = L; pl.rec = rec; pl.flags = ctx->d_flags[bi];
        pl.pdl = use_pdl && !ev && !ctx->stamps_on;      // events or stamps: plain stream order, so that a launch is separable
        pl.gate = early_geom;
        pl.table = rs.ok ? NULL : table; pl.tab_ncol = tab_ncol; pl.tab_flag_base = (long) geom_tiles;
        int rc;
        if (rs.ok) {
            // full spectrum, aligned rows: one persistent CTA per SM writes whole rows (gort_rsurf_rows.cuh)
            rc = launch_rows(ctx, s, sh, pl, rs, lut, table, (long) geom_tiles, rsurf);
        } else {
            // wavelengths per thread: the value in {4, 3, 2} whose chunking wastes the fewest columns (ties: fewer
            // chunks, then larger LPT)
            int lpt = 4;
            {
                const long n_col = pitch % 16 == 0 ? ((long) (sh.n_wl + 15) / 16 * 16 < pitch ? (long) (sh.n_wl + 15) / 16 * 16 : pitch) : sh.n_wl;
                long best_waste = -1; int best_chunks = 0;
                for (int cand = 4; cand >= 2; cand--) {
                    const long nc = (n_col + cand * WIDE_PICK_THREADS - 1) / (cand * WIDE_PICK_THREADS);
                    long thr = (n_col + nc * cand - 1) / (nc * cand);
                    thr = (thr + 31) / 32 * 32;
                    const long waste = nc * cand * thr - n_col;
                    if (best_waste < 0 || waste < best_waste || (waste == best_waste && nc < best_chunks)) { best_waste = waste; best_chunks = (int) nc; lpt = cand; }
                }
            }
#define WIDE_ARGS ctx, s, sh, pl, structure, lut, rleaf, tleaf, rsoil, rsurf, scomp
            // Output path: rows through shared memory and TMA bulk stores (3 rows per CTA barrier, LPT = 4) when the
            // rows are 128-byte aligned, else per-thread stores
            const bool tma = !ctx->dbg_no_tma && pitch % 16 == 0 && ((size_t) rsurf & 15) == 0 && ((size_t) scomp & 15) == 0;
            const bool tab = pl.table != NULL;
            if (scomp && tma && tab) rc = launch_wide<2, true, 2, WIDE_TMA_ROWS_SCOMP, true>(WIDE_ARGS);
            else if (scomp && tma) rc = launch_wide<2, true, 2, WIDE_TMA_ROWS_SCOMP>(WIDE_ARGS);
            else if (scomp) rc = launch_wide<2, true, 2, 0>(WIDE_ARGS);
            else if (tma && tab) rc = launch_wide<4, false, 2, WIDE_TMA_ROWS, true>(WIDE_ARGS);
            else if (tma) rc = launch_wide<4, false, 2, WIDE_TMA_ROWS>(WIDE_ARGS);
            else if (lpt == 4) rc = launch_wide<4, false, 2, 0>(WIDE_ARGS);
            else if (lpt == 3) rc = launch_wide<3, false, 2, 0>(WIDE_ARGS);
            else rc = launch_wide<2, false, 2, 0>(WIDE_ARGS);
#undef WIDE_ARGS
        }
        if (rc != GORT_OK) return rc;
    } else {
        const int threads = 128;
        long total = L * sh.n_wl;
        long blocks = (total + threads - 1) / threads;
        rsurf_flat_kernel<<<(unsigned) blocks, threads, 0, s>>>(sh.n_sets, sh.n_geom, sh.n_wl, sh.spectra_per_set, pitch,
                                                                structure, lut, rec, rleaf, tleaf, rsoil, rsurf, scomp);
    }
    ctx->launches++;
    if (ev) { cudaError_t e = cudaEventRecord(ev[2], s); if (e != cudaSuccess) return check_cuda(ctx, e, "cudaEventRecord"); ctx->prof_n++; }
    ctx->last_was_wide = (sh.n_wl >= 64) && !ev;
    ctx->last_out_lo[0] = (const char *) rsurf; ctx->last_out_hi[0] = (const char *) (rsurf + (size_t) L * pitch);
    ctx->last_out_lo[1] = (const char *) scomp; ctx->last_out_hi[1] = scomp ? (const char *) (scomp + 4 * (size_t) L * pitch) : NULL;
    ctx->last_out_lo[2] = (const char *) kprop; ctx->last_out_hi[2] = kprop ? (const char *) (kprop + 4 * (size_t) L) : NULL;
    return check_cuda(ctx, cudaGetLastError(), "gort_brdf launch");
}

// ------------------------------------------------------------------------------------------------
// Energy balance (gortt_energy / gortt_albedo, gortt_albedo.c:7-138).  One CTA of 512 threads per (set, sun line).
//
// The reference evaluates gortt_rsurf at 32 x 16 Gauss-Legendre nodes of the view hemisphere for every
// wavelength and sums rsurf * weights (:89-136): 512 x W evaluations per sun angle.  All nodes share the sun, so
// in the regrouped form of the view loop (gort_rsurf_wide.cuh)
//        rsurf(node, lambda) = cA(node) A(l) + Kc(node) PDF(l) + cG(node) G(l) + cZ(node) Z(l) + Kt(node) T(l)
// the five (sun, lambda) terms are common to all nodes and the quadrature is LINEAR in the node coefficients:
//        albedo(l) = [S cA] A(l) + [S Kc] PDF(l) + [S cG] G(l) + [S cZ] Z(l) + [S Kt] T(l),   S = sum over nodes
//                                                                                  with weight w_i w_j |mu_j|.
// Two kernels:
//   energy_zenith_kernel  one thread per (sun line, view-zenith node): everything of the geometry record that does
//                         not depend on the azimuth -- primed trig of both zeniths, the raa = 0 and raa = pi passes
//                         of gortt_kc, the crown terms, the exp terms, beta, LUT interpolation, the zenith part of
//                         the hotspot.  The reference recomputes all of it at each of the 32 azimuth nodes.
//   energy_kernel         one CTA of 512 threads per (set, sun line): thread n -> node (azimuth i = n % 32,
//                         zenith j = 16 + n / 32): the pass at its own relative azimuth and the pair part of the
//                         hotspot, the weighted coefficients, their sums by warp shuffle + a fixed shared-memory
//                         tree; then one thread per wavelength: the (set, lambda) and (sun, lambda) terms once,
//                         5 FMAs, and the energy balance of gortt_albedo.c:37-52.
// Work per (set, sun) drops from 512 x W view evaluations + 512 full geometry records to 16 zenith records +
// 512 azimuth passes + W spectral evaluations; the sums run in a different order than the reference's nested
// loops (differences ~1e-16 relative).
#define GORT_EN_THREADS 512
#define GORT_EN_NZ (GORT_NQUAD / 2)       // view-zenith nodes (mu > 0)
#define GORT_EN_ZREC 32                   // doubles per zenith record

// zenith record layout (doubles)
enum { ZR_VZA = 0, ZR_VZA_P, ZR_SZA_P, ZR_TS, ZR_TV, ZR_SECS, ZR_SECV, ZR_CS, ZR_CV, ZR_SS, ZR_SV,
       ZR_MV, ZR_THETA_MI, ZR_GAMMA_V, ZR_F0F0, ZR_F180F180, ZR_EV, ZR_ES, ZR_T0, ZR_BETA,
       ZR_PN0S, ZR_PES, ZR_PEV, ZR_SSZ, ZR_CSZ, ZR_SVZ, ZR_CVZ, ZR_LSZA, ZR_LVZA, ZR_FD, ZR_X, ZR_END };
static_assert(ZR_END <= GORT_EN_ZREC, "zenith record too small");

__global__ void __launch_bounds__(128)
energy_zenith_kernel(int n_sets, int n_geom, int geom_per_set, gort_options opt,
                     const double* __restrict__ structure, const double* __restrict__ lut,
                     const double* __restrict__ angles, const double* __restrict__ gl, double* __restrict__ zrec)
{
    const long L = (long) n_sets * n_geom;
    const long item = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= L * GORT_EN_NZ) return;
    const long line = item / GORT_EN_NZ;
    const int jj = (int) (item - line * GORT_EN_NZ);
    const int m = (int) (line / n_geom);
    const long a = geom_per_set ? line : (line - (long) m * n_geom);
    const long na = geom_per_set ? L : n_geom;
    const Canopy c = canopy_load(structure, n_sets, m, lut);
    const double* lut_m = lut + (size_t) m * GORT_LUT_STRIDE;
    const Line g = line_from_degrees(angles[0 * na + a], angles[1 * na + a], angles[2 * na + a], angles[3 * na + a]);
    const double xr = 0.5 * (1. + 1.), xm = 0.5 * (1. - 1.);                     // gortt_albedo.c:82-83
    const double x = xm + xr * gl[GORT_NQUAD / 2 + jj];                          // :103
    const double vza = acos(x);                                                  // :105
    const double fd = opt.use_fd ? opt.fd : cos(g.sza) / (cos(g.sza) + 0.09);    // gortt.c:290-291
    const Primed P = primed_trig(c, vza, g.sza);
    const CrownLite s = crown_lite(c, P.t);
    const bool vgs = fabs(vza) > fabs(g.sza);
    const Pass a0 = kc_pass(c, P, s, vgs, 0.0, 1.0, 0.0);                        // gortt_brdf.c:143-146
    const Pass a180 = kc_pass(c, P, s, vgs, GORT_PI, -1.0, GORT_SIN_PI);         // :147-150
    const Tail tl = tail_terms(c, P, opt);
    double pn0_s, pe_s, pn0_v, pe_v;
    zenith_lerp(lut_m, g.sza, pn0_s, pe_s);                                      // gortt.c:872-915
    zenith_lerp(lut_m, vza, pn0_v, pe_v);
    double ssz, csz, svz, cvz;
    sincos(g.sza, &ssz, &csz);
    sincos(vza, &svz, &cvz);
    double* z = zrec + (size_t) item * GORT_EN_ZREC;
    z[ZR_VZA] = vza; z[ZR_VZA_P] = P.vza_p; z[ZR_SZA_P] = P.sza_p;
    z[ZR_TS] = P.t.ts; z[ZR_TV] = P.t.tv; z[ZR_SECS] = P.t.secs; z[ZR_SECV] = P.t.secv;
    z[ZR_CS] = P.t.cs; z[ZR_CV] = P.t.cv; z[ZR_SS] = P.t.ss; z[ZR_SV] = P.t.sv;
    z[ZR_MV] = s.Mv; z[ZR_THETA_MI] = s.theta_Mi; z[ZR_GAMMA_V] = s.Gamma_v;
    z[ZR_F0F0] = a0.f * a0.F; z[ZR_F180F180] = a180.f * a180.F;
    z[ZR_EV] = tl.e_v; z[ZR_ES] = tl.e_s; z[ZR_T0] = tl.t0; z[ZR_BETA] = tl.beta;
    z[ZR_PN0S] = pn0_s; z[ZR_PES] = pe_s; z[ZR_PEV] = pe_v;
    z[ZR_SSZ] = ssz; z[ZR_CSZ] = csz; z[ZR_SVZ] = svz; z[ZR_CVZ] = cvz;
    z[ZR_LSZA] = -log(pe_s) / c.kfavd;                                           // gortt_brdf.c:659-660
    z[ZR_LVZA] = -log(pe_v) / c.kfavd;
    z[ZR_FD] = fd; z[ZR_X] = x;
}

__global__ void __launch_bounds__(GORT_EN_THREADS, 2)
energy_kernel(int n_sets, int n_geom, int n_wl, int geom_per_set, int spectra_per_set, gort_options opt,
              const double* __restrict__ structure, const double* __restrict__ lut,
              const double* __restrict__ angles, const double* __restrict__ gl /*[2][32]*/,
              const double* __restrict__ zrec,
              const double* __restrict__ rleaf, const double* __restrict__ tleaf,
              const double* __restrict__ rsoil,
              double* __restrict__ albedo, double* __restrict__ favegt, double* __restrict__ fasoil)
{
    __shared__ double part[5][GORT_EN_THREADS / 32];    // per-warp partial sums of the weighted coefficients
    __shared__ double coef[5];
    __shared__ double sunv[6];                          // fd mus t0 tp0 pe_s pn0_s

    const long L = (long) n_sets * n_geom;
    const long line = blockIdx.x;
    const int m = (int) (line / n_geom);
    const long a = geom_per_set ? line : (line - (long) m * n_geom);
    const long na = geom_per_set ? L : n_geom;
    const int tid = threadIdx.x;
    const Canopy c = canopy_load(structure, n_sets, m, lut);
    double fd;
    {
        const int i = tid & 31, jj = tid >> 5;
        const double* z = zrec + ((size_t) line * GORT_EN_NZ + jj) * GORT_EN_ZREC;      // same record for the whole warp
        const double xr = 0.5 * (1. + 1.);
        const double ym = 0.5 * (2. * GORT_PI - 0.), yr = 0.5 * (2. * GORT_PI + 0.);  // gortt_albedo.c:84-85
        // azimuth of this node: saa after the reference's normalisation (gortt.c:253-274 via line_from_degrees)
        const Line g = line_from_degrees(angles[0 * na + a], angles[1 * na + a], angles[2 * na + a], angles[3 * na + a]);
        double y = ym + yr * gl[i];                                              // :91
        double vaa = y;
        for (int it = 0; it < 8 && vaa > 2 * GORT_PI; it++) vaa -= 2 * GORT_PI;  // :96
        const double raa = fold_raa(g.saa - vaa);                                // :97-98
        double sr, cr;
        sincos(raa, &sr, &cr);
        Primed P;
        P.vza_p = z[ZR_VZA_P]; P.sza_p = z[ZR_SZA_P];
        P.t.ts = z[ZR_TS]; P.t.tv = z[ZR_TV]; P.t.secs = z[ZR_SECS]; P.t.secv = z[ZR_SECV];
        P.t.cs = z[ZR_CS]; P.t.cv = z[ZR_CV]; P.t.ss = z[ZR_SS]; P.t.sv = z[ZR_SV];
        CrownLite s;
        s.Mv = z[ZR_MV]; s.theta_Mi = z[ZR_THETA_MI]; s.Gamma_v = z[ZR_GAMMA_V];
        const double vza = z[ZR_VZA];
        const bool vgs = fabs(vza) > fabs(g.sza);
        const Pass pa = kc_pass(c, P, s, vgs, raa, cr, sr);
        Tail tl;
        tl.e_v = z[ZR_EV]; tl.e_s = z[ZR_ES]; tl.t0 = z[ZR_T0]; tl.beta = z[ZR_BETA];
        // pair part of gortt_kuusk, gortt_brdf.c:650-702
        Hot h;
        h.pn0_s = z[ZR_PN0S]; h.pe_s = z[ZR_PES];
        {
            const double cos_xi = z[ZR_CSZ] * z[ZR_CVZ] + z[ZR_SSZ] * z[ZR_SVZ] * cr;
            const double lsza = z[ZR_LSZA], lvza = z[ZR_LVZA];
            const double arg = lsza * lsza + lvza * lvza - 2. * lsza * lvza * cos_xi;
            double t1, t2;
            if (arg > 0.0) {
                double lsv = sqrt(arg);
                t2 = (1.0 - exp(-lsv / c.r)) / (lsv / c.r);
            } else {
                t2 = 1.0;
            }
            if ((lsza * lvza) > 0.0) t1 = sqrt(lsza * lvza);
            else t1 = 0.0;
            const double H = exp(c.kfavd * t1 * t2);
            h.kuusk = h.pe_s * z[ZR_PEV] * H;
        }
        fd = z[ZR_FD];
        const GeomRec r = geom_combine(c, P, pa, z[ZR_F0F0], z[ZR_F180F180], tl, h, raa, fd);
        const double x = z[ZR_X];
        const double wn = (gl[GORT_NQUAD + GORT_NQUAD / 2 + jj] * fabs(x) * xr) * (gl[GORT_NQUAD + i] * yr);   // :128-129, :132-133
        double v[5] = {wn * r.cA, wn * r.Kc, wn * r.cG, wn * r.cZ, wn * r.Kt};
#pragma unroll
        for (int k = 0; k < 5; k++) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], off);
            if ((tid & 31) == 0) part[k][tid >> 5] = v[k];
        }
        if (tid == 0) {
            sunv[0] = r.fd; sunv[1] = r.mus; sunv[2] = r.t0; sunv[3] = r.tp0; sunv[4] = r.pe_s; sunv[5] = r.pn0_s;
        }
    }
    __syncthreads();
    if (tid < 5) {
        double sum = 0.0;
        for (int w = 0; w < GORT_EN_THREADS / 32; w++) sum += part[tid][w];
        coef[tid] = sum;
    }
    __syncthreads();
    const double mus = sunv[1], t0 = sunv[2], tp0 = sunv[3], pe = sunv[4], Pn0 = sunv[5];
    const double CA = coef[0], CP = coef[1], CG = coef[2], CZ = coef[3], CT = coef[4];
    const size_t sb = spectra_per_set ? (size_t) m * n_wl : 0;
    for (int w = tid; w < n_wl; w += GORT_EN_THREADS) {
        const double rs = rsoil[sb + w];
        const LeafTerms Lf = leaf_terms(c, rleaf[sb + w], tleaf[sb + w], rs);
        const SunTerms S = sun_terms(c, Lf, fd, mus, t0, tp0, pe);
        const double sum_y = fma(CA, Lf.A, fma(CP, S.PDF, fma(CG, S.G, fma(CZ, S.Z, CT * S.T))));
        const size_t o = (size_t) line * n_wl + w;
        const double alb = sum_y / GORT_PI;                                      // :136
        const double Fu2 = S.G * Pn0 + S.Z * (1. - Pn0);                         // gortt_albedo.c:48
        const double Fd2 = Pn0 + S.Z * (1. - Pn0) / rs;                          // :49
        albedo[o] = alb;
        favegt[o] = 1. - alb - Fd2 + Fu2;                                        // :51
        fasoil[o] = Fd2 - Fu2;                                                   // :52
    }
}

int launch_energy(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const double *structure,
                  const double *lut, const double *angles, const double *rleaf, const double *tleaf,
                  const double *rsoil, double *albedo, double *favegt, double *fasoil)
{
    if (sh.n_sets <= 0 || sh.n_geom <= 0 || sh.n_wl <= 0)
        return set_error(ctx, GORT_ERR_INVALID, "gort_energy: n_sets, n_geom and n_wl must be positive");
    const long L = (long) sh.n_sets * sh.n_geom;
    note_other_work(ctx);
    double *zrec = (double *) workspace(ctx, sizeof(double) * GORT_EN_ZREC * GORT_EN_NZ * (size_t) L);
    if (!zrec) return GORT_ERR_NOMEM;
    {
        const long items = L * GORT_EN_NZ;
        energy_zenith_kernel<<<(unsigned) ((items + 127) / 128), 128, 0, s>>>(sh.n_sets, sh.n_geom, sh.geom_per_set, sh.opt, structure,
                                                                             lut, angles, ctx->d_gauleg, zrec);
        ctx->launches++;
    }
    energy_kernel<<<(unsigned) L, GORT_EN_THREADS, 0, s>>>(sh.n_sets, sh.n_geom, sh.n_wl, sh.geom_per_set,
                                                           sh.spectra_per_set, sh.opt, structure, lut, angles,
                                                           ctx->d_gauleg, zrec, rleaf, tleaf, rsoil, albedo, favegt, fasoil);
    ctx->launches++;
    return check_cuda(ctx, cudaGetLastError(), "gort_energy launch");
}

// ------------------------------------------------------------------------------------------------
// Finite-difference Jacobian helpers (gort_jacobian_batch): scale one structure row, form the difference quotient.
__global__ void __launch_bounds__(256)
jac_perturb_kernel(int n_sets, int row, double factor, const double* __restrict__ st_in, double* __restrict__ st_out)
{
    const long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= 6L * n_sets) return;
    const int r = (int) (e / n_sets);
    st_out[e] = r == row ? st_in[e] * factor : st_in[e];
}

// jac = (fp - fm) / (2 h p) per member; lai != 0: p = LAI at fixed geometry, (fp - fm) / (2 h LAI) with LAI = favd lambda pi r^2 b 4/3
__global__ void __launch_bounds__(256)
jac_diff_kernel(int n_sets, long per_set, int row, int lai, double h, const double* __restrict__ st,
                const double* __restrict__ fp, const double* __restrict__ fm, double* __restrict__ jac)
{
    const long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= per_set * n_sets) return;
    const int m = (int) (e / per_set);
    const size_t N = (size_t) n_sets;
    double p = st[(size_t) row * N + m];
    if (lai) p = st[5 * N + m] * (st[0 * N + m] * st[1 * N + m] * st[1 * N + m] * GORT_PI * st[2 * N + m] * 4.0) / 3.0;   // gortt.c:1129 inverted
    jac[e] = (fp[e] - fm[e]) / (2.0 * h * p);
}

int launch_jac_perturb(gort_ctx *ctx, cudaStream_t s, int n_sets, int row, double factor, const double *st_in, double *st_out)
{
    note_other_work(ctx);
    jac_perturb_kernel<<<(unsigned) ((6L * n_sets + 255) / 256), 256, 0, s>>>(n_sets, row, factor, st_in, st_out);
    ctx->launches++;
    return check_cuda(ctx, cudaGetLastError(), "jac_perturb_kernel launch");
}

int launch_jac_diff(gort_ctx *ctx, cudaStream_t s, int n_sets, long per_set, int row, int lai, double h, const double *st,
                    const double *fp, const double *fm, double *jac)
{
    note_other_work(ctx);
    jac_diff_kernel<<<(unsigned) ((per_set * n_sets + 255) / 256), 256, 0, s>>>(n_sets, per_set, row, lai, h, st, fp, fm, jac);
    ctx->launches++;
    return check_cuda(ctx, cudaGetLastError(), "jac_diff_kernel launch");
}

// ------------------------------------------------------------------------------------------------
// gauleg, gortt_albedo.c:141-199, n = 32 on (-1, 1).  One thread per root.
__global__ void gauleg_kernel(double* __restrict__ out)
{
    const int n = GORT_NQUAD;
    const double x1 = -1., x2 = 1.;
    int i = threadIdx.x;
    int mm = (n + 1) / 2;
    if (i >= mm) return;
    double xm = 0.5 * (x2 + x1), xl = 0.5 * (x2 - x1);
    double z = cos(3.141592654 * (i + 0.75) / (n + 0.5)), z1, pp;
    int guard = 0;
    do {
        double p1 = 1.0, p2 = 0.0, p3;
        for (int j = 1; j <= n; j++) {
            p3 = p2;
            p2 = p1;
            p1 = ((2.0 * j - 1.0) * z * p2 - (j - 1.0) * p3) / j;
        }
        pp = n * (z * p1 - p2) / (z * z - 1.0);
        z1 = z;
        z = z1 - p1 / pp;
    } while (fabs(z - z1) > 3.0e-11 && ++guard < 100);
    out[i] = xm - xl * z;
    out[n - 1 - i] = xm + xl * z;
    double w = 2.0 * xl / ((1.0 - z * z) * pp * pp);
    out[n + i] = w;
    out[n + n - 1 - i] = w;
}

int launch_gauleg(gort_ctx *ctx, cudaStream_t s, double *d_out)
{
    gauleg_kernel<<<1, 32, 0, s>>>(d_out);
    ctx->launches++;
    return check_cuda(ctx, cudaGetLastError(), "gauleg launch");
}

// ------------------------------------------------------------------------------------------------
// FP64 FMA microbenchmark: the measured denominator for the FP64 roofline (SURVEY.md 8d).
__global__ void __launch_bounds__(256) dfma_kernel(double* out, int iters, double seed)
{
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.9999999, b = 1e-7;
    for (int i = 0; i < iters; i++) {
        a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
        a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
    }
    out[(size_t) blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

int launch_dfma_peak(gort_ctx *ctx, cudaStream_t s, double *tflops)
{
    note_other_work(ctx);
    const int blocks = ctx->sm_count * 8, threads = 256, iters = 4096;
    double *d = (double *) workspace(ctx, sizeof(double) * (size_t) blocks * threads);
    if (!d) return GORT_ERR_NOMEM;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(e0, s);
        dfma_kernel<<<blocks, threads, 0, s>>>(d, iters, 1.0);
        cudaEventRecord(e1, s);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best) best = ms;
        ctx->launches++;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    double flops = 2.0 * 8.0 * iters * (double) blocks * threads;
    *tflops = flops / (best * 1e-3) / 1e12;
    return check_cuda(ctx, cudaGetLastError(), "dfma microbenchmark");
}

}  // namespace gort
