// gort_rsurf_wide.cuh -- the per-wavelength loop of gortt_rsurf (gortt.c:460-567) for wide spectra
// (W >= 64), the dominant kernel of the BRDF path.
//
// Work decomposition (grid.x = wavelength chunks, grid.y = contiguous line ranges):
//   * a CTA owns one wavelength chunk and walks a CONTIGUOUS range of input lines, sized so that the
//     whole grid is one resident wave.  Warp w of the CTA owns the 32*LPT consecutive wavelengths
//     [w*32*LPT, (w+1)*32*LPT) of the chunk; its j-th store of a line lands 256*j bytes after the first,
//     so the LPT stores of a line share one address register and use immediate offsets;
//   * the packed 128-byte line records written by geom_kernel are staged into shared memory
//     WIDE_STAGE_LINES at a time and cut into "runs" of lines that share parameter set and sun
//     (flags computed by geom_kernel from the input angles);
//   * the (set, lambda) terms (exp, sqrt, four divides) are computed once per set into shared memory;
//   * the (sun, lambda) terms are re-derived only at the start of a run and then live in registers:
//     A, PDF, G, Z, T;
//   * inside a run only the view-dependent part remains per (line, lambda).  gortt.c:557,
//         rsurf = Kc*C + Kg*G + Kt*T + Kz*Z,   C = fd*(A*q + PD + ke*(G*K'g + Z*K'z)) + FCf,
//     is regrouped by per-(sun, lambda) term,
//         rsurf = cA*A + Kc*PDF + cG*G + cZ*Z + Kt*T,
//     with the five per-line coefficients prepared by geom_kernel: 3 broadcast LDS.128 per line, then
//     5 FP64 instructions per evaluation, no branches.  Output: with 128-byte aligned rows the results of three
//     consecutive rows are dropped into a shared-memory ring and handed to the TMA engine as bulk stores
//     (cp.async.bulk, SASS UBLKCP: one CTA barrier per three rows; bulk stores of >= 4.6 KB reach 6.0 TB/s in
//     isolation where per-thread stores reach 5.3); otherwise one coalesced 8-byte store per evaluation.
//     (With scomp requested the crown signature C itself is an output and the long form is used.)
// HBM traffic is 8 B per evaluation (rsurf) -- the binding roofline for this kernel (DESIGN.md).
// Output rows are `pitch` doubles apart; a pitch that is a multiple of 16 doubles keeps every warp store
// line-aligned, and the kernel then also fills the padding columns up to the end of the row's last 128-byte
// line (with copies of the last column): a row that ends in a partially written line costs the memory system
// a read-modify-write, measured at 41.6 us vs 37.1 us per 196 MB for the same store stream
// (tools/microbench/loop_bw.cu, profiles/r1_microbench_loop_bw.txt).
//
// Pipeline across kernels and calls (all of it optional: without programmatic dependent launch the same code
// runs strictly in stream order and every wait below is already satisfied):
//   * the kernel is launched as a programmatic dependent of geom_kernel and never waits for that grid to
//     complete; it builds its (set, lambda) table first and then waits, stage by stage, on the per-tile flags
//     geom_kernel publishes with its records;
//   * before its first store a CTA waits until the CTA with the same index in the previous launch of the same
//     shape has finished (that CTA wrote the same output region), then releases its own dependents: the NEXT
//     call's geom_kernel, which therefore runs underneath this launch's store phase;
//   * at exit a CTA publishes its epoch.
//   Steady state for repeated calls: the store stream of call i+1 starts CTA by CTA as the CTAs of call i
//   retire, with the geometry of call i+1 already in HBM.  Measured on C2: 54.7 -> 39 us per call.
#pragma once
#include "gort_device.cuh"

namespace gort {

#define WIDE_MAX_THREADS 384      // register cap of the kernel: 65536 / (2 * 384) -> 80
#define WIDE_PICK_THREADS 288     // largest block the launch heuristic picks: two CTAs then leave an SM room for one geom_kernel CTA
#define WIDE_PICK_THREADS_TMA 192 // same, TMA output path: (9 + 2*3) arrays of 4*192 doubles + 16 KB of records, twice, fit 227 KB
#define WIDE_TMA_ROWS 3           // rows per CTA barrier on the TMA output path
#define WIDE_TMA_ROWS_SCOMP 2     // the same with component signatures (40 B per evaluation in the ring)
#define WIDE_STAGE_LINES 128      // lines staged in shared memory per pass (16 KB)
#define WIDE_NLEAF 9              // omega gam Tff Rff pff tff rs Xf A

struct WideArgs {
    int n_sets, n_geom, n_wl, spectra_per_set;
    int n_col;                    // columns written per row: n_wl, or up to the end of the row's last 128-byte line when the pitch allows
    int chunk;                    // wavelengths per CTA (= LPT * blockDim.x)
    unsigned long long *tl;       // optional timeline [grid][8] of %globaltimer stamps (GORT_TIMELINE, development aid)
    int pdl;                      // launched with programmatic stream serialization after geom_kernel
    const unsigned long long *tile_flags;   // this call's flag array, per 32-line tile: call number whose records geom_kernel has published
    unsigned long long call_no;
    unsigned long long *fault;    // set to the call number if a bounded wait below ever expires
    unsigned long long *done;     // [grid size] per-CTA epoch: the last launch in which CTA k of this grid shape finished
    unsigned long long wait_target;   // epoch of the previous launch with the SAME grid shape and outputs (0: nothing to wait for)
    unsigned long long epoch;         // this launch's epoch
    long pitch;                   // output row stride in doubles (>= n_wl)
    long lines_per_cta;
    const double *structure, *lut, *rec, *rleaf, *tleaf, *rsoil;
    double *rsurf, *scomp;
};

template <int LPT, bool SCOMP, int TMAB>
__global__ void __launch_bounds__(WIDE_MAX_THREADS, 2)
rsurf_wide_kernel(const WideArgs a)
{
    constexpr int STAGE = WIDE_STAGE_LINES;
#define WIDE_TL(k) do { if (a.tl && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.tl[(size_t) (blockIdx.y * gridDim.x + blockIdx.x) * 8 + (k)] = t_; } } while (0)
    WIDE_TL(0);                                                               // CTA entry
    extern __shared__ __align__(128) double2 smem2[];                        // records of a stage are whole 128-byte lines
    double2* srec = smem2;                                                    // [STAGE][8] packed records
    unsigned* runmask = reinterpret_cast<unsigned*>(srec + 8 * STAGE);   // [STAGE / 32] run-start bits (16 bytes reserved)
    double* leaf = reinterpret_cast<double*>(runmask + 4);                 // [WIDE_NLEAF][chunk], 16-byte aligned
    double* ring = leaf + (size_t) WIDE_NLEAF * a.chunk;                              // TMAB > 0: two halves of TMAB output rows (x5 with component signatures)
    __shared__ int s_fault;       // a bounded wait expired: this CTA stores nothing more (and the host is told)
    if (threadIdx.x == 0) s_fault = 0;
    __syncthreads();

    const long L = (long) a.n_sets * a.n_geom;
    const unsigned cta = blockIdx.y * gridDim.x + blockIdx.x;
    const long line_begin = (long) blockIdx.y * a.lines_per_cta;
    const long line_end = min(L, line_begin + a.lines_per_cta);
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int wbase = blockIdx.x * a.chunk;
    const int chunk = a.chunk;
    // slot j of this thread: column kq + 32*j of the chunk
    const int kq = (tid >> 5) * (32 * LPT) + (tid & 31);
    bool ok[LPT];
#pragma unroll
    for (int j = 0; j < LPT; j++) ok[j] = (wbase + kq + 32 * j) < a.n_col;

    int m = (int) (line_begin / a.n_geom);
    long set_end = (long) (m + 1) * a.n_geom;                     // first line of the next set
    double k_open = 0.0, ke = 0.0;
    bool leaf_ready = false;

    // (set, lambda) terms of this chunk into shared memory, computed by every CTA: in the steady state this runs under
    // the co-resident CTA's stores (DESIGN.md 4.1)
    auto fill_leaf = [&](int mm) {
        const Canopy c = canopy_load(a.structure, a.n_sets, mm, a.lut);
        k_open = c.k_open; ke = c.k_openep;
        const size_t sb = a.spectra_per_set ? (size_t) mm * a.n_wl : 0;
        // this thread's LPT columns: all spectra loads are issued before the first dependent use
        double rl[LPT], tl[LPT], rs[LPT];
#pragma unroll
        for (int j = 0; j < LPT; j++) {
            const int w = min(wbase + kq + 32 * j, a.n_wl - 1);
            rl[j] = a.rleaf[sb + w]; tl[j] = a.tleaf[sb + w]; rs[j] = a.rsoil[sb + w];
        }
#pragma unroll
        for (int j = 0; j < LPT; j++) {
            const int k = kq + 32 * j;
            LeafTerms Lf = leaf_terms(c, rl[j], tl[j], rs[j]);
            leaf[0 * chunk + k] = Lf.omega; leaf[1 * chunk + k] = Lf.gam; leaf[2 * chunk + k] = Lf.Tff;
            leaf[3 * chunk + k] = Lf.Rff;   leaf[4 * chunk + k] = Lf.pff; leaf[5 * chunk + k] = Lf.tff;
            leaf[6 * chunk + k] = Lf.rs;    leaf[7 * chunk + k] = Lf.Xf;  leaf[8 * chunk + k] = Lf.A;
        }
    };

    bool prefetched = false;      // the first stage's record copies were issued in the prologue
    if (line_begin < line_end) {
        // Prologue that does not depend on geom_kernel's line records: under PDL it overlaps with that grid.  In plain
        // stream order (the geometry kernel is complete: every flag is set, no acquire needed) the asynchronous copies of
        // the first stage's records are issued first, so that they are in flight while the (set, lambda) table is built.
        if (!a.pdl) {
            const int nl0 = (int) min((long) STAGE, line_end - line_begin);
            const double2* g = reinterpret_cast<const double2*>(a.rec + (size_t) line_begin * GORT_REC_STRIDE);
            const unsigned sbase = (unsigned) __cvta_generic_to_shared(srec);
            for (int i = tid; i < nl0 * 8; i += nthr)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(sbase + 16u * i), "l"(g + i) : "memory");
            asm volatile("cp.async.commit_group;" ::: "memory");
            prefetched = true;
        }
        fill_leaf(m);
        leaf_ready = true;
    }
    WIDE_TL(1);                                                               // (set, lambda) table done
    if (line_begin >= line_end) {
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (tid == 0) a.done[cta] = a.epoch;
        return;
    }
    bool gate_open = false;       // this CTA has not stored anything yet
    int half = 0;                 // TMA path: which half of the row ring the next batch fills
    const unsigned row_bytes = 8u * (unsigned) max(0, min(chunk, a.n_col - wbase));

    double sA[LPT], sP[LPT], sG[LPT], sZ[LPT], sT[LPT];
    double sPD[SCOMP ? LPT : 1], sFCf[SCOMP ? LPT : 1];
#pragma unroll
    for (int j = 0; j < LPT; j++) { sA[j] = sP[j] = sG[j] = sZ[j] = sT[j] = 0.0; }

    for (long s0 = line_begin; s0 < line_end; s0 += STAGE) {
        const int nl = (int) min((long) STAGE, line_end - s0);
        __syncthreads();                                          // previous stage fully consumed
        {   // ---- wait for geom_kernel's tiles of this stage (acquire on their flags; every CTA of geom_kernel is
            //      resident or done before this kernel can be scheduled, so the wait cannot deadlock), then stage
            //      the packed records of lines [s0, s0+nl): 8 x 16 bytes per line, asynchronous copies (LDGSTS) so
            //      that every load of the stage is in flight at once ----
            const long tile0 = s0 >> 5, tile1 = (s0 + nl - 1) >> 5;
            for (long t = tile0 + tid; t <= tile1; t += nthr) {
                unsigned long long v, t0 = 0, t1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                for (;;) {
                    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(a.tile_flags + t) : "memory");
                    if (v >= a.call_no) break;
                    __nanosleep(100);
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if (t1 - t0 > 2000000000ull) { *a.fault = a.call_no; s_fault = 1; break; }   // 2 s: never hang; reported by gort_synchronize
                }
            }
            __syncthreads();
            if (s_fault) break;                                   // the records never arrived: store nothing
            if (s0 == line_begin) WIDE_TL(2);                     // geometry records of the first stage ready
            if (!(prefetched && s0 == line_begin)) {
                const double2* g = reinterpret_cast<const double2*>(a.rec + (size_t) s0 * GORT_REC_STRIDE);
                const unsigned sbase = (unsigned) __cvta_generic_to_shared(srec);
                for (int i = tid; i < nl * 8; i += nthr)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(sbase + 16u * i), "l"(g + i) : "memory");
                asm volatile("cp.async.commit_group;" ::: "memory");
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        // a "run" = a maximal stretch of lines sharing set and sun: starts at line 0 of the stage or at a
        // flagged line and ends before the next flagged line.  One ballot per 32 lines gives the start mask.
        for (int i0 = (tid >> 5) * 32; i0 < nl; i0 += nthr) {
            const int i = i0 + (tid & 31);
            const bool start = i < nl && (int) __double_as_longlong(srec[8 * i + 2].y) != 0;
            const unsigned bal = __ballot_sync(0xffffffffu, start);
            if ((tid & 31) == 0) runmask[i0 >> 5] = bal;
        }
        __syncthreads();

        int l = 0;
        while (l < nl) {
            int f = (int) __double_as_longlong(srec[8 * l + 2].y);
            if (s0 + l == line_begin) f = 3;                      // a CTA's first line starts everything
            if (f & 2) {
                // ---- new parameter set ----
                const long ln = s0 + l;
                if (ln >= set_end) { m++; set_end += a.n_geom; }  // lines advance one run at a time within a set
                if (!leaf_ready) {
                    __syncthreads();                              // everyone is done reading the old leaf terms
                    fill_leaf(m);
                }
                leaf_ready = false;
                __syncthreads();
            }
            if (f & 1) {
                // ---- new sun: (sun, lambda) terms into registers ----
                const double fd = srec[8 * l + 3].y;
                const double2 s0v = srec[8 * l + 4], s1v = srec[8 * l + 5];       // (mus,t0) (tp0,pe_s)
                Canopy c;
                c.k_open = k_open; c.k_openep = ke;
                const double K = k_open + ke;
#pragma unroll
                for (int j = 0; j < LPT; j++) {
                    const int k = kq + 32 * j;                    // < chunk
                    LeafTerms Lf;
                    Lf.omega = leaf[0 * chunk + k]; Lf.gam = leaf[1 * chunk + k]; Lf.Tff = leaf[2 * chunk + k];
                    Lf.Rff = leaf[3 * chunk + k];   Lf.pff = leaf[4 * chunk + k]; Lf.tff = leaf[5 * chunk + k];
                    Lf.rs = leaf[6 * chunk + k];    Lf.Xf = leaf[7 * chunk + k];
                    Lf.tpff = Lf.tff * (1.0 - K) + K;             // gortt_brdf.c:381-382, as in leaf_terms
                    Lf.Zf = (Lf.tpff - ke) * Lf.rs;               // gortt.c:492
                    SunTerms S = sun_terms(c, Lf, fd, s0v.x, s0v.y, s1v.x, s1v.y);
                    sA[j] = leaf[8 * chunk + k];
                    sP[j] = S.PDF; sG[j] = S.G; sZ[j] = S.Z; sT[j] = S.T;
                    if (SCOMP) { sPD[j] = S.PD; sFCf[j] = S.FCf; }
                }
            }
            if (!gate_open) {
                WIDE_TL(3);                                                   // records staged, first sun terms in registers
                // Cross-call pipeline.  Under programmatic dependent launch this CTA may have started while the
                // previous call's per-wavelength kernel was still storing to the same output buffer.  Everything
                // up to here touched only inputs, records and registers; before the first store wait until the
                // CTA that owned this very output region in the previous launch (same grid shape, so same index)
                // has finished.  It is resident or done by the time this kernel can be scheduled, so the wait
                // cannot deadlock; it is bounded anyway.  Then let the NEXT call's geometry kernel start: it runs
                // underneath this kernel's store phase, and by then every CTA of the previous launch is done, so
                // the record buffer it overwrites is free.
                if (tid == 0) {
                    unsigned long long v, t0 = 0, t1;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                    for (;;) {
                        asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(a.done + cta) : "memory");
                        if (v >= a.wait_target) break;
                        __nanosleep(200);
                        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                        if (t1 - t0 > 2000000000ull) { *a.fault = a.call_no; s_fault = 1; break; }   // 2 s: never hang; reported by gort_synchronize
                    }
                }
                __syncthreads();
                asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
                gate_open = true;
                WIDE_TL(4);                                                   // gate passed: first store follows
                if (s_fault) break;                               // the region's previous owner never finished: store nothing
            }
            // ---- the run: only the view-dependent part per (line, lambda) ----
            int e = nl;                                           // first run start after line l
            for (int wd = l >> 5; wd < (nl + 31) >> 5; wd++) {
                unsigned mk = runmask[wd];
                if (wd == (l >> 5)) mk &= (l & 31) == 31 ? 0u : (0xffffffffu << ((l & 31) + 1));
                if (mk) { e = wd * 32 + __ffs(mk) - 1; break; }
            }
            double* out = a.rsurf + (size_t) (s0 + l) * a.pitch + wbase + kq;
            const double2* vr = srec + 8 * l;
            if (TMAB > 0 && !SCOMP) {
                // Output through shared memory and the TMA engine, TMAB rows per CTA barrier: every thread drops
                // its LPT results of up to TMAB consecutive rows into one half of a 2*TMAB-row ring, one thread
                // hands each row chunk to cp.async.bulk (SASS UBLKCP) while the CTA fills the other half.
                while (l < e) {
                    const int nb = min(TMAB, e - l);
                    double* sb = ring + (size_t) half * TMAB * chunk + kq;
#pragma unroll
                    for (int b = 0; b < TMAB; b++) {
                        if (b < nb) {
                            const double2 v0 = vr[8 * b], v1 = vr[8 * b + 1];
                            const double cT = vr[8 * b + 2].x;
#pragma unroll
                            for (int j = 0; j < LPT; j++)
                                sb[b * chunk + 32 * j] = fma(v0.x, sA[j], fma(v0.y, sP[j], fma(v1.x, sG[j], fma(v1.y, sZ[j], cT * sT[j]))));
                        }
                    }
                    // the half the NEXT batch fills was handed to the TMA engine one batch ago: its reads of shared
                    // memory must be over before this barrier releases the CTA into that half
                    if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncthreads();
                    if (tid == 0) {
                        for (int b = 0; b < nb; b++) {
                            const unsigned sa = (unsigned) __cvta_generic_to_shared(ring + ((size_t) half * TMAB + b) * chunk);
                            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                         :: "l"(a.rsurf + (size_t) (s0 + l + b) * a.pitch + wbase), "r"(sa), "r"(row_bytes) : "memory");
                        }
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    half ^= 1;
                    l += nb; vr += 8 * nb;
                }
            } else if (TMAB > 0 && SCOMP) {
                // Component signatures through the same ring: per row the chunk of rsurf and, behind it, the chunk of
                // { C, G, T, Z } quadruples (32 B per evaluation, two STS.128 per column); one thread hands both pieces
                // of every row to cp.async.bulk.  Whole 128-byte lines leave the SM instead of per-thread 16-byte
                // pieces of a 32-byte AoS element (the per-thread path reaches 0.46 of the HBM rate).
                const size_t half_stride = (size_t) TMAB * 5 * chunk;
                while (l < e) {
                    const int nb = min(TMAB, e - l);
                    double* sr = ring + (size_t) half * half_stride + kq;                          // [TMAB][chunk]
                    double* ss = ring + (size_t) half * half_stride + (size_t) TMAB * chunk;       // [TMAB][chunk][4]
#pragma unroll
                    for (int b = 0; b < TMAB; b++) {
                        if (b < nb) {
                            const double Kc = vr[8 * b].y, Kt = vr[8 * b + 2].x;
                            const double2 v3 = vr[8 * b + 3], v6 = vr[8 * b + 6], v7 = vr[8 * b + 7];   // (q,fd) (K'g,K'z) (Kg,Kz)
#pragma unroll
                            for (int j = 0; j < LPT; j++) {
                                const double zg = fma(sG[j], v6.x, sZ[j] * v6.y);             // Z*K'z + G*K'g   gortt.c:514
                                double Cd = fma(sA[j], v3.x, sPD[j]);                         // CdC + CdCG      gortt.c:504-507
                                Cd = fma(ke, zg, Cd);                                         // + CdG           gortt.c:528
                                const double C = fma(v3.y, Cd, sFCf[j]);                      // gortt.c:531
                                sr[b * chunk + 32 * j] = fma(v7.y, sZ[j], fma(Kt, sT[j], fma(v7.x, sG[j], Kc * C)));   // gortt.c:557
                                double2* q4 = reinterpret_cast<double2*>(ss + ((size_t) b * chunk + kq + 32 * j) * 4);
                                q4[0] = make_double2(C, sG[j]);
                                q4[1] = make_double2(sT[j], sZ[j]);
                            }
                        }
                    }
                    if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncthreads();
                    if (tid == 0) {
                        for (int b = 0; b < nb; b++) {
                            const size_t go = (size_t) (s0 + l + b) * a.pitch + wbase;
                            const unsigned sa = (unsigned) __cvta_generic_to_shared(ring + (size_t) half * half_stride + (size_t) b * chunk);
                            const unsigned sq = (unsigned) __cvta_generic_to_shared(ss + (size_t) b * chunk * 4);
                            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                         :: "l"(a.rsurf + go), "r"(sa), "r"(row_bytes) : "memory");
                            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                         :: "l"(a.scomp + 4 * go), "r"(sq), "r"(4u * row_bytes) : "memory");
                        }
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    half ^= 1;
                    l += nb; vr += 8 * nb;
                }
            } else if (!SCOMP) {
#pragma unroll 4
                for (; l < e; l++, vr += 8, out += a.pitch) {
                    const double2 v0 = vr[0], v1 = vr[1];          // (cA,Kc) (cG,cZ)
                    const double cT = vr[2].x;                     // Kt
#pragma unroll
                    for (int j = 0; j < LPT; j++) {
                        const double r = fma(v0.x, sA[j], fma(v0.y, sP[j], fma(v1.x, sG[j], fma(v1.y, sZ[j], cT * sT[j]))));
                        if (ok[j]) out[32 * j] = r;
                    }
                }
            } else {
                for (; l < e; l++, vr += 8, out += a.pitch) {
                    const double Kc = vr[0].y, Kt = vr[2].x;
                    const double2 v3 = vr[3], v6 = vr[6], v7 = vr[7];   // (q,fd) (K'g,K'z) (Kg,Kz)
#pragma unroll
                    for (int j = 0; j < LPT; j++) {
                        const double zg = fma(sG[j], v6.x, sZ[j] * v6.y);             // Z*K'z + G*K'g   gortt.c:514
                        double Cd = fma(sA[j], v3.x, sPD[j]);                         // CdC + CdCG      gortt.c:504-507
                        Cd = fma(ke, zg, Cd);                                         // + CdG           gortt.c:528
                        const double C = fma(v3.y, Cd, sFCf[j]);                      // gortt.c:531
                        const double r = fma(v7.y, sZ[j], fma(Kt, sT[j], fma(v7.x, sG[j], Kc * C)));   // gortt.c:557
                        if (ok[j]) {
                            out[32 * j] = r;
                            double* sc = a.scomp + 4 * (size_t) (out + 32 * j - a.rsurf);
                            *reinterpret_cast<double2*>(sc) = make_double2(C, sG[j]);
                            *reinterpret_cast<double2*>(sc + 2) = make_double2(sT[j], sZ[j]);
                        }
                    }
                }
            }
        }
        if (s_fault) break;
    }
    if (!gate_open) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // publish: all stores of this CTA happen-before the flag (bulk stores complete, barrier, then fence + release
    // by one thread)
    if (TMAB > 0 && tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    __syncthreads();
    WIDE_TL(5);                                                               // all stores issued
    if (tid == 0) { __threadfence(); asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(a.done + cta), "l"(a.epoch) : "memory"); }
}

}  // namespace gort
