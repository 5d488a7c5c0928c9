// gort_tangent.cu -- forward-mode tangent of the BRDF with respect to favd (and LAI), sm_100a, FP64.
//
// The regrouped BRDF (gort_rsurf_wide.cuh, DESIGN.md 4.1) is
//        rsurf = cA A + Kc PDF + cG G + cZ Z + Kt T
// with per-line coefficients and per-(sun, lambda) terms.  A and G do not depend on favd, and neither do Kc and Kt, so
//        d rsurf = dcA A + Kc dPDF + dcG G + dcZ Z + cZ dZ + Kt dT.
//   geom_tangent_kernel   one thread per line: dcA, dcG, dcZ and the tangents of the sun inputs t0, tp0, pe_s, next to the
//                         primal record the existing geometry kernel wrote (which it reads for Kc, fd, K'g, K'z, t0)
//   rsurf_tangent_kernel  per (column chunk, line range): the (set, lambda) terms and their tangents once per set, the
//                         (sun, lambda) terms and their tangents once per run of lines with the same sun (the run flags of
//                         the primal records), then six FMAs and one store per evaluation.
#include "gort_device.cuh"
#include "gort_internal.h"

namespace gort {

#define GORT_TREC_STRIDE 6       // doubles per tangent line record: (dcA, dcG) (dcZ, dt0) (dtp0, dpe_s)
#define TAN_THREADS 128
#define TAN_LPT 2                // wavelength columns per thread

__global__ void __launch_bounds__(128)
geom_tangent_kernel(int n_sets, int n_geom, int geom_per_set, const double* __restrict__ structure,
                    const double* __restrict__ lut, const double* __restrict__ dlut, const double* __restrict__ angles,
                    const double* __restrict__ rec, double* __restrict__ trec)
{
    const long L = (long) n_sets * n_geom;
    const long line = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= L) return;
    const int m = (int) (line / n_geom);
    const long a = geom_per_set ? line : (line - (long) m * n_geom);
    const long na = geom_per_set ? L : n_geom;
    const Canopy c = canopy_load(structure, n_sets, m, lut);
    const Line g = line_from_degrees(angles[0 * na + a], angles[1 * na + a], angles[2 * na + a], angles[3 * na + a]);
    const Primed P = primed_trig(c, g.vza, g.sza);
    double sr, cr;
    sincos(g.raa, &sr, &cr);
    const double* dm = dlut + (size_t) m * GORT_LUT_STRIDE;
    const HotTan h = hotspot_tangent(c, lut + (size_t) m * GORT_LUT_STRIDE, dm, g.vza, g.sza, cr);
    // primal record: (cA,Kc) (cG,cZ) (Kt,flags) (q,fd) | (mus,t0) (tp0,pe_s) (K'g,K'z) (Kg,Kz)
    const double2* rr = reinterpret_cast<const double2*>(rec + (size_t) line * GORT_REC_STRIDE);
    const double Kc = rr[0].y, fd = rr[3].y, t0 = rr[4].y;
    const double2 kp = rr[6];
    const double kf = Kc * fd;
    const double dkoe = dm[2 * GORT_NTH + 1];
    const double dq = h.dkuusk / (2.0 * P.t.cs * P.t.cv);                  // q = kuusk / (2 cos sza' cos vza')
    const double dt0 = -(0.5 * elai_tangent(c) * P.t.secs) * t0;           // t0 = exp(-(0.5 elai sec sza'))
    double2* o = reinterpret_cast<double2*>(trec + (size_t) line * GORT_TREC_STRIDE);
    o[0] = make_double2(kf * dq, kf * dkoe * kp.x);                        // dcA, dcG
    o[1] = make_double2(kf * dkoe * kp.y, dt0);                            // dcZ, dt0
    o[2] = make_double2(h.dpn0_s + h.dpe_s, h.dpe_s);                      // dtp0, dpe_s
}

struct TanArgs {
    int n_sets, n_geom, n_wl, spectra_per_set, lai;
    int tw, slots;                  // column threads of a line slot, line slots of a CTA
    long lines_per_cta;
    const double *structure, *lut, *dlut, *rec, *trec, *rleaf, *tleaf, *rsoil;
    double *drsurf;
};

// Thread (slot, cw) of CTA (x, y) owns columns x * tw * LPT + cw + k tw and, of the CTA's lines y * lines_per_cta + i,
// those with i = slot mod slots.  The CTA stages the primal and tangent records of TAN_TILE lines at a time in shared
// memory with coalesced loads (a thread walking its lines through global loads waits a memory latency per line).  With
// one slot per CTA (W > 128: tw = ceil(W / (LPT n_chunks)) > 64) a thread walks consecutive lines and rebuilds its sun
// terms only where the primal record flags a new sun; with several (W <= 128) it rebuilds them at every line.  Either way they are a function of the record values
// alone, so a member's result does not depend on the batch it is in.
#define TAN_TILE 32
#define TAN_RECQ 9               // double2 per staged line: primal (cA,Kc) .. (tp0,pe_s), then the tangent record
__global__ void __launch_bounds__(TAN_THREADS)
rsurf_tangent_kernel(const TanArgs a)
{
    __shared__ double2 s_rec[TAN_TILE][TAN_RECQ];
    const int slot = threadIdx.x / a.tw, cw = threadIdx.x - slot * a.tw;
    const long L = (long) a.n_sets * a.n_geom;
    const long l0 = (long) blockIdx.y * a.lines_per_cta;
    const long l1 = min(L, l0 + a.lines_per_cta);
    int w[TAN_LPT];
    bool on[TAN_LPT];
#pragma unroll
    for (int k = 0; k < TAN_LPT; k++) {
        w[k] = blockIdx.x * a.tw * TAN_LPT + cw + k * a.tw;
        on[k] = slot < a.slots && w[k] < a.n_wl;
    }
    Canopy c;
    LeafTerms lf[TAN_LPT];
    LeafTan dl[TAN_LPT];
    SunTan sn[TAN_LPT];
    double dkoe = 0.0, scale = 1.0;
    int m_cur = -1;
    bool first = true;
    for (long t0 = l0; t0 < l1; t0 += TAN_TILE) {
        const int nt = (int) min((long) TAN_TILE, l1 - t0);
        __syncthreads();                                   // everybody has left the previous tile
        for (int e = threadIdx.x; e < nt * TAN_RECQ; e += blockDim.x) {
            const int li = e / TAN_RECQ, q = e - li * TAN_RECQ;
            const size_t line = (size_t) (t0 + li);
            s_rec[li][q] = q < 6 ? reinterpret_cast<const double2*>(a.rec + line * GORT_REC_STRIDE)[q]
                                 : reinterpret_cast<const double2*>(a.trec + line * GORT_TREC_STRIDE)[q - 6];
        }
        __syncthreads();
        if (!on[0]) continue;
        for (int li = slot; li < nt; li += a.slots) {
            const long line = t0 + li;
            const int m = (int) (line / a.n_geom);
            // (cA,Kc) (cG,cZ) (Kt,flags) (q,fd) (mus,t0) (tp0,pe_s) | (dcA,dcG) (dcZ,dt0) (dtp0,dpe_s)
            const double2* r = s_rec[li];
            const long long flags = __double_as_longlong(r[2].y);
            bool new_sun = first || a.slots > 1 || (flags & 1);
            first = false;
            if (m != m_cur) {
                m_cur = m;
                c = canopy_load(a.structure, a.n_sets, m, a.lut);
                dkoe = a.dlut[(size_t) m * GORT_LUT_STRIDE + 2 * GORT_NTH + 1];
                // d favd / d LAI at fixed crown geometry: the map favd = 3 LAI / (4 lambda pi r^2 b) of gortt.c:1129
                scale = a.lai ? 3.0 / (c.lambda * c.r * c.r * GORT_PI * c.b * 4.0) : 1.0;
                const double delai = elai_tangent(c);
#pragma unroll
                for (int k = 0; k < TAN_LPT; k++) {
                    if (!on[k]) continue;
                    const size_t sb = (a.spectra_per_set ? (size_t) m * a.n_wl : 0) + w[k];
                    lf[k] = leaf_terms(c, a.rleaf[sb], a.tleaf[sb], a.rsoil[sb]);
                    dl[k] = leaf_tangent(c, lf[k], delai, dkoe);
                }
                new_sun = true;
            }
            if (new_sun) {
                const double2 v3 = r[3], v4 = r[4], v5 = r[5], t1v = r[7], t2v = r[8];
#pragma unroll
                for (int k = 0; k < TAN_LPT; k++)
                    if (on[k]) sn[k] = sun_tangent(c, lf[k], dl[k], dkoe, v3.y, v4.x, v4.y, v5.x, v5.y, t1v.y, t2v.x, t2v.y);
            }
            const double2 v0 = r[0], v1 = r[1], v2 = r[2], t0v = r[6], t1v = r[7];
#pragma unroll
            for (int k = 0; k < TAN_LPT; k++) {
                if (!on[k]) continue;
                double d = fma(v1.y, sn[k].dZ, v2.x * sn[k].dT);      // cZ dZ + Kt dT
                d = fma(t1v.x, sn[k].Z, d);                            // + dcZ Z
                d = fma(t0v.y, sn[k].G, d);                            // + dcG G
                d = fma(v0.y, sn[k].dPDF, d);                          // + Kc dPDF
                d = fma(t0v.x, lf[k].A, d);                            // + dcA A
                a.drsurf[(size_t) line * a.n_wl + w[k]] = d * scale;
            }
        }
    }
}

int launch_brdf_tangent(gort_ctx *ctx, cudaStream_t s, const gort_shape &sh, const double *structure, const double *lut,
                        const double *dlut, const double *angles, const double *rleaf, const double *tleaf,
                        const double *rsoil, double *drsurf, int lai)
{
    const long L = (long) sh.n_sets * sh.n_geom;
    double *rec, *trec;
    unsigned long long *flags;
    {
        int rc = next_records(ctx, s, L, &rec, &flags);
        if (rc != GORT_OK) return rc;
    }
    trec = (double *) workspace(ctx, sizeof(double) * GORT_TREC_STRIDE * (size_t) L);
    if (!trec) return GORT_ERR_NOMEM;
    // the primal records, in plain stream order
    {
        int rc = launch_geom(ctx, s, sh, structure, lut, angles, rec, NULL, flags, false);
        if (rc != GORT_OK) return rc;
    }
    geom_tangent_kernel<<<(unsigned) ((L + 127) / 128), 128, 0, s>>>(sh.n_sets, sh.n_geom, sh.geom_per_set, structure,
                                                                     lut, dlut, angles, rec, trec);
    // columns: chunks of at most TAN_THREADS * TAN_LPT, lanes spread evenly; small W packs several line slots per CTA
    const int n_chunks = (sh.n_wl + TAN_THREADS * TAN_LPT - 1) / (TAN_THREADS * TAN_LPT);
    TanArgs a;
    a.n_sets = sh.n_sets; a.n_geom = sh.n_geom; a.n_wl = sh.n_wl; a.spectra_per_set = sh.spectra_per_set; a.lai = lai;
    a.tw = (sh.n_wl + n_chunks * TAN_LPT - 1) / (n_chunks * TAN_LPT);
    a.slots = TAN_THREADS / a.tw;
    a.structure = structure; a.lut = lut; a.dlut = dlut; a.rec = rec; a.trec = trec;
    a.rleaf = rleaf; a.tleaf = tleaf; a.rsoil = rsoil; a.drsurf = drsurf;
    // a few resident waves of CTAs over contiguous line ranges
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, rsurf_tangent_kernel, TAN_THREADS, 0) != cudaSuccess || occ < 1) occ = 1;
    long nby = (4L * ctx->sm_count * occ) / n_chunks;
    if (nby < 1) nby = 1;
    if (nby > L) nby = L;
    a.lines_per_cta = (L + nby - 1) / nby;
    nby = (L + a.lines_per_cta - 1) / a.lines_per_cta;
    rsurf_tangent_kernel<<<dim3((unsigned) n_chunks, (unsigned) nby), TAN_THREADS, 0, s>>>(a);
    ctx->launches += 2;
    note_other_work(ctx);
    return check_cuda(ctx, cudaGetLastError(), "gort_brdf_tangent launch");
}

}  // namespace gort
