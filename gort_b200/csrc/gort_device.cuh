// gort_device.cuh -- device-side building blocks shared by the GORT kernels (sm_100a, FP64).
//
// Compiled with -fmad=false: every a*b+c written with operators stays an unfused multiply and
// add, in the reference's operation order, so that the geometry / gap-probability code sees the
// same cancellations the reference sees (SURVEY.md App. B1: r*r - h2*h2 must stay exactly 0).
// Where contraction is wanted (the per-wavelength loop) the code calls fma() explicitly.
//
// Reference citations are to /root/reference (tquaife/gort).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include "../../include/gort_b200.h"

#define GORT_PI 3.14159265358979323846      // M_PI
#define GORT_1_PI 0.31830988618379067154    // M_1_PI
#define GORT_SIN_PI 1.2246467991473532e-16  // sin(M_PI) in FP64, used for the raa = 180 deg pass

namespace gort {

// Branch-free FP64 division for the per-wavelength terms: MUFU.RCP64H seed, two Newton steps on the
// reciprocal, one correction of the quotient (result within 1 ULP of the IEEE quotient for normal
// operands).  The IEEE operator compiles to a sequence with a slow-path branch, which stops ptxas from
// interleaving the independent per-wavelength chains of one thread; this one keeps them in one basic
// block.  b == 0 keeps the IEEE result (a/0 = +-inf, 0/0 = NaN) through the selects.
__device__ __forceinline__ double fdiv(double a, double b)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
    double e = fma(-b, r, 1.0);
    r = isfinite(e) ? fma(r, e, r) : r;
    e = fma(-b, r, 1.0);
    r = isfinite(e) ? fma(r, e, r) : r;
    double q = a * r;
    double rem = fma(-b, q, a);
    return isfinite(rem) ? fma(rem, r, q) : q;
}

// ---- per-set canopy scalars needed by the BRDF / energy path (gortt.c:641-697) ---------------
struct Canopy {
    double lambda, r, b, h1, h2, favd;
    double rr;        // r*r                       gortt.c:642
    double h;         // 2 r (b/r) + h2 - h1       gortt.c:644
    double ellip;     // b/r                       gortt.c:641
    double elai;      // favd*(1.333333*lambda*pi*ellip*r^3)   gortt.c:657
    double kfavd;     // k*favd with k = 0.5       gortt.c:655,658
    double k_open, k_openep;   // LUT scalars
};

__device__ __forceinline__ Canopy canopy_load(const double* __restrict__ structure, int n_sets, int m,
                                              const double* __restrict__ lut)
{
    Canopy c;
    c.lambda = structure[0 * (size_t) n_sets + m];
    c.r      = structure[1 * (size_t) n_sets + m];
    c.b      = structure[2 * (size_t) n_sets + m];
    c.h1     = structure[3 * (size_t) n_sets + m];
    c.h2     = structure[4 * (size_t) n_sets + m];
    c.favd   = structure[5 * (size_t) n_sets + m];
    c.ellip = c.b / c.r;
    c.rr = c.r * c.r;
    double rrr = c.rr * c.r;
    c.h = 2.0 * c.r * c.ellip + c.h2 - c.h1;
    c.elai = c.favd * ((1.333333) * c.lambda * GORT_PI * c.ellip * rrr);
    c.kfavd = 0.5 * c.favd;
    const double* l = lut + (size_t) m * GORT_LUT_STRIDE;
    c.k_open = l[2 * GORT_NTH];
    c.k_openep = l[2 * GORT_NTH + 1];
    return c;
}

// ---- one input line after the reference's angle preparation (gortt.c:240-291) ------------------
struct Line {
    double vza, vaa, sza, saa, raa;   // radians, normalised
};

__device__ __forceinline__ double dtor(double x) { return x * GORT_PI / 180.0; }

// gortt.c:279 and gortt_albedo.c:97
__device__ __forceinline__ double fold_raa(double raa)
{
    return fabs((raa - 2 * GORT_PI * (int) (0.5 + raa * GORT_1_PI * 0.5)));
}

__device__ __forceinline__ Line line_from_degrees(double vza_d, double vaa_d, double sza_d, double saa_d)
{
    Line g;
    g.vza = dtor(vza_d); g.vaa = dtor(vaa_d); g.sza = dtor(sza_d); g.saa = dtor(saa_d);
    if (g.sza < 0.0) { g.saa += GORT_PI; g.sza *= -1.0; }              // gortt.c:253-260
    if (g.vza < 0.0) { g.vaa += GORT_PI; g.vza *= -1.0; }
    // gortt.c:264-274; bounded so that a non-finite azimuth cannot spin forever
    for (int it = 0; it < 4096 && g.saa > 2 * GORT_PI; it++) g.saa -= 2 * GORT_PI;
    for (int it = 0; it < 4096 && g.vaa > 2 * GORT_PI; it++) g.vaa -= 2 * GORT_PI;
    for (int it = 0; it < 4096 && g.saa < 0; it++) g.saa += 2 * GORT_PI;
    for (int it = 0; it < 4096 && g.vaa < 0; it++) g.vaa += 2 * GORT_PI;
    g.raa = fold_raa(g.saa - g.vaa);                                   // gortt.c:278-279
    return g;
}

// ---- wavelength-independent terms of one (set, line): the "geometry record" --------------------
// Everything gortt_rsurf computes before its wavelength loop (gortt.c:424-449) plus the
// wavelength-independent factors the loop re-derives per band (Kuusk hotspot, t_0, sec terms).
//
// The record is split into ROLES with no data dependence between them (primed trig is recomputed by
// each role that needs it), so that geom_kernel can run the roles of one line on different warps and
// cut the dependent-instruction chain of a line from ~4200 to ~1100 SASS instructions; the energy
// and band kernels call the same role functions one after another and get the same bits.
struct GeomRec {
    double Kc, Kg, Kt, Kz, Kpg, Kpz;   // gortt.c:429-449
    double fd;                          // gortt.c:291
    double mus;                         // cos(sza')
    double q;                           // kuusk / (2 cos sza' cos vza')   gortt.c:504-507
    double tp0;                         // p_neq0_heq0_sza + p_ngt0_heq0_sza   gortt_brdf.c:447
    double pe_s;                        // p_ngt0_heq0_sza
    double t0;                          // exp(-k elai / cos sza')   gortt_brdf.c:534
    double pn0_s;                       // p_neq0_heq0_sza (energy balance, gortt_albedo.c:37)
    // rsurf = Kc*C + Kg*G + Kt*T + Kz*Z (gortt.c:557) regrouped by per-(sun, lambda) term:
    //   rsurf = cA*A + Kc*(fd*PD + FCf) + cG*G + cZ*Z + Kt*T
    double cA;                          // Kc fd q
    double cG;                          // Kc fd k_openep K'g + Kg
    double cZ;                          // Kc fd k_openep K'z + Kz
};
// packed 128-byte line record in HBM, as double2 pairs:
//   [0] (cA, Kc) [1] (cG, cZ) [2] (Kt, flags) [3] (q, fd) | [4] (mus, t0) [5] (tp0, pe_s) [6] (K'g, K'z) [7] (Kg, Kz)
#define GORT_REC_STRIDE 16      // doubles per packed line record

// gortt.c:872-915 for one zenith angle.  The reference indexes p_n0[0][ceil(pos)] with no bound;
// for zenith = 90 deg rounding can give 91 (one past the table): clamp to the last row.
__device__ __forceinline__ void zenith_lerp(const double* __restrict__ lut, double za, double& pn0, double& pe)
{
    const double dth = 1 * GORT_PI / 180.0;       // gortt.c:76
    double pos = fabs(za) / dth;
    int ci = (int) ceil(pos), fi = (int) floor(pos);
    double d = pos - fi;
    ci = min(max(ci, 0), GORT_NTH - 1);
    fi = min(max(fi, 0), GORT_NTH - 1);
    pn0 = d * lut[ci] + (1.0 - d) * lut[fi];
    pe = d * lut[GORT_NTH + ci] + (1.0 - d) * lut[GORT_NTH + fi];
}

#define GORT_MAX(x, y) ((x) > (y) ? (x) : (y))
#define GORT_MIN(x, y) ((x) < (y) ? (x) : (y))

struct Trig {   // trig of the primed zeniths, shared by the three principal-plane passes
    double ts, tv, secs, secv, cs, cv, ss, sv;
};

struct Primed {
    double vza_p, sza_p;
    Trig t;
};

// gortt_prime_theta (gortt.c:581-588): theta' = atan((b/r) tan theta), and the tan / sin / cos / sec of
// theta' that gortt_overlap, gortt_kg and gortt_kc_fFbeta evaluate again and again.  With x = (b/r) tan theta:
// tan(atan x) = x, cos(atan x) = 1/sqrt(1+x^2), sin(atan x) = x/sqrt(1+x^2) -- each within 1 ULP of what the
// reference's libm chain returns (itself 1-2 ULP), for a third of the dependent instructions.  Near grazing
// incidence (|x| >= 1e5, theta' within 1e-5 rad of 90 deg) the reference's cos(atan x) is dominated by the
// rounding of the angle itself, so there the literal chain is kept.
__device__ __forceinline__ void primed_side(double ellip, double za, double& za_p, double& tn, double& sn,
                                            double& cn, double& sec)
{
    const double x = ellip * tan(za);
    za_p = atan(x);
    if (fabs(x) < 1e5) {
        tn = x;
        sec = sqrt(1.0 + x * x);
        cn = 1.0 / sec;
        sn = x * cn;
    } else {
        tn = tan(za_p);
        sincos(za_p, &sn, &cn);
        sec = 1.0 / cn;
    }
}

__device__ __forceinline__ Primed primed_trig(const Canopy& c, double vza, double sza)
{
    Primed P;
    primed_side(c.ellip, sza, P.sza_p, P.t.ts, P.t.ss, P.t.cs, P.t.secs);
    primed_side(c.ellip, vza, P.vza_p, P.t.tv, P.t.sv, P.t.cv, P.t.secv);
    return P;
}

// gortt_brdf.c:23-100 (live branches only)
__device__ __forceinline__ double overlap_fn(const Canopy& c, const Trig& t, double cr, double sr)
{
    double d = t.ts * t.ts + t.tv * t.tv - 2.0 * t.ts * t.tv * cr;
    double D = sqrt(GORT_MAX(0.0, d));
    double tt = t.ts * t.tv * sr;
    double t2 = sqrt(D * D + tt * tt);
    double t1 = (t.secs + t.secv);
    double cos_t = (c.h / c.b) * t2 / t1;
    cos_t = GORT_MAX(-1.0, cos_t);
    cos_t = GORT_MIN(1.0, cos_t);
    double th = acos(cos_t);
    return GORT_MAX(0.0, (th - sin(th) * cos_t) * (t.secs + t.secv) / GORT_PI);
}

// gortt_brdf.c:7-20
__device__ __forceinline__ double kg_from_overlap(const Canopy& c, const Trig& t, double overlap)
{
    return exp(-(c.lambda * (c.r * c.r) * GORT_PI * (t.secs + t.secv - overlap)));
}

struct CrownLite {   // raa-independent pieces of gortt_kc_fFbeta (gortt_brdf.c:195-207)
    double Mv, theta_Mi, Gamma_v;
};

__device__ __forceinline__ CrownLite crown_lite(const Canopy& c, const Trig& t)
{
    CrownLite s;
    double xs = c.lambda * GORT_PI * c.rr * t.secs;
    double xv = c.lambda * GORT_PI * c.rr * t.secv;
    double Mi = (1.0 - (1.0 - exp(-xs)) / xs);
    s.Mv = (1.0 - (1.0 - exp(-xv)) / xv);
    s.theta_Mi = acos(1.0 - 2.0 * Mi);
    s.Gamma_v = GORT_PI * c.rr * t.secv;
    return s;
}

// gortt_brdf.c:223-232
__device__ __forceinline__ double crown_beta(const Canopy& c, double sza_p, double secv)
{
    if (sza_p < 0.000000001) return 0.0;
    double Gamma_v = GORT_PI * c.rr * secv;
    double D = c.r * (1.0 / tan(sza_p / 2.0));
    double lg = c.lambda * Gamma_v;
    return (lg) / (lg + (c.h2 - c.h1) / D) * (1.0 - exp(-lg - (c.h2 - c.h1) / D)) / (1.0 - exp(-lg));
}

struct Pass { double f, F, Kg; };
struct PassA { double Kg, F, M, Gamma_c; };   // the part of a pass that does not need CrownLite

// gortt_kg + first half of gortt_kc_fFbeta (gortt_brdf.c:7-20, :171-194) for one relative azimuth
__device__ __forceinline__ PassA kc_pass_a(const Canopy& c, const Primed& P, double cr, double sr)
{
    const Trig& t = P.t;
    PassA o;
    double overlap = overlap_fn(c, t, cr, sr);
    o.Kg = kg_from_overlap(c, t, overlap);
    double phase_prime = t.cv * t.cs + t.sv * t.ss * cr;
    double Gamma = GORT_PI * c.rr * (t.secs + t.secv - overlap);
    o.Gamma_c = GORT_PI * c.rr * t.secv * 0.5 * (1.0 + phase_prime);
    o.F = o.Gamma_c / Gamma;
    o.M = 1.0 - (1.0 - o.Kg) / (c.lambda * Gamma);
    return o;
}

// second half of gortt_kc_fFbeta (gortt_brdf.c:195-238)
__device__ __forceinline__ Pass kc_pass_b(const Primed& P, const PassA& a, const CrownLite& s, bool view_gt_sun,
                                          double raa, double cr)
{
    Pass o;
    o.Kg = a.Kg; o.F = a.F;
    double PiMi = (1 - cos(s.theta_Mi * (1 - (P.sza_p - P.vza_p * cr) / GORT_PI))) / 2.0;
    double PvMv = s.Mv - (1.0 - cos(P.vza_p * cr - P.sza_p)) / 2.0;
    double Po;
    if ((raa < dtor(270.)) && (raa > dtor(90.))) Po = PvMv;
    else if (view_gt_sun) Po = PiMi;
    else Po = PvMv;
    o.f = a.F * (1.0 - s.Gamma_v * (PvMv + PiMi - Po) / a.Gamma_c) / (1.0 - a.M);
    return o;
}

__device__ __forceinline__ Pass kc_pass(const Canopy& c, const Primed& P, const CrownLite& s, bool view_gt_sun,
                                        double raa, double cr, double sr)
{
    return kc_pass_b(P, kc_pass_a(c, P, cr, sr), s, view_gt_sun, raa, cr);
}

struct Hot { double kuusk, pn0_s, pe_s; };

// gortt_set_zenith_dependant_probabilities (gortt.c:872-915) + gortt_kuusk (gortt_brdf.c:638-702; uses the
// TRUE zeniths, k = k_vza = 0.5)
__device__ __forceinline__ Hot hotspot(const Canopy& c, const double* __restrict__ lut_m, double vza, double sza, double cr)
{
    Hot o;
    double pn0_v, pe_v;
    zenith_lerp(lut_m, sza, o.pn0_s, o.pe_s);
    zenith_lerp(lut_m, vza, pn0_v, pe_v);
    double ssz, csz, svz, cvz;
    sincos(sza, &ssz, &csz);
    sincos(vza, &svz, &cvz);
    double cos_xi = csz * cvz + ssz * svz * cr;
    double lsza = -log(o.pe_s) / c.kfavd;
    double lvza = -log(pe_v) / c.kfavd;
    double arg = lsza * lsza + lvza * lvza - 2. * lsza * lvza * cos_xi;
    double t1, t2;
    if (arg > 0.0) {
        double lsv = sqrt(arg);
        t2 = (1.0 - exp(-lsv / c.r)) / (lsv / c.r);
    } else {
        t2 = 1.0;
    }
    if ((lsza * lvza) > 0.0) t1 = sqrt(lsza * lvza);
    else t1 = 0.0;
    double H = exp(c.kfavd * t1 * t2);
    o.kuusk = o.pe_s * pe_v * H;
    return o;
}

struct Tail { double e_v, e_s, t0, beta; };

// exp terms of gortt.c:439-449 and gortt_brdf.c:534, and the mutual-shadowing beta
__device__ __forceinline__ Tail tail_terms(const Canopy& c, const Primed& P, const gort_options& opt)
{
    Tail o;
    o.e_v = exp(-(c.lambda * GORT_PI * c.rr) / P.t.cv);
    o.e_s = exp(-(c.lambda * GORT_PI * c.rr) / P.t.cs);
    o.t0 = exp(-(0.5 * c.elai * P.t.secs));
    o.beta = opt.use_beta ? opt.beta : crown_beta(c, P.sza_p, P.t.secv);
    return o;
}

// gortt_kc (gortt_brdf.c:118-169) + gortt.c:439-449 + the regrouped view coefficients
__device__ __forceinline__ GeomRec geom_combine(const Canopy& c, const Primed& P, const Pass& a, double f0F0,
                                                double f180F180, const Tail& tl, const Hot& h, double raa, double fd)
{
    GeomRec o;
    double frac = raa / GORT_PI;
    if (frac > 1.0) frac = 2.0 - frac;
    double f = (1. - frac) * f0F0 + frac * f180F180;
    f = tl.beta * f + (1.0 - tl.beta) * a.F;
    double Kg = a.Kg;
    double Kc = f * (1.0 - Kg);
    double Kz = tl.e_v - Kg;
    double Kt = 1.0 - Kc - Kz - Kg;
    Kt = GORT_MAX(0.0, Kt);
    double Kpg = tl.e_s - Kg;
    double Kpz = 1.0 - tl.e_v - Kpg;
    o.Kc = Kc; o.Kg = Kg; o.Kt = Kt; o.Kz = Kz; o.Kpg = Kpg; o.Kpz = Kpz;
    o.fd = fd;
    o.mus = P.t.cs;
    o.q = h.kuusk / (2.0 * P.t.cs * P.t.cv);
    o.tp0 = h.pn0_s + h.pe_s;
    o.pe_s = h.pe_s;
    o.t0 = tl.t0;
    o.pn0_s = h.pn0_s;
    double kf = Kc * fd;
    o.cA = kf * o.q;
    double kfe = kf * c.k_openep;
    o.cG = kfe * Kpg + Kg;
    o.cZ = kfe * Kpz + Kz;
    return o;
}

// Everything wavelength-independent for one line, all roles on one thread.  vza/sza/raa in radians,
// already normalised.
__device__ __forceinline__ GeomRec geom_record(const Canopy& c, const double* __restrict__ lut_m,
                                               const gort_options& opt, double vza, double sza, double raa,
                                               double fd)
{
    const Primed P = primed_trig(c, vza, sza);
    const CrownLite s = crown_lite(c, P.t);
    const bool vgs = fabs(vza) > fabs(sza);
    double sr, cr;
    sincos(raa, &sr, &cr);
    const Pass a = kc_pass(c, P, s, vgs, raa, cr, sr);
    const Pass a0 = kc_pass(c, P, s, vgs, 0.0, 1.0, 0.0);
    const Pass a180 = kc_pass(c, P, s, vgs, GORT_PI, -1.0, GORT_SIN_PI);
    const Tail tl = tail_terms(c, P, opt);
    const Hot h = hotspot(c, lut_m, vza, sza, cr);
    return geom_combine(c, P, a, a0.f * a0.F, a180.f * a180.F, tl, h, raa, fd);
}

// ---- the per-wavelength loop (gortt.c:460-567) split by what each term depends on -------------
// (set, wavelength) only
struct LeafTerms {
    double omega, gam, Tff, Rff, pff, tff, tpff, A, rs, Xf, Zf;
};
// + sun zenith (and fd)
struct SunTerms {
    double G, Z, T, PD, FCf;   // PD = p_df + CdCG ; FCf = (1-fd)*Cf
    double PDF;                // fd*PD + FCf: the crown signature without its hotspot and ground-coupling parts
};

__device__ __forceinline__ LeafTerms leaf_terms(const Canopy& c, double rleaf, double tleaf, double rsoil)
{
    LeafTerms L;
    L.omega = rleaf + tleaf;                                   // gortt.c:469
    L.gam = sqrt(1 - L.omega);                                 // gortt.c:470
    L.rs = rsoil;
    L.Tff = exp(-(2.0 * L.gam * 0.5 * c.elai));                // gortt_brdf.c:492
    L.Rff = fdiv(1.0 - L.gam, 1.0 + L.gam);                    // :574
    double den = 1. - (L.Tff * L.Rff) * (L.Tff * L.Rff);       // :403, :512
    L.pff = fdiv(L.Rff * (1. - L.Tff * L.Tff), den);               // :510-512
    L.tff = fdiv(L.Tff * (1. - L.Rff * L.Rff), den);               // :401-403
    double K = c.k_open + c.k_openep;                          // :381
    L.tpff = L.tff * (1.0 - K) + K;                            // :382
    double gfunc = fdiv(-(4.0 / 9.0) * (rleaf - tleaf), L.omega);   // :591
    L.A = (1.0 - L.omega) * L.omega * (1.0 - gfunc);           // gortt.c:504-506 without kuusk
    L.Xf = fdiv(rsoil, 1.0 - rsoil * L.pff) * (L.tpff - c.k_open);   // gortt.c:520-521
    L.Zf = (L.tpff - c.k_openep) * rsoil;                      // gortt.c:492
    return L;
}

__device__ __forceinline__ SunTerms sun_terms(const Canopy& c, const LeafTerms& L, double fd, double mus,
                                              double t0, double tp0, double pe_s)
{
    SunTerms S;
    double two_mu_g = 2.0 * mus * L.gam;
    double Rdf = fdiv(1.0 - L.gam, 1.0 + two_mu_g);                                  // gortt_brdf.c:552
    double Tdf = (L.omega / 2.0) * fdiv(1. + 2. * mus, 1. - two_mu_g * two_mu_g) * (L.Tff - t0);   // :467-471
    double SS = t0 * Rdf + Tdf * L.Rff;
    double tdf = Tdf - L.pff * SS;                                                   // :423-424
    double pdf = Rdf - L.tff * SS;                                                   // :628-630
    double tpdf = tdf * (1 - tp0);                                                   // :361
    double omf = 1 - fd;
    S.G = fd * L.rs + omf * L.rs;                                                    // gortt.c:481-484
    double Zd = (tpdf + pe_s) * L.rs;                                                // gortt.c:491
    S.Z = fd * Zd + omf * L.Zf;                                                      // gortt.c:494
    double K = c.k_open + c.k_openep;
    double CfG = (K * S.G + (1 - K) * S.Z) * c.k_openep;                             // gortt.c:516-517
    double CdCG = (tpdf + tp0) * L.Xf;                                               // gortt.c:519-521
    double CfCG = L.tpff * L.Xf;                                                     // gortt.c:523-525
    double Cf = L.pff + CfG + CfCG;                                                  // gortt.c:512,529
    S.T = fd * CdCG + omf * CfCG;                                                    // gortt.c:541-550
    S.PD = pdf + CdCG;
    S.FCf = omf * Cf;
    S.PDF = fd * S.PD + S.FCf;
    return S;
}

// the only part that depends on the view direction: 9 FP64 instructions
__device__ __forceinline__ double view_rsurf(const Canopy& c, const LeafTerms& L, const SunTerms& S,
                                             double fd, double q, double Kc, double Kg, double Kt, double Kz,
                                             double Kpg, double Kpz, double& C_out)
{
    double zg = fma(S.G, Kpg, S.Z * Kpz);                    // Z*K'z + G*K'g          gortt.c:514
    double Cd = fma(L.A, q, S.PD);                           // CdC + CdCG             gortt.c:504-507
    Cd = fma(c.k_openep, zg, Cd);                            // + CdG                  gortt.c:528
    double C = fma(fd, Cd, S.FCf);                           // gortt.c:531
    C_out = C;
    return fma(Kz, S.Z, fma(Kt, S.T, fma(Kg, S.G, Kc * C))); // gortt.c:557
}

// ---- forward-mode tangent with respect to favd (gort_brdf_tangent_batch_dev) --------------------------------------
// favd enters the BRDF through elai, kfavd and the LUT record (epgap rows, k_openep); dlut is the record's tangent.
// Everything else of the record (Kc, Kg, Kt, Kz, K'g, K'z, fd, mus) does not depend on it.  At the few kinks the
// derivative is that of the branch the forward computation takes.

// d elai / d favd: elai without its favd factor (gortt.c:657)
__device__ __forceinline__ double elai_tangent(const Canopy& c)
{
    return (1.333333) * c.lambda * GORT_PI * c.ellip * (c.rr * c.r);
}

// tangents of the Kuusk hotspot (gortt_brdf.c:638-702) and of the sun-side LUT interpolation; the forward values are
// formed again exactly as hotspot() forms them, so every branch is the forward's
struct HotTan { double dkuusk, dpn0_s, dpe_s; };
__device__ __forceinline__ HotTan hotspot_tangent(const Canopy& c, const double* __restrict__ lut_m,
                                                  const double* __restrict__ dlut_m, double vza, double sza, double cr)
{
    HotTan o;
    double pn0_s, pe_s, pn0_v, pe_v, dpn0_v, dpe_v;
    zenith_lerp(lut_m, sza, pn0_s, pe_s);
    zenith_lerp(lut_m, vza, pn0_v, pe_v);
    zenith_lerp(dlut_m, sza, o.dpn0_s, o.dpe_s);          // zenith_lerp is linear in the rows
    zenith_lerp(dlut_m, vza, dpn0_v, dpe_v);
    double ssz, csz, svz, cvz;
    sincos(sza, &ssz, &csz);
    sincos(vza, &svz, &cvz);
    const double cos_xi = csz * cvz + ssz * svz * cr;
    const double dk = 0.5;                                 // d kfavd / d favd
    const double lsza = -log(pe_s) / c.kfavd;
    const double lvza = -log(pe_v) / c.kfavd;
    const double dlsza = (-(o.dpe_s / pe_s) - lsza * dk) / c.kfavd;
    const double dlvza = (-(dpe_v / pe_v) - lvza * dk) / c.kfavd;
    const double arg = lsza * lsza + lvza * lvza - 2. * lsza * lvza * cos_xi;
    double t1, t2, dt1 = 0.0, dt2 = 0.0;
    if (arg > 0.0) {
        const double lsv = sqrt(arg);
        const double darg = 2.0 * (lsza * dlsza + lvza * dlvza - cos_xi * (dlsza * lvza + lsza * dlvza));
        const double x = lsv / c.r, ex = exp(-x);
        t2 = (1.0 - ex) / x;
        dt2 = (ex - t2) / x * (darg / (2.0 * lsv) / c.r);   // d/dx (1 - e^-x)/x = (e^-x - t2)/x
    } else {
        t2 = 1.0;
    }
    if ((lsza * lvza) > 0.0) {
        t1 = sqrt(lsza * lvza);
        dt1 = (dlsza * lvza + lsza * dlvza) / (2.0 * t1);
    } else {
        t1 = 0.0;
    }
    const double H = exp(c.kfavd * t1 * t2);
    const double dH = H * (dk * t1 * t2 + c.kfavd * (dt1 * t2 + t1 * dt2));
    o.dkuusk = (o.dpe_s * pe_v + pe_s * dpe_v) * H + pe_s * pe_v * dH;
    return o;
}

// tangents of the (set, lambda) terms; dkoe = d k_openep / d favd (k_open has none)
struct LeafTan { double dTff, dpff, dtff, dtpff, dXf, dZf; };
__device__ __forceinline__ LeafTan leaf_tangent(const Canopy& c, const LeafTerms& L, double delai, double dkoe)
{
    LeafTan D;
    D.dTff = -(L.gam * delai) * L.Tff;
    const double tr = L.Tff * L.Rff;
    const double den = 1. - tr * tr;
    const double dden = -2.0 * tr * L.Rff * D.dTff;
    D.dpff = fdiv(-2.0 * L.Rff * L.Tff * D.dTff - L.pff * dden, den);
    D.dtff = fdiv(D.dTff * (1. - L.Rff * L.Rff) - L.tff * dden, den);
    const double K = c.k_open + c.k_openep;
    D.dtpff = D.dtff * (1.0 - K) + (1.0 - L.tff) * dkoe;
    const double u = fdiv(L.rs, 1.0 - L.rs * L.pff);
    D.dXf = (u * u * D.dpff) * (L.tpff - c.k_open) + u * D.dtpff;
    D.dZf = (D.dtpff - dkoe) * L.rs;
    return D;
}

// the (sun, lambda) terms the tangent evaluation needs: G and Z, and the tangents of Z, PDF and T (sun_terms' chain)
struct SunTan { double G, Z, dZ, dPDF, dT; };
__device__ __forceinline__ SunTan sun_tangent(const Canopy& c, const LeafTerms& L, const LeafTan& D, double dkoe,
                                              double fd, double mus, double t0, double tp0, double pe_s,
                                              double dt0, double dtp0, double dpe_s)
{
    SunTan O;
    const double two_mu_g = 2.0 * mus * L.gam;
    const double Rdf = fdiv(1.0 - L.gam, 1.0 + two_mu_g);
    const double cT = (L.omega / 2.0) * fdiv(1. + 2. * mus, 1. - two_mu_g * two_mu_g);
    const double Tdf = cT * (L.Tff - t0), dTdf = cT * (D.dTff - dt0);
    const double SS = t0 * Rdf + Tdf * L.Rff, dSS = dt0 * Rdf + dTdf * L.Rff;
    const double tdf = Tdf - L.pff * SS, dtdf = dTdf - D.dpff * SS - L.pff * dSS;
    const double dpdf = -(D.dtff * SS + L.tff * dSS);
    const double tpdf = tdf * (1 - tp0), dtpdf = dtdf * (1 - tp0) - tdf * dtp0;
    const double omf = 1 - fd;
    O.G = fd * L.rs + omf * L.rs;
    O.Z = fd * ((tpdf + pe_s) * L.rs) + omf * L.Zf;
    O.dZ = fd * ((dtpdf + dpe_s) * L.rs) + omf * D.dZf;
    const double K = c.k_open + c.k_openep;
    const double dCfG = (dkoe * (O.G - O.Z) + (1 - K) * O.dZ) * c.k_openep + (K * O.G + (1 - K) * O.Z) * dkoe;
    const double dCdCG = (dtpdf + dtp0) * L.Xf + (tpdf + tp0) * D.dXf;
    const double dCfCG = D.dtpff * L.Xf + L.tpff * D.dXf;
    O.dT = fd * dCdCG + omf * dCfCG;
    O.dPDF = fd * (dpdf + dCdCG) + omf * (D.dpff + dCfG + dCfCG);
    return O;
}

}  // namespace gort
