// gort_lut.cu -- KOpen / P(n) gap-probability LUT generation (sm_100a, FP64, -fmad=false).
//
// Replaces gortt_init_params (gortt.c:632-868) + gortt_gap_probabilities
// (gortt_pn_kopen.c:7-129 and everything it calls, :134-924, :1083-1140) and
// gortt_gap_probabilities_Q08 (gortt_pn_kopen.c:1144-1200), restricted to what reaches the
// outputs (SURVEY.md 3.3): p_n0[0][t], epgap[0][t], k_open[0], k_openep[0].  The reference's
// vb / fb / t_open / dt_open / dk_open tables are never read by the BRDF or albedo path and are
// not computed.
//
// Mapping: one CTA per canopy parameter set, one thread per zenith index t (91 of 96 lanes):
//   v_g[h][t] -> p_n0[h][t] (15 layers)  ->  p_s0  ->  E[S]  ->  for every entry height sp_i and
//   crown count n: P(n | s'), within-crown path s and its histogram bin  ->  epgap[0][t];
//   thread 0 then runs the trapezoid rule over theta in the reference's order.
// The path-length histogram pd_s[0][t][bin] is not materialised: epgap[0][t] = sum over bins of
// exp(-s_bin tau') pd_s[bin] is accumulated entry by entry with the entry's bin index, which is
// the same sum in a different association (differences ~1e-16 relative).
//
// Code size matters here: with everything inlined and the Simpson loops unrolled the kernel was 18 000 SASS
// instructions and its top stall was instruction fetch (stall_no_instruction ~70 % of samples in the geometry
// code, ncu profiles/r1_lut).  The geometry helpers are therefore __noinline__ and their loops not unrolled.
//
// Parity hazards honoured (SURVEY.md App. B1-B3): no FMA contraction (r*r - h2*h2 must be exactly
// 0 when h2 == r), running-sum loop counters (z += dz_p, h += dh), (int)(s/ds + 0.5) binning,
// the |a3| < 1e-10 clamp, float-typed Simpson factors.
#include "gort_device.cuh"
#include "gort_internal.h"

namespace gort {

#define LUT_THREADS 96
#define LUT_MAXCROWNS 30
#define LUT_NH_ES 20
#define LUT_NOINT 20

struct Crown {
    double r, rr, rrr;
    double h1_p, h2_p, z2_p, dz_p, ds, lv_p, tau_p;
};

struct Ang {            // trig of one theta_p
    double th, s, c, t;  // angle, sin, cos, tan
};

// gortt_pn_kopen.c:285-305
__device__ __forceinline__ double left_circle_area(double r, double x_cut)
{
    double area_tot = GORT_PI * r * r;
    double ang_sector = acos(fabs(x_cut) / r) * 2.0;
    double area_sector = area_tot * ang_sector / (2.0 * GORT_PI);
    double area_triangle = fabs(x_cut) * sqrt(r * r - x_cut * x_cut);
    if (x_cut > 0.0) return area_tot - (area_sector - area_triangle);
    return area_sector - area_triangle;
}

// gortt_pn_kopen.c:309-323
__device__ __forceinline__ double right_ellipse_area(double r, double b, double x_cut)
{
    double x_cut_p = x_cut / (b / r);
    double a_p = GORT_PI * r * r;
    a_p -= left_circle_area(r, x_cut_p);
    return a_p * (b / r);
}

// gortt_pn_kopen.c:170-229 with the "weird" section :233-282 inlined
// (scalars by value: a noinline function taking the Crown / Ang structs by reference forces them into local memory --
// ncu counted 292 MB of DRAM writes for an 82 MB result in the tube kernel)
__device__ __noinline__ double cross_section_v(double r, double rr, double as, double ac, double at, double h, double z)
{
    if (z < h - r) return 0.0;
    double h_low = h - r * as;
    double h_high = h + r * as;
    if (z <= h_low) {
        double q = rr - (h - z) * (h - z);
        double r_p = (q <= 0) ? 0 : sqrt(q);
        return GORT_PI * r_p * r_p;
    } else if (z > h_low && z < h_high) {
        double zdiff = h - z;
        double r_p = sqrt(rr - zdiff * zdiff);
        double x_cc = zdiff * at;
        double x_p = x_cc / (1.0 - ac * ac);
        double a_cp = left_circle_area(r_p, x_p - x_cc);
        double a_ep = right_ellipse_area(r, r * (1.0 / ac), x_p);
        return a_cp + a_ep;
    }
    return GORT_PI * rr * (1.0 / ac);
}
__device__ __forceinline__ double cross_section(const Crown& c, const Ang& a, double h, double z)
{
    return cross_section_v(c.r, c.rr, a.s, a.c, a.t, h, z);
}

// gortt_pn_kopen.c:149-167
__device__ __forceinline__ double proj_volume(const Crown& c, const Ang& a, double h)
{
    double vol = 0.0;
    int guard = 0;
    for (double z = c.h1_p + c.dz_p / 2.0; z <= c.h2_p && guard < 100000; z += c.dz_p, guard++)
        vol += cross_section(c, a, h, z) * (c.dz_p);
    return vol;
}

// sqrt for the Simpson integrand (the call site was 18 % of the LUT path's instructions): MUFU.RSQ64H seed (2^-22) and
// ONE coupled third-order Newton step on the reciprocal root, y (1 + e/2 + 3 e^2/8) with e = 1 - x y^2: the remaining
// error is O(e^3) ~ 2^-66, so x * y is the root to within 2 ULP.  CUDA's IEEE sqrt adds a correction step, a range
// check, a slow-path call and a reconvergence barrier (17 SASS instructions against 7); the integrand feeds a 41-point
// quadrature whose result weights the crown-count terms smoothly, so 2 ULP here move epgap by ~1e-16.
// Valid for x == 0 and normal x well inside the exponent range (here 0 or [1e-10, r^2]); negative x gives NaN.
__device__ __forceinline__ double sqrt_lite(double x)
{
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(x, -(y * y), 1.0);
    const double y1 = fma(fma(e, 0.375, 0.5), y * e, y);
    return x == 0.0 ? 0.0 : x * y1;
}
// the same with the reference's clamp (gortt_pn_kopen.c:867: |a3| < 1e-10 -> 0) folded into the final select.  The
// comparison is made on the bit pattern (|x| < 1e-10 exactly, NaN compares false as in the reference): integer ALU
// instead of one more instruction on the FP64 pipe, which is what bounds lut_tube_kernel.
__device__ __forceinline__ double sqrt_clamped(double x)
{
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(x, -(y * y), 1.0);
    const double y1 = fma(fma(e, 0.375, 0.5), y * e, y);
    const unsigned hi = (unsigned) __double2hiint(x) & 0x7fffffffu, lo = (unsigned) __double2loint(x);
    const bool tiny = hi < 0x3DDB7CDFu || (hi == 0x3DDB7CDFu && lo < 0xD9D7BDBBu);       // |x| < 1e-10 = 0x3DDB7CDFD9D7BDBB
    return tiny ? 0.0 : x * y1;
}

__constant__ double c_simpson_index[2 * LUT_NOINT] = {
    0.0, 1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0, 8.0, 9.0, 10.0, 11.0, 12.0, 13.0, 14.0, 15.0, 16.0, 17.0, 18.0, 19.0,
    20.0, 21.0, 22.0, 23.0, 24.0, 25.0, 26.0, 27.0, 28.0, 29.0, 30.0, 31.0, 32.0, 33.0, 34.0, 35.0, 36.0, 37.0, 38.0, 39.0};

// gortt_pn_kopen.c:858-872, as the reference writes it (used for the two end points)
__device__ __forceinline__ double triang_fcn(double x, double b, double r, double tan_the)
{
    double a1 = tan_the * (x - b);
    double a2 = r * r - x * x;
    double a3 = a2 - a1 * a1;
    if (fabs(a3) < 0.0000000001) a3 = 0.0;
    return 2.0 * a1 * sqrt_lite(a3);
}

// gortt_pn_kopen.c:811-854: Simpson's rule with 2 x 20 intervals over x in [b, x0] of
//        f(x) = 2 tan(th) (x - b) sqrt(r^2 - x^2 - tan^2(th) (x - b)^2).
// At the sample points x = b + i h the radicand is a quadratic in i,
//        a3(i) = (r^2 - b^2) - 2 b h i - (1 + tan^2) h^2 i^2,
// evaluated by Horner's rule (2 FMAs instead of the reference's 6 unfused operations; the absolute error stays
// ~1e-16 r^2 as in the reference's own form, and the |a3| < 1e-10 clamp of :867 is applied to it the same way), and
// f = (2 tan h i) sqrt(a3).  The reference's (double)(float) loop factors are small integers, exact in either type.
__device__ __noinline__ double triang(double b, double r, double sint, double cost, double tant)
{
    double a1 = r * r - b * b * sint * sint;
    double x0 = b * (sint * sint) + sqrt(a1) * cost;
    const int m = LUT_NOINT;
    double h = .50 * (x0 - b) / (double) (float) m;
    const double c0 = r * r - b * b, c1 = -2.0 * b * h, c2 = -(1.0 + tant * tant) * (h * h), d = 2.0 * tant * h;
    // f(x_i) = (d i) sqrt(a3(i)): the factor d is taken out of the two sums (one FMA per point instead of two
    // multiplications and an addition) and the sample indices come from a constant table instead of a running FP64 sum.
    double sum1 = 0.0, sum2 = 0.0;
#pragma unroll 2
    for (int i = 0; i < m - 1; i++) {
        const double f = c_simpson_index[2 * i + 1], g = c_simpson_index[2 * i + 2];
        sum1 = fma(f, sqrt_clamped(fma(fma(c2, f, c1), f, c0)), sum1);   // odd points 1, 3, .., 37
        sum2 = fma(g, sqrt_clamped(fma(fma(c2, g, c1), g, c0)), sum2);   // even points 2, 4, .., 38
    }
    {
        const double f = c_simpson_index[2 * m - 1];
        sum1 = fma(f, sqrt_clamped(fma(fma(c2, f, c1), f, c0)), sum1);   // point 39
    }
    double volume = d * fma(4.0, sum1, 2.0 * sum2);
    volume += triang_fcn(x0, b, r, tant);
    volume += triang_fcn(b, b, r, tant);
    volume *= h / 3.0;
    return volume;
}

// gortt_pn_kopen.c:796-806
__device__ __forceinline__ double sector(double a1, double a2, double r)
{
    double b1 = r * r * a1 - (a1 * a1 * a1) / 3.0;
    double b2 = r * r * a2 - (a2 * a2 * a2) / 3.0;
    return GORT_PI * (b2 - b1) / 2.0;
}

// gortt_pn_kopen.c:771-792
__device__ __forceinline__ double trisec(double hh, double hh_b, const Ang& a, double r)
{
    double tmp = (hh - hh_b);
    double x = -1.0 * tmp * a.s + sqrt(r * r - tmp * tmp) * a.c;
    double b = -tmp / a.s;
    return triang(b, r, a.s, a.c, a.t) + sector(x, r, r);
}

// gortt_pn_kopen.c:876-886
__device__ __forceinline__ double cylind_fcn(double x, double r)
{
    return .50 * x * sqrt(r * r - x * x) + .50 * r * r * asin(x / r);
}

// gortt_pn_kopen.c:891-924
__device__ __noinline__ double cylind(double r, double h1, double h2, double h)
{
    double slope = h / (h2 - h1);
    double tmp1 = sqrt(r * r - h1 * h1);
    double tmp2 = sqrt(r * r - h2 * h2);
    double volume = tmp1 * tmp1 * tmp1 - tmp2 * tmp2 * tmp2;
    volume /= 3.0;
    volume -= h1 * (cylind_fcn(h2, r) - cylind_fcn(h1, r));
    volume *= 2.0 * slope;
    if (h2 < r) {
        double phi = acos(h2 / r);
        double s1 = r * r * phi;
        double s2 = r * sin(phi) * h2;
        volume += (s1 - s2) * h;
    }
    return volume;
}

// gortt_cylind (gortt_pn_kopen.c:891-924) called with h2 == r, as both call sites that are live for h = 0 do (:702,
// :743).  Then, with the unfused arithmetic this file is compiled with, r*r - h2*h2 is exactly 0 (App. B1), so
// tmp2 = 0, cylind_fcn(h2, r) = 0 + .5 r^2 asin(1) and the h2 < r tail is skipped: two square roots, one asin and one
// division fewer than the general routine, same value.
__device__ __forceinline__ double cylind_to_r(double r, double h1, double h)
{
    double slope = h / (r - h1);
    double tmp1 = sqrt(r * r - h1 * h1);
    double volume = tmp1 * tmp1 * tmp1 - 0.0;
    volume /= 3.0;
    volume -= h1 * ((.50 * r * 0.0 + .50 * r * r * asin(1.0)) - cylind_fcn(h1, r));
    volume *= 2.0 * slope;
    return volume;
}

// gortt_pn_kopen.c:665-768; hp_h = height_p[h], hp_s = height_p[h_s]
__device__ __forceinline__ double tube_vol(const Crown& c, const Ang& a, double hp_h, double hp_s, double h_b)
{
    const double r = c.r;
    double V, V_sp1, V_sp2, V_cyln, h_t, h_tt;
    double tmp_s = (hp_s - hp_h) / a.c;
    double V_0 = GORT_PI * c.rr * tmp_s;
    V_0 += (4.0 / 3.0) * GORT_PI * c.rrr;

    if ((hp_h - r) >= h_b) {
        V = 0.0;
    } else if ((hp_h - r * a.s) >= h_b) {
        h_t = r - (hp_h - h_b);
        V = (GORT_PI / 3.0) * h_t * h_t * (3.0 * r - h_t);
    } else if ((hp_h + r * a.s) >= h_b) {
        V_sp1 = (2.0 / 3.0) * GORT_PI * c.rrr;
        V_sp1 -= trisec(hp_h, h_b, a, r);
        h_tt = (h_b - (hp_h - r * a.s)) / a.c;
        if (hp_s - r * a.s >= h_b) {
            double hh1 = (hp_h - h_b) / a.s;
            V_cyln = cylind(r, hh1, r, h_tt);
            V_sp2 = 0.0;
        } else {
            double hh1 = (hp_h - h_b) / a.s;
            double hh2 = (hp_s - h_b) / a.s;
            double hh = (hp_s - hp_h) / a.c;
            V_cyln = cylind(r, hh1, hh2, hh);
            V_sp2 = trisec(h_b, hp_s, a, r);
        }
        V = V_sp1 + V_cyln + V_sp2;
    } else if (hp_s - r * a.s >= h_b) {
        double tmp_h = (h_b - hp_h) / a.c;
        V_cyln = GORT_PI * r * r * tmp_h;
        V_sp1 = (2.0 / 3.0) * GORT_PI * c.rrr;
        V = V_sp1 + V_cyln;
    } else if (hp_s + r * a.s >= h_b) {
        h_tt = (hp_s + r * a.s - h_b) / a.c;
        double hh1 = (h_b - hp_s) / a.s;
        double tmp_h = (hp_s - hp_h) / a.c;
        V_cyln = GORT_PI * r * r * tmp_h - cylind_to_r(r, hh1, h_tt);
        V_sp2 = trisec(h_b, hp_s, a, r);
        V_sp1 = (2.0 / 3.0) * GORT_PI * c.rrr;
        V = V_cyln + V_sp2 + V_sp1;
    } else if (hp_s + r >= h_b) {
        h_t = r - (h_b - hp_s);
        V_sp1 = (GORT_PI / 3.0) * h_t * h_t * (3.0 * r - h_t);
        V = V_0 - V_sp1;
    } else {
        V = V_0;
    }
    return V;
}

// gortt_pn_kopen.c:566-645; hz = height_p[z]
__device__ __forceinline__ double mean_single_crown_path(const Crown& c, const Ang& a, double hz, double h)
{
    if (hz > h + c.r - 0.0001) return 0.0;
    if (hz < h - c.r + 0.0001) return 4.0 * c.r / 3.0;
    double V_sphere = 4.0 * GORT_PI * c.rrr / 3.0;
    double zdiff = fabs(h - hz);
    double ht = c.r - zdiff;
    double V_slice = GORT_PI * ht * ht / 3.0 * (3.0 * c.r - ht);
    double V_tot = (hz > h) ? V_slice : V_sphere - V_slice;
    V_tot /= a.c;
    double proj_area;
    if (h < hz) proj_area = cross_section(c, a, h, (h - zdiff));
    else proj_area = cross_section(c, a, h, (h + zdiff));
    return V_tot / proj_area;
}

// gortt_pn_kopen.c:534-563
__device__ __forceinline__ double expected_single_crown_path(const Crown& c, const Ang& a, double hz)
{
    double ES = 0.0;
    double dh = (c.h2_p - c.h1_p) / (double) LUT_NH_ES;
    int guard = 0;
    for (double h = c.h1_p + dh / 2.0; h <= c.h2_p && guard < 100000; h += dh, guard++)
        ES += mean_single_crown_path(c, a, hz, h) * ((1.0 / (c.h2_p - c.h1_p)) * dh);
    return ES;
}

// ------------------------------------------------------------------------------------------------------------------
// The full gap-probability path as a PIPELINE OF FLAT KERNELS (round 2).
//
// The reference's nest is  zenith t (91) x entry height sp_i (13) x crown count n (30)  (gortt_pn_kopen.c:457-527)
// behind a shape-only geometry phase (cross-sections :149-323, tube volumes :665-924).  Round 1 ran all of it in one
// kernel, one thread per zenith: 96 registers, 3 warps per CTA, 22.7 % of the warp slots, FP64 pipe 45 % busy, 78 KB of
// code executed by warps in different phases (instruction-fetch stalls), 98 % of the EnKF member update.  A first
// restructuring inside one kernel (entry heights dealt to four thread rows) stayed barrier- and fetch-bound (ncu:
// 2.6 barrier-stalled and 1.0 fetch-stalled warps per issue).  Now every phase is its own small kernel in which a WARP
// is one (item, 32 consecutive zeniths) pair -- neighbouring zeniths take the same branches of the sphere / cylinder
// geometry -- every warp of a CTA does the same amount of work, and the per-zenith arrays travel through HBM / L2
// (24.5 KB per crown shape, ~1 ms per 10^5 shapes, against ~20 ms of arithmetic):
//
//   lut_plan_kernel     per set: head of its shape group (consecutive sets sharing r, b, h1, h2 bit for bit, capped),
//                       head and size of its sub-group (group members that also share the stem density, <= LUT_SUB)
//   lut_prep_kernel     per (shape, zenith): theta', its sin / cos / tan, E[S]                   gortt.c:783-797, :534-563
//   lut_vg_kernel       per (shape, zenith third): warp = cross-section j, then warp = layer h   gortt_pn_kopen.c:24-32, :149-323
//   lut_tube_kernel     per (shape, zenith third): warp = entry height: tube-volume difference   :496, :665-924
//   lut_crown_kernel    per (sub-group, zenith third): warp = entry height: the crown-count loop :489-527, once per
//                       sub-group; per member only the within-crown gap sums; 13 partial sums added in a fixed order
//   kopen_kernel        per set: trapezoid rule over the 91 zeniths                              :351-375
//
// Shape groups and sub-groups keep what round 1 introduced: LUT grids and ensembles that vary stem density / leaf
// area over fixed crown shapes (BASELINE.json configs 4a and 5) pay the geometry once per group and the crown-count
// loop once per sub-group.  The bin attenuation exp(-s_bin tau') of gortt_calc_epgap (:1110-1114) depends on (set, bin)
// only -- not on zenith, entry height or crown count -- so it is tabulated once per member and zenith third (LUT_TAB
// bins, one exp each, the literal formula) instead of being evaluated at every change of bin inside the crown-count
// loop (~10 exp per (zenith, entry height) before).
// A set gets the same bits alone, inside a group or sub-group, or at a chunk boundary.
#define LUT_GROUP_CAP 64
#define LUT_SUB 8                       // members per sub-group (same shape AND same stem density)
#define LUT_NSP (GORT_NLAYERS - 2)     // entry heights sp_i = 1 .. 13 (sp_i = 14 contributes p_s0 = 0)
#define LUT_ZW 96                       // zenith slots per set in the workspace arrays (3 warps)
#define LUT_TAB 512                     // tabulated bins of exp(-s_bin tau'); bins beyond use the formula directly
#define LUT_NA 32                       // distinct cross-sections per zenith: 14 + K, K < 16
#define LUT_CHUNK 16384                 // sets per pass: bounds the workspace (24.5 KB per set)
// 1/n!, n = 0..30, each the FP64 quotient 1.0 / n! (the reference tabulates n! in gortt.c:752-754 and divides)
__constant__ double c_inv_fact[LUT_MAXCROWNS + 1] = {
    1.0,
    1.0,
    0.5,
    0.16666666666666666,
    0.041666666666666664,
    0.008333333333333333,
    0.001388888888888889,
    0.0001984126984126984,
    2.48015873015873e-05,
    2.7557319223985893e-06,
    2.755731922398589e-07,
    2.505210838544172e-08,
    2.08767569878681e-09,
    1.6059043836821613e-10,
    1.1470745597729725e-11,
    7.647163731819816e-13,
    4.779477332387385e-14,
    2.8114572543455206e-15,
    1.5619206968586225e-16,
    8.22063524662433e-18,
    4.110317623312165e-19,
    1.9572941063391263e-20,
    8.896791392450574e-22,
    3.8681701706306835e-23,
    1.6117375710961184e-24,
    6.446950284384474e-26,
    2.4795962632247972e-27,
    9.183689863795546e-29,
    3.2798892370698385e-30,
    1.1309962886447718e-31,
    3.769987628815906e-33};

// Workspace of one pass (n = sets of the pass), all per set index of the pass; shape-level rows are filled for group
// heads only.
struct LutWork {
    int *head;          // [n]      index of the set's group head
    int *sub;           // [n]      sub-group size if the set is a sub-group head, else 0
    double *trig;       // [n][4][LUT_ZW]    sin, cos, tan of theta', E[S]
    double *vg;         // [n][15][LUT_ZW]   v_g[h][t]
    double *tube;       // [n][13][LUT_ZW]   tube-volume difference per entry height
    double *es_all;     // [n][15][LUT_ZW]   E[S] towards every layer (only the intermediates path, launch_lut_dead)
    double *shp;        // [n][LUT_SHP]      derived crown-shape scalars and the 15 layer heights (seven FP64 divisions per
                        //                   set, done once by lut_plan_kernel instead of by every thread of every kernel)
    // Compact work lists of the pass (lut_plan_kernel; order arbitrary, results do not depend on it), so that the heavy
    // kernels run as persistent CTAs over exactly the items that exist instead of launching one (mostly empty) CTA per
    // set: the C5 grid has one group head per 64 sets and one sub-group head per 8.
    int *hl;            // [n]      group heads
    int *s1;            // [n]      heads of single-member sub-groups
    int *s8;            // [n]      heads of sub-groups of 2 .. LUT_SUB members
    int *cnt;           // [LUT_NCNT]  lengths of hl, s1, s8; then the tickets of the persistent kernels (tube, crown<1>,
                        //             crown<LUT_SUB>): items are handed out in order of request, not by a fixed stride --
                        //             their durations differ (tube length, table size) and a fixed stride left a 10 % tail
};
#define LUT_NCNT 8
#define LUT_SHP 32

__device__ __forceinline__ bool same_shape(const double* __restrict__ st, size_t n, int a, int b)
{
    return st[1 * n + a] == st[1 * n + b] && st[2 * n + a] == st[2 * n + b] &&
           st[3 * n + a] == st[3 * n + b] && st[4 * n + a] == st[4 * n + b];
}

// Crown shape of set m: gortt_init_params, gortt.c:641-697 (the shape-only part) and the layer heights of :778-781
struct Shape { Crown c; double ellip, h1, h2, z2, dz; };
__device__ __forceinline__ Shape shape_compute(const double* __restrict__ structure, size_t N, int m)
{
    Shape S;
    const double r = structure[1 * N + m], b = structure[2 * N + m];
    S.h1 = structure[3 * N + m]; S.h2 = structure[4 * N + m];
    S.ellip = b / r;
    S.c.r = r; S.c.rr = r * r; S.c.rrr = S.c.rr * r;
    const double z1 = S.h1 - r * S.ellip;
    S.z2 = S.h2 + r * S.ellip;
    S.c.z2_p = S.z2 / S.ellip;
    S.c.h1_p = S.h1 / S.ellip;
    S.c.h2_p = S.h2 / S.ellip;
    S.dz = (double) (S.z2 - z1) / ((double) GORT_NLAYERS - 1.0);
    S.c.ds = S.dz;
    S.c.dz_p = S.dz / S.ellip;
    S.c.lv_p = 0.0; S.c.tau_p = 0.0;
    return S;
}
// slots of the per-set shape table
enum { SHP_ELLIP = 0, SHP_R, SHP_H1, SHP_H2, SHP_Z2, SHP_DZ, SHP_Z2P, SHP_H1P, SHP_H2P, SHP_DZP, SHP_HP = 16 };
__device__ __forceinline__ void shape_store(double* __restrict__ o, const Shape& S)
{
    o[SHP_ELLIP] = S.ellip; o[SHP_R] = S.c.r; o[SHP_H1] = S.h1; o[SHP_H2] = S.h2; o[SHP_Z2] = S.z2; o[SHP_DZ] = S.dz;
    o[SHP_Z2P] = S.c.z2_p; o[SHP_H1P] = S.c.h1_p; o[SHP_H2P] = S.c.h2_p; o[SHP_DZP] = S.c.dz_p;
    for (int i = 0; i < GORT_NLAYERS; i++) o[SHP_HP + i] = (S.z2 - S.dz * (double) (GORT_NLAYERS - 1 - i)) / S.ellip;   // height_p[i], gortt.c:778-781
}
__device__ __forceinline__ Shape shape_load(const LutWork& w, int i)
{
    const double* __restrict__ o = w.shp + (size_t) i * LUT_SHP;
    Shape S;
    S.ellip = o[SHP_ELLIP]; S.h1 = o[SHP_H1]; S.h2 = o[SHP_H2]; S.z2 = o[SHP_Z2]; S.dz = o[SHP_DZ];
    const double r = o[SHP_R];
    S.c.r = r; S.c.rr = r * r; S.c.rrr = S.c.rr * r;
    S.c.z2_p = o[SHP_Z2P]; S.c.h1_p = o[SHP_H1P]; S.c.h2_p = o[SHP_H2P];
    S.c.ds = S.dz; S.c.dz_p = o[SHP_DZP];
    S.c.lv_p = 0.0; S.c.tau_p = 0.0;
    return S;
}
// height_p[i] of set i's shape
__device__ __forceinline__ double layer_height_p(const LutWork& w, int i, int layer)
{
    return w.shp[(size_t) i * LUT_SHP + SHP_HP + layer];
}

// Groups and sub-groups, for every pass of a call at once (one launch: the kernel is a serial walk per thread, and one
// launch per 16 384 sets cost 8 x 46 us on the C5 grid).  Set e of the call belongs to pass e / chunk and has index
// i = e % chunk inside it; m0 + e is its global index.  Group boundaries sit at multiples of group_cap of the GLOBAL
// index and at pass boundaries (chunk is a multiple of group_cap), so the partition does not depend on the pass size.
// head[] holds pass-local indices; the work lists and their counters are per pass (w.cnt[4 * pass + ..]).
// One atomic per warp and pass instead of one per set: the lanes that append to the same pass's list are counted by a
// ballot, the first of them reserves the slots.  (With every set a group head, 10^5 atomics on one address cost ~1 ms.)
__device__ __forceinline__ void list_append(bool mine, int pass, int* cnt, int* list, int value)
{
    const unsigned active = __activemask();
    const unsigned same = __match_any_sync(active, pass);          // a warp straddles at most two passes
    const unsigned who = __ballot_sync(active, mine) & same;
    if (!mine) return;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(who) - 1;
    int slot = 0;
    if (lane == leader) slot = atomicAdd(cnt, __popc(who));
    slot = __shfl_sync(who, slot, leader);
    list[slot + __popc(who & ((1u << lane) - 1u))] = value;
}

__global__ void __launch_bounds__(128)
lut_plan_kernel(int n, int m0, int chunk, int group_cap, const double* __restrict__ structure, size_t N, LutWork w)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int c = e / chunk, base = c * chunk;
    const int i = e - base;
    const int n_pass = min(chunk, n - base);
    const int mb = m0 + base;                          // global index of the pass's first set
    const int m = mb + i;
    // group head: walk back while the predecessor has the same shape and no boundary is crossed
    int h = i;
    while (h > 0 && ((mb + h) % group_cap) != 0 && same_shape(structure, N, mb + h, mb + h - 1)) h--;
    w.head[e] = h;
    // sub-groups: the run of equal stem density that contains m, inside the group, cut every LUT_SUB members
    const double lambda = structure[0 * N + m];
    int rs = i;
    while (rs > h && structure[0 * N + mb + rs - 1] == lambda) rs--;
    int nj = 0;
    if ((i - rs) % LUT_SUB == 0) {
        nj = 1;
        while (nj < LUT_SUB && i + nj < n_pass && ((mb + i + nj) % group_cap) != 0 &&
               same_shape(structure, N, mb + i + nj, mb + i + nj - 1) && structure[0 * N + mb + i + nj] == lambda) nj++;
    }
    w.sub[e] = nj;
    shape_store(w.shp + (size_t) e * LUT_SHP, shape_compute(structure, N, m));
    if (w.cnt) {
        list_append(h == i, c, w.cnt + LUT_NCNT * c + 0, w.hl + base, i);
        list_append(nj == 1, c, w.cnt + LUT_NCNT * c + 1, w.s1 + base, i);
        list_append(nj > 1, c, w.cnt + LUT_NCNT * c + 2, w.s8 + base, i);
    }
}

// theta' and its trig, E[S]: one thread per (group head, zenith)
__global__ void __launch_bounds__(128)
lut_prep_kernel(int n, int m0, const double* __restrict__ structure, size_t N, LutWork w)
{
    const long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    const int i = (int) (e / LUT_ZW), t = (int) (e - (long) i * LUT_ZW);
    if (i >= n || w.head[i] != i || t >= GORT_NTH) return;
    const Shape S = shape_load(w, i);
    const double dth = 1 * GORT_PI / 180.0;
    double theta = dth * (double) t;                                             // gortt.c:783-797
    if (theta >= GORT_PI / 2.0) theta = GORT_PI / 2.0 - 1.0 * GORT_PI / 180.0;
    double th = atan(tan(theta) * S.ellip);
    if (th >= GORT_PI / 2.0) th = GORT_PI / 2.0 - 1.0 * GORT_PI / 180.0;
    Ang a;
    a.th = th; a.s = sin(th); a.c = cos(th); a.t = tan(th);
    double* o = w.trig + (size_t) i * 4 * LUT_ZW + t;
    o[0 * LUT_ZW] = a.s; o[1 * LUT_ZW] = a.c; o[2 * LUT_ZW] = a.t;
    o[3 * LUT_ZW] = t < GORT_NTH - 1 ? expected_single_crown_path(S.c, a, layer_height_p(w, i, 0)) : 0.0;   // :445
}

__device__ __forceinline__ Ang ang_load(const LutWork& w, int i, int t)
{
    const double* o = w.trig + (size_t) i * 4 * LUT_ZW + t;
    Ang a;
    a.th = 0.0; a.s = o[0 * LUT_ZW]; a.c = o[1 * LUT_ZW]; a.t = o[2 * LUT_ZW];
    return a;
}

// v_g[h][t], gortt_pn_kopen.c:29, :149-167: midpoint rule over the crown-centre height z of the projected cross-section
// of a crown centred at z seen from layer height h.  The cross-section depends on h - z only, the layer heights and
// the midpoints are both dz' apart, so the 15 x K evaluations take only 14 + K distinct values: each is evaluated once
// (at its first (h, z) pair) and the 15 sums are formed in the reference's order.  (The other pairs differ from it by
// the rounding of h - z, ~1e-16.)  One thread per (group head, zenith); its cross-sections sit in its own column of
// shared memory (no barrier: nobody else reads them).
#define LUT_VG_THREADS 128
__global__ void __launch_bounds__(LUT_VG_THREADS, 7)
lut_vg_kernel(int n, int m0, const double* __restrict__ structure, size_t N, LutWork w)
{
    // 14 + K <= 29 distinct cross-sections of this thread.  (The crown-centre heights used to sit in a second array; at
    // 47 KB per CTA only 16 warps fitted an SM -- ncu: 21 % of the warp slots, FP64 pipe 37 %.  They are a running sum,
    // :162, and are now simply formed again in the order they are needed.)
    __shared__ double s_A[30][LUT_VG_THREADS];
    const long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    const int i = (int) (e / LUT_ZW), t = (int) (e - (long) i * LUT_ZW);
    if (i >= n || w.head[i] != i || t >= GORT_NTH) return;
    const Shape S = shape_load(w, i);
    const Ang a = ang_load(w, i, t);
    double* vg = w.vg + (size_t) i * GORT_NLAYERS * LUT_ZW + t;
    // number of crown-centre heights of the midpoint rule, gortt_pn_kopen.c:162: a running sum
    const double z0 = S.c.h1_p + S.c.dz_p / 2.0;
    int K = 0;
    {
        double z = z0;
        for (; z <= S.c.h2_p && K < 16; z += S.c.dz_p) K++;
        if (K == 16 && z <= S.c.h2_p) K = 17;                    // more than 16 midpoints: the literal rule below
    }
    if (K < 1 || K >= 16) {
#pragma unroll 1
        for (int h = 0; h < GORT_NLAYERS; h++) vg[(size_t) h * LUT_ZW] = proj_volume(S.c, a, layer_height_p(w, i, h));
        return;
    }
    // distinct cross-sections j = 0 .. 13 + K: (h, z) = (0, z_{K-1-j}) for j < K, (j-K+1, z_0) after
    {
        const double h0 = layer_height_p(w, i, 0);
        double z = z0;
#pragma unroll 1
        for (int k = 0; k < K; k++, z += S.c.dz_p) s_A[K - 1 - k][threadIdx.x] = cross_section(S.c, a, h0, z);
    }
#pragma unroll 1
    for (int j = K; j < GORT_NLAYERS + K - 1; j++)
        s_A[j][threadIdx.x] = cross_section(S.c, a, layer_height_p(w, i, j - (K - 1)), z0);
#pragma unroll 1
    for (int h = 0; h < GORT_NLAYERS; h++) {
        double vol = 0.0;
        for (int k = 0; k < K; k++) vol += s_A[h - k + K - 1][threadIdx.x] * (S.c.dz_p);
        vg[(size_t) h * LUT_ZW] = vol;
    }
}

// Tube-volume difference per entry height, gortt_pn_kopen.c:496.  Item = (group head, zenith third, entry height) = one
// warp's work; the warps share nothing, so they run as persistent warps (four to a CTA, ten CTAs per SM) striding over
// the items of the head list.  (A 13-warp CTA per (set, third) held its registers until its slowest entry height was
// done -- ncu: 43 % of the warp slots busy against 61 % allowed by the registers -- and launched 3 CTAs per set whether
// or not the set was a group head.)
#define LUT_TUBE_WARPS 4
#define LUT_TUBE_OCC 10
__global__ void __launch_bounds__(32 * LUT_TUBE_WARPS, LUT_TUBE_OCC)
lut_tube_kernel(LutWork w)
{
    const int lane = threadIdx.x & 31;
    const int n_items = w.cnt[0] * (3 * LUT_NSP);
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(&w.cnt[3], 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int hi = item / (3 * LUT_NSP), wid = item - hi * (3 * LUT_NSP);
        const int i = w.hl[hi];
        const int third = wid / LUT_NSP, k = wid - third * LUT_NSP;
        const int t = third * 32 + lane;
        if (t >= GORT_NTH - 1) continue;                                         // epgap only for t < nth - 1, :1099
        const Shape S = shape_load(w, i);
        const Ang a = ang_load(w, i, t);
        const double hp0 = layer_height_p(w, i, 0);
        const double hps = layer_height_p(w, i, GORT_NLAYERS - 2 - k);              // :457, sp_i = 13 down to 1
        w.tube[((size_t) i * LUT_NSP + k) * LUT_ZW + t] = tube_vol(S.c, a, hp0, hps, S.c.h2_p) - tube_vol(S.c, a, hp0, hps, S.c.h1_p);
    }
}

// Where finished LUT rows go.  `local` is this GPU's copy (kopen_kernel reads the rows back from it); `dst` are further
// copies of the same rows -- tables in the memory of peer GPUs mapped into this process (NVLink P2P), or one NVSwitch
// multicast address that reaches every GPU of the group (`mc`: the store is then a multimem.st).  The rows leave with the
// stores that produce them: posted writes over NVLink underneath the crown-count arithmetic of the other CTAs, instead of
// an all-gather after the kernels.
struct LutOut {
    double* local;
    int n, mc;
    double* dst[GORT_LUT_MAX_DST];
};

__device__ __forceinline__ void lut_store(const LutOut& o, size_t off, double v)
{
    o.local[off] = v;
    for (int q = 0; q < o.n; q++) {
        double* a = o.dst[q] + off;
        if (o.mc) asm volatile("multimem.st.relaxed.sys.global.f64 [%0], %1;" :: "l"(a), "d"(v) : "memory");
        else *a = v;
    }
}

// Crown-count loop and within-crown gap sums.  Item = (sub-group head, zenith third) = one CTA's work, warp = entry
// height; persistent CTAs stride over the items of the sub-group list of their kind (SUB = 1: single-member sub-groups,
// SUB = LUT_SUB: the others).
template <int SUB>
struct CrownSmem {
    double tab[LUT_TAB][SUB];                // exp(-s_bin tau') per (bin, member): a bin's members are one 64-byte row,
                                             // read with four 16-byte loads instead of eight 8-byte ones
    double part[LUT_NSP][SUB][32];           // partial within-crown gap sums per entry height
};
// the tangent kernels add the partial sums of the favd tangent
template <int SUB>
struct CrownSmemTan {
    CrownSmem<SUB> p;
    double dpart[LUT_NSP][SUB][32];
};
#define LUT_CROWN_OCC(SUB) ((SUB) == 1 ? 3 : 2)
#define LUT_CROWN_TAN_OCC(SUB) ((SUB) == 1 ? 3 : 1)

// TAN = true: the same records and dlut, their favd tangent (p_n0 rows 0, epgap rows).  favd enters the record only
// through the bin attenuation exp(-s_bin tau'), s_bin = row ds, tau' = 0.5 favd b/r, whose favd derivative is
// -0.5 (b/r) ds row exp(-s_bin tau').  The factor -0.5 (b/r) ds is common to the sub-group (one shape), so the tangent
// accumulates sum row wgt exp(-s_bin tau') next to the primal sum -- one more FMA per member and crown count -- and is
// scaled once when the row is stored.  The bins, the weights and the primal arithmetic are those of the primal kernel.
template <int SUB, bool TAN>
__global__ void __launch_bounds__(32 * LUT_NSP, TAN ? LUT_CROWN_TAN_OCC(SUB) : LUT_CROWN_OCC(SUB))
lut_crown_kernel(int m0, const double* __restrict__ structure, size_t N, LutWork w, const LutOut out,
                 double* __restrict__ dlut)
{
    extern __shared__ __align__(16) unsigned char crown_smem_raw[];
    CrownSmem<SUB>& sm = *reinterpret_cast<CrownSmem<SUB>*>(crown_smem_raw);
    double (*s_tab)[SUB] = sm.tab;
    double (*s_part)[SUB][32] = sm.part;
    double (*s_dpart)[SUB][32] = TAN ? reinterpret_cast<CrownSmemTan<SUB>*>(crown_smem_raw)->dpart : nullptr;
    const int lane = threadIdx.x & 31, k = threadIdx.x >> 5;
    const int* __restrict__ list = SUB == 1 ? w.s1 : w.s8;
    const int n_items = 3 * w.cnt[SUB == 1 ? 1 : 2];
    // Shared memory across items: the table of item n+1 is written while slow warps may still read the partial sums of
    // item n (another array); they have all left item n's crown-count loop (the barrier before the partial sums), and
    // nobody enters item n+1's loop before the barrier after its table.
  __shared__ int s_item;
  for (;;) {
    if (threadIdx.x == 0) s_item = atomicAdd(&w.cnt[SUB == 1 ? 4 : 5], 1);
    __syncthreads();                                    // also: everybody has left the previous item's partial sums
    const int item = s_item;
    if (item >= n_items) break;
    const int i = list[item / 3];
    const int nj = w.sub[i];
    const int hd = w.head[i];
    const int t = (item % 3) * 32 + lane;
    const int m = m0 + i;
    const Shape S = shape_load(w, i);
    const double lambda = structure[0 * N + m];
    const double lv = lambda / (S.h2 - S.h1);
    const double lv_p = lv * S.ellip;
    // bin attenuations of the sub-group's members: exp(-s_bin tau'), s_bin = bin * ds, tau' = k favd'  (:1110-1114).
    // Bins in use: s < n E[S] <= 30 * (21/20) * 4r/3 = 42 r  (s = s'(1 - e^(-n E[S]/s')) < n E[S]; E[S] is a 20- or
    // 21-term midpoint sum of 4r/3 (:534-563)), so only bins up to 42 r / ds + 1 are ever addressed.
    const int n_tab = (int) fmin((double) LUT_TAB, 42.0 * S.c.r / S.c.ds + 2.0);
    for (int e = threadIdx.x; e < nj * n_tab; e += 32 * LUT_NSP) {
        const int j = e / n_tab, bin = e - j * n_tab;
        const double favd_p = structure[5 * N + m + j] * S.ellip;
        const double sbin = (double) bin * S.c.ds;
        s_tab[bin][j] = exp(-sbin * (0.5 * favd_p));
    }
    const bool live = t < GORT_NTH, path = t < GORT_NTH - 1;
    double e_t[SUB], de_t[SUB];
#pragma unroll
    for (int j = 0; j < SUB; j++) e_t[j] = 0.0;
    if (TAN) {
#pragma unroll
        for (int j = 0; j < SUB; j++) de_t[j] = 0.0;
    }
    const double* vg = w.vg + (size_t) hd * GORT_NLAYERS * LUT_ZW + t;
    double pn0_0 = 0.0;
    if (live && k == 0) pn0_0 = exp(-1.0 * lv_p * vg[0]);                        // gortt_pn_kopen.c:30: the p_n0 row of the LUT
    __syncthreads();
    if (path) {
        const double* tr = w.trig + (size_t) hd * 4 * LUT_ZW + t;
        const double a_c = tr[1 * LUT_ZW], es = tr[3 * LUT_ZW];
        const int sp_i = GORT_NLAYERS - 2 - k;
        const double P_s_p = exp(-1.0 * lv_p * vg[(size_t) (sp_i + 1) * LUT_ZW]) - exp(-1.0 * lv_p * vg[(size_t) sp_i * LUT_ZW]);   // :43, :482
        const double temp1 = w.tube[((size_t) hd * LUT_NSP + k) * LUT_ZW + t] * lv_p;   // :497
        const double E = exp(-temp1);
        const double hp0 = layer_height_p(w, i, 0);
        const double sp = (double) (layer_height_p(w, i, sp_i) - hp0) / a_c;       // :464
        // crown-count loop, gortt_pn_kopen.c:489-527, with its loop invariants hoisted:
        //   P(n) P(s') = temp1^n e^-temp1 / (n! (1 - e^-temp1)) P(s')        :501-502, :522
        //   s          = s' (1 - exp(-n E[S]/s'))                            :508
        // exp(-n x) is advanced as q^n (q = exp(-x)) and s/ds + 0.5 formed with one FMA; because s selects a histogram
        // bin through (int)(s/ds + 0.5) (:134-139, :522) the literal formula is evaluated instead whenever the fast
        // form lands within 1e-9 of a bin boundary, so the bin is always the one the literal formula gives.
        const double c0 = E / (1.0 - E) * P_s_p;
        const double q = exp(-(es / sp));
        const double spd = sp * (1.0 / S.c.ds), spd5 = spd + 0.5;
        // Hot loop without branches: the bin comes from the fast form; a crown count whose fast form lands within 1e-9
        // of a bin boundary, or whose bin lies beyond the table, only raises a flag (and reads a clamped table row).
        // A flagged (zenith, entry height) -- about one in 10^6 -- is then redone from scratch with the literal formulas.
        double pw = c0, qn = 1.0, ub_last = 4194304.0;
        bool redo = !(q >= 0.0 && q <= 1.0 && spd > 0.0);
        // floor(u) and the distance of u from the nearest integer without the conversion unit (FRND / F2I run at a
        // quarter of the FP64 rate and made this loop XU-bound: ncu 36 % XU against 45 % FP64): 0.5 <= u < 2^22, so
        // u + 2^22 has the exponent of 2^22, its mantissa holds floor(u) above bit 30 and the fraction of u, in units
        // of 2^-30 = 9.3e-10, below.  The 2^22 is folded into the FMA's addend (one rounding to 2^-30 units instead of
        // two; the addend's own rounding and the FMA's are at most one unit together).  A fraction within 2 units of
        // either end (|u - rint(u)| < 1.9e-9, a superset of the 1e-9 rule plus that unit) raises the flag.
        // With 0 <= q <= 1 and s'/ds > 0 the u of successive crown counts never decrease (q^n does not increase, the
        // FMA is monotonic), so the range tests -- u left the binade, or the bin lies beyond the table -- are made
        // once, on the last u, after the loop; inside it only the fraction is tested and the table row clamped.
        const double spd5m = spd5 + 4194304.0;
#pragma unroll
        for (int nn = 1; nn <= LUT_MAXCROWNS; nn++) {                            // :489
            pw *= temp1;                                                         // temp1^n e^-t / (1 - e^-t) P(s')
            qn *= q;
            const double wgt = pw * c_inv_fact[nn];
            const double ubd = fma(-spd, qn, spd5m);
            const long long ub = __double_as_longlong(ubd);
            const int idx = (int) ((ub >> 30) & 0x3fffff);
            const unsigned frac = (unsigned) ub & 0x3fffffffu;
            redo |= (frac - 2u) > (0x3fffffffu - 4u);
            ub_last = ubd;
            const int row = min(idx, n_tab - 1);
            const double rw = TAN ? (double) row * wgt : 0.0;
            // gortt_calc_epgap + gortt_calc_pgap, :1110-1114, :1138
            if (SUB == 1) {
                e_t[0] = fma(s_tab[row][0], wgt, e_t[0]);
                if (TAN) de_t[0] = fma(s_tab[row][0], rw, de_t[0]);
            } else {
                const double2* __restrict__ tp = reinterpret_cast<const double2*>(&s_tab[row][0]);
#pragma unroll
                for (int j2 = 0; j2 < SUB / 2; j2++) {
                    const double2 v = tp[j2];
                    e_t[2 * j2] = fma(v.x, wgt, e_t[2 * j2]);
                    e_t[2 * j2 + 1] = fma(v.y, wgt, e_t[2 * j2 + 1]);
                    if (TAN) {
                        de_t[2 * j2] = fma(v.x, rw, de_t[2 * j2]);
                        de_t[2 * j2 + 1] = fma(v.y, rw, de_t[2 * j2 + 1]);
                    }
                }
            }
        }
        const double u_last = ub_last - 4194304.0;
        redo |= !(u_last >= 0.0 && u_last < (double) (n_tab - 1));
        if (redo) {
#pragma unroll
            for (int j = 0; j < SUB; j++) e_t[j] = 0.0;
            if (TAN) {
#pragma unroll
                for (int j = 0; j < SUB; j++) de_t[j] = 0.0;
            }
            pw = c0; qn = 1.0;
#pragma unroll 1
            for (int nn = 1; nn <= LUT_MAXCROWNS; nn++) {
                pw *= temp1;
                qn *= q;
                const double wgt = pw * c_inv_fact[nn];
                double u = fma(-spd, qn, spd5);
                if (fabs(u - rint(u)) < 1e-9)
                    u = sp * (1.0 - exp(-1.0 * (double) nn * es / sp)) / S.c.ds + 0.5;   // the literal formula, :508, :134-139
                const int idx = (int) u;
                const double rw = TAN ? (double) idx * wgt : 0.0;
                if (idx >= 0 && idx < n_tab) {
#pragma unroll
                    for (int j = 0; j < SUB; j++) e_t[j] = fma(s_tab[idx][j], wgt, e_t[j]);
                    if (TAN) {
#pragma unroll
                        for (int j = 0; j < SUB; j++) de_t[j] = fma(s_tab[idx][j], rw, de_t[j]);
                    }
                } else {
                    const double sbin = (double) idx * S.c.ds;
#pragma unroll
                    for (int j = 0; j < SUB; j++) {                              // beyond the table: the formula itself
                        const double tau_j = 0.5 * (structure[5 * N + m + (j < nj ? j : 0)] * S.ellip);
                        if (TAN) {
                            const double x = exp(-sbin * tau_j);
                            e_t[j] = fma(x, wgt, e_t[j]);
                            de_t[j] = fma(x, rw, de_t[j]);
                        } else {
                            e_t[j] = fma(exp(-sbin * tau_j), wgt, e_t[j]);
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < SUB; j++) s_part[k][j][lane] = e_t[j];
    if (TAN) {
#pragma unroll
        for (int j = 0; j < SUB; j++) s_dpart[k][j][lane] = de_t[j];
    }
    __syncthreads();
    // rows of the LUT record: p_n0[0][t] and epgap[0][t] (the 13 entry heights added in the reference's order, :457);
    // the openness factors are formed by kopen_kernel afterwards
    if (live) {
        if (k == 0) for (int j = 0; j < nj; j++) lut_store(out, (size_t) (m + j) * GORT_LUT_STRIDE + t, pn0_0);
        if (TAN && k == 0) for (int j = 0; j < nj; j++) dlut[(size_t) (m + j) * GORT_LUT_STRIDE + t] = 0.0;   // p_n0 has no favd
        for (int j = k; j < nj; j += LUT_NSP) {
            double e = s_part[0][j][lane];
#pragma unroll
            for (int q2 = 1; q2 < LUT_NSP; q2++) e += s_part[q2][j][lane];
            lut_store(out, (size_t) (m + j) * GORT_LUT_STRIDE + GORT_NTH + t, e);
            if (TAN) {
                double de = s_dpart[0][j][lane];
#pragma unroll
                for (int q2 = 1; q2 < LUT_NSP; q2++) de += s_dpart[q2][j][lane];
                dlut[(size_t) (m + j) * GORT_LUT_STRIDE + GORT_NTH + t] = de * (-(0.5 * S.ellip) * S.c.ds);
            }
        }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// The intermediates of gortt_gap_probabilities that never reach the BRDF (SURVEY.md 8f row 1): gortt_calc_vb
// (gortt_pn_kopen.c:925-972), gortt_calc_fb (:975-1006), gortt_calc_t_open (:1010-1078) and the dk_open / k_open[h] rows of
// gortt_calc_kopen (:351-375).  gortt_calc_t_open is ~90 % of the reference's LUT time: a z x h x zenith x crown-count
// nest (15 x 15 x 91 x 30) that re-integrates E[S] (gortt_get_es, a 20-step sum) inside its innermost loop.  Here E[S]
// towards every layer is tabulated first (lut_es_all_kernel, once per crown shape), and the nest runs with
// warp = (z, h) pair, lanes = zeniths, exp(-n x) advanced as q^n and temp1^n by multiplication, the zenith sum as a
// lane-strided sum + shuffle tree (the reference adds the 91 zeniths left to right: same terms, different association).
__global__ void __launch_bounds__(128)
lut_es_all_kernel(int n, int m0, const double* __restrict__ structure, size_t N, LutWork w)
{
    const long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    const int t = (int) (e % LUT_ZW);
    const int z = (int) ((e / LUT_ZW) % GORT_NLAYERS);
    const int i = (int) (e / ((long) LUT_ZW * GORT_NLAYERS));
    if (i >= n || w.head[i] != i || t >= GORT_NTH) return;
    const Shape S = shape_load(w, i);
    const Ang a = ang_load(w, i, t);
    w.es_all[((size_t) i * GORT_NLAYERS + z) * LUT_ZW + t] = expected_single_crown_path(S.c, a, layer_height_p(w, i, z));   // gortt_get_es(p, z, t)
}

struct DeadOut { double *vb, *fb, *t_open, *dt_open, *dk_open, *k_open; };

#define LUT_DEAD_WARPS GORT_NLAYERS
__global__ void __launch_bounds__(32 * LUT_DEAD_WARPS, 2)
lut_dead_kernel(int n, int m0, const double* __restrict__ structure, size_t N, LutWork w, DeadOut o)
{
    __shared__ double s_vb[GORT_NLAYERS], s_hp[GORT_NLAYERS];
    __shared__ double s_sin2[LUT_ZW], s_cos[LUT_ZW];
    __shared__ double s_f1[GORT_NLAYERS][LUT_ZW];          // p_n0[h][t] sin(2 theta_t)
    const int i = blockIdx.x, m = m0 + i, hd = w.head[i];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const Shape S = shape_load(w, i);
    const double lambda = structure[0 * N + m], favd = structure[5 * N + m];
    const double lv_p = (lambda / (S.h2 - S.h1)) * S.ellip;                       // gortt.c:671, :677
    const double tau_p = 0.5 * (favd * S.ellip);                                  // :675-676
    const double dth = 1 * GORT_PI / 180.0;
    const double r = S.c.r;
    if (threadIdx.x < GORT_NLAYERS) {
        // gortt_calc_vb, :938-970: sphere centred at layer height, cut by the h1 and h2 planes
        const double hp = layer_height_p(w, i, threadIdx.x);
        double Vol = 4.0 * GORT_PI * S.c.rrr / 3.0, tmp;
        if (hp + r > S.c.h2_p) { tmp = hp + r - S.c.h2_p; Vol -= GORT_PI * tmp * tmp * (3.0 * r - tmp) / 3.0; }
        if (hp - r < S.c.h1_p) { tmp = S.c.h1_p - (hp - r); Vol -= GORT_PI * tmp * tmp * (3.0 * r - tmp) / 3.0; }
        if (Vol < -0.0000001) Vol = __longlong_as_double(0x7ff8000000000000LL);   // the reference exits here: NaN marks the set
        else if (Vol < 0) Vol = 0.0;
        s_vb[threadIdx.x] = Vol; s_hp[threadIdx.x] = hp;
        if (o.vb) o.vb[(size_t) m * GORT_NLAYERS + threadIdx.x] = Vol;
    }
    for (int t = threadIdx.x; t < LUT_ZW; t += blockDim.x) {
        double theta = dth * (double) min(t, GORT_NTH - 1);                       // gortt.c:783-787
        if (theta >= GORT_PI / 2.0) theta = GORT_PI / 2.0 - 1.0 * GORT_PI / 180.0;
        s_sin2[t] = sin(2.0 * theta);
        s_cos[t] = w.trig[(size_t) hd * 4 * LUT_ZW + 1 * LUT_ZW + min(t, GORT_NTH - 1)];
    }
    __syncthreads();
    // ---- p_n0[h][t] for every layer: fb (:981-1003) and the integrands of k_open[h] / dk_open[h] ----
    {
        const int h = wp;
        const double one_m_e = 1.0 - exp(-lv_p * s_vb[h]);
        for (int t = lane; t < GORT_NTH; t += 32) {
            const double pn0 = exp(-1.0 * lv_p * w.vg[((size_t) hd * GORT_NLAYERS + h) * LUT_ZW + t]);
            s_f1[h][t] = pn0;
            double d = 1.0 - pn0;
            if (d < 2.2250738585072014e-308 * 2.) d = 2.2250738585072014e-308 * 2.;       // DBL_MIN * 2, :990
            if (o.fb) o.fb[((size_t) m * GORT_NLAYERS + h) * GORT_NTH + t] = one_m_e / d;
        }
    }
    __syncthreads();
    {
        // gortt_calc_kopen, :351-375: trapezoid panels over the zeniths for layer h = warp
        const int h = wp;
        double ko = 0.0, dk = 0.0;
        for (int t = 1 + lane; t < GORT_NTH; t += 32) {
            const double p1 = s_f1[h][t], p0 = s_f1[h][t - 1];
            ko += (p1 * s_sin2[t] + p0 * s_sin2[t - 1]) / 2.0 * dth;
            const double q1 = h == GORT_NLAYERS - 1 ? 0.0 : s_f1[h + 1][t] - p1;          // p_s0, :40-45
            const double q0 = h == GORT_NLAYERS - 1 ? 0.0 : s_f1[h + 1][t - 1] - p0;
            dk += (q1 * s_sin2[t] + q0 * s_sin2[t - 1]) / 2.0 * dth;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) { ko += __shfl_xor_sync(0xffffffffu, ko, off); dk += __shfl_xor_sync(0xffffffffu, dk, off); }
        if (lane == 0) {
            if (o.k_open) o.k_open[(size_t) m * GORT_NLAYERS + h] = ko;
            if (o.dk_open) o.dk_open[(size_t) m * GORT_NLAYERS + h] = dk;
        }
    }
    if (!o.t_open && !o.dt_open) return;
    // ---- gortt_calc_t_open, :1033-1075: 120 (z, h >= z) pairs dealt round-robin to the warps ----
    for (int pair = wp; pair < GORT_NLAYERS * (GORT_NLAYERS + 1) / 2; pair += LUT_DEAD_WARPS) {
        int z = 0, rem = pair;
        while (rem >= GORT_NLAYERS - z) { rem -= GORT_NLAYERS - z; z++; }
        const int h = z + rem;
        double Tsum = 0.0, dTsum = 0.0;
        if (z != h) {
            const double dsz = (1.0 - exp(lv_p * s_vb[z])) * S.c.dz_p;             // sic: + exponent, :1055
            const double dhp = fabs(s_hp[z] - s_hp[h]);
            for (int t = lane; t < GORT_NTH; t += 32) {
                const double cth = s_cos[t];
                const double s_p = dhp / cth;                                      // :1047
                const double es = w.es_all[((size_t) hd * GORT_NLAYERS + z) * LUT_ZW + t];
                const double temp1 = lv_p * GORT_PI * r * r * s_p;                 // :1051
                const double E = exp(-temp1);
                const double c0 = E / (1.0 - E);
                const double q = exp(-(es / s_p));
                const double fac = 1.0 - exp(tau_p * (dsz / cth));                 // :1056
                double pw = 1.0, qn = 1.0, T = 0.0, dT = 0.0;
#pragma unroll 2
                for (int nn = 1; nn <= LUT_MAXCROWNS; nn++) {
                    pw *= temp1; qn *= q;
                    const double s = s_p * (1.0 - qn);                             // :1050
                    const double P_n = pw * c0 * c_inv_fact[nn];                   // :1052-1053
                    const double pe = P_n * exp(-s * tau_p);
                    T += pe;                                                       // :1054
                    dT += pe * fac;                                                // :1056
                }
                Tsum += s_sin2[t] * T * dth;                                       // :1059
                dTsum += s_sin2[t] * dT * dth;
            }
        } else {
            const double dsz = 0.5 * (1.0 - exp(-lv_p * s_vb[z])) * S.c.dz_p;      // :1070
            for (int t = lane; t < GORT_NTH; t += 32) {
                const double dT = 1.0 - exp(-tau_p * (dsz / s_cos[t]));
                dTsum += s_sin2[t] * dT * dth;                                     // :1072
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) { Tsum += __shfl_xor_sync(0xffffffffu, Tsum, off); dTsum += __shfl_xor_sync(0xffffffffu, dTsum, off); }
        if (lane == 0) {
            const size_t b = (size_t) m * GORT_NLAYERS * GORT_NLAYERS;
            if (o.t_open) { o.t_open[b + h * GORT_NLAYERS + z] = Tsum; o.t_open[b + z * GORT_NLAYERS + h] = Tsum; }
            if (o.dt_open) { o.dt_open[b + h * GORT_NLAYERS + z] = dTsum; o.dt_open[b + z * GORT_NLAYERS + h] = dTsum; }
        }
    }
}

// gortt_pn_kopen.c:1144-1200; with TAN also dlut, the favd tangent of the closed form: l is linear in favd
// (dl = b 4/3 cc), a = cc (exp(k1 cc^2) - exp(-k2 l)) gives da = cc k2 exp(-k2 l) dl, and
// epg = exp(-a / cos theta') - pn0 gives depg = -(da / cos theta') exp(-a / cos theta'); the same trapezoid on the
// tangent rows gives dk_openep.  p_n0 and k_open have no favd.
template <bool TAN>
__device__ __forceinline__ void q08_record(int n_sets, const double* __restrict__ structure, double* __restrict__ lut,
                                           double* __restrict__ dlut)
{
    __shared__ double s_pn0[GORT_NTH];
    __shared__ double s_epg[GORT_NTH];
    __shared__ double s_sin2[GORT_NTH];
    __shared__ double s_depg[TAN ? GORT_NTH : 1];
    const int m = blockIdx.x;
    const int t = threadIdx.x;
    const double lambda = structure[0 * (size_t) n_sets + m];
    const double r      = structure[1 * (size_t) n_sets + m];
    const double b      = structure[2 * (size_t) n_sets + m];
    const double favd   = structure[5 * (size_t) n_sets + m];
    const double ellip = b / r;
    const double rr = r * r;
    const double dth = 1 * GORT_PI / 180.0;
    if (t < GORT_NTH) {
        double theta = dth * (double) t;
        if (theta >= GORT_PI / 2.0) theta = GORT_PI / 2.0 - 1.0 * GORT_PI / 180.0;
        double theta_p = atan(tan(theta) * ellip);
        if (theta_p >= GORT_PI / 2.0) theta_p = GORT_PI / 2.0 - 1.0 * GORT_PI / 180.0;
        double cc = GORT_PI * rr * lambda;                               // :1164
        double l = favd * b * 4. / 3. * cc;                              // :1166
        double k2 = 0.348535 * pow(cc, (-1.08069 - 0.0874595 * cc));     // :1168
        double k1 = 0.0014166;
        double a = cc * (exp(k1 * cc * cc) - exp(-k2 * l));              // :1171
        double pn0 = exp(-cc / (cos(theta_p)));                          // :1185
        double epg = exp(-a / (cos(theta_p))) - pn0;                     // :1186
        s_pn0[t] = pn0; s_epg[t] = epg; s_sin2[t] = sin(2.0 * theta);
        double* o = lut + (size_t) m * GORT_LUT_STRIDE;
        o[t] = pn0;
        o[GORT_NTH + t] = epg;
        if (TAN) {
            const double dl = b * 4. / 3. * cc;
            const double da = cc * (k2 * exp(-k2 * l)) * dl;
            const double ct = cos(theta_p);
            const double depg = -(da / ct) * exp(-a / ct);
            s_depg[t] = depg;
            double* d = dlut + (size_t) m * GORT_LUT_STRIDE;
            d[t] = 0.0;
            d[GORT_NTH + t] = depg;
        }
    }
    __syncthreads();
    if (t == 0) {
        double ko = 0.0, ke = 0.0;
        // :1176-1177 read rows that are still calloc'd zeros
        double tmp1_last = 0.0 * s_sin2[0], tmp2_last = 0.0 * s_sin2[0];
        for (int i = 1; i < GORT_NTH; i++) {
            double tmp1 = s_pn0[i] * s_sin2[i];
            ko += (tmp1 + tmp1_last) / 2.0 * dth;
            tmp1_last = tmp1;
            double tmp2 = s_epg[i] * s_sin2[i];
            ke += (tmp2 + tmp2_last) / 2.0 * dth;
            tmp2_last = tmp2;
        }
        double* o = lut + (size_t) m * GORT_LUT_STRIDE;
        o[2 * GORT_NTH] = ko;
        o[2 * GORT_NTH + 1] = ke;
        if (TAN) {
            double dke = 0.0, last = 0.0 * s_sin2[0];
            for (int i = 1; i < GORT_NTH; i++) {
                const double tmp = s_depg[i] * s_sin2[i];
                dke += (tmp + last) / 2.0 * dth;
                last = tmp;
            }
            double* d = dlut + (size_t) m * GORT_LUT_STRIDE;
            d[2 * GORT_NTH] = 0.0;
            d[2 * GORT_NTH + 1] = dke;
        }
    }
}

__global__ void __launch_bounds__(LUT_THREADS)
lut_q08_kernel(int n_sets, const double* __restrict__ structure, double* __restrict__ lut)
{
    q08_record<false>(n_sets, structure, lut, nullptr);
}

__global__ void __launch_bounds__(LUT_THREADS)
lut_q08_tangent_kernel(int n_sets, const double* __restrict__ structure, double* __restrict__ lut, double* __restrict__ dlut)
{
    q08_record<true>(n_sets, structure, lut, dlut);
}

// gortt_calc_kopen, gortt_pn_kopen.c:351-375 for h = 0: k_open = trapezoid rule of p_n0 sin(2 theta) over the 91
// zeniths, k_openep the same for epgap.  One warp per parameter set: the panels (f_i + f_{i-1})/2 * dth, i = 1..90,
// three per lane, then a shuffle tree (the reference adds them left to right: same panels, different association).
__global__ void __launch_bounds__(128)
kopen_kernel(int n_sets, const LutOut out)
{
    const double* lut = out.local;
    const int m = (int) (((long) blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (m >= n_sets) return;
    const int lane = threadIdx.x & 31;
    const double dth = 1 * GORT_PI / 180.0;
    const double* o = lut + (size_t) m * GORT_LUT_STRIDE;
    double ko = 0.0, ke = 0.0;
    for (int i = 1 + lane; i < GORT_NTH; i += 32) {
        double th1 = dth * (double) i, th0 = dth * (double) (i - 1);                 // gortt.c:783-787
        if (th1 >= GORT_PI / 2.0) th1 = GORT_PI / 2.0 - 1.0 * GORT_PI / 180.0;
        if (th0 >= GORT_PI / 2.0) th0 = GORT_PI / 2.0 - 1.0 * GORT_PI / 180.0;
        const double s1 = sin(2.0 * th1), s0 = sin(2.0 * th0);
        ko += (o[i] * s1 + o[i - 1] * s0) / 2.0 * dth;
        ke += (o[GORT_NTH + i] * s1 + o[GORT_NTH + i - 1] * s0) / 2.0 * dth;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        ko += __shfl_xor_sync(0xffffffffu, ko, off);
        ke += __shfl_xor_sync(0xffffffffu, ke, off);
    }
    if (lane == 0) {
        lut_store(out, (size_t) m * GORT_LUT_STRIDE + 2 * GORT_NTH, ko);
        lut_store(out, (size_t) m * GORT_LUT_STRIDE + 2 * GORT_NTH + 1, ke);
    }
}

// Rows that were produced locally only (the Q08 kernel) copied to the further destinations.
__global__ void __launch_bounds__(256)
lut_rows_out_kernel(size_t n_values, const LutOut out)
{
    for (size_t e = (size_t) blockIdx.x * blockDim.x + threadIdx.x; e < n_values; e += (size_t) gridDim.x * blockDim.x) {
        const double v = out.local[e];
        for (int q = 0; q < out.n; q++) {
            double* a = out.dst[q] + e;
            if (out.mc) asm volatile("multimem.st.relaxed.sys.global.f64 [%0], %1;" :: "l"(a), "d"(v) : "memory");
            else *a = v;
        }
    }
}

int launch_lut_dead(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, double *vb, double *fb,
                    double *t_open, double *dt_open, double *dk_open, double *k_open)
{
    note_other_work(ctx);
    const int cap = LUT_GROUP_CAP;
    const int chunk = n_sets < LUT_CHUNK / 2 ? n_sets : LUT_CHUNK / 2;
    const size_t per_set = sizeof(double) * ((4 + 2 * GORT_NLAYERS + LUT_NSP) * LUT_ZW + LUT_SHP) + 2 * sizeof(int);
    char *base = (char *) workspace(ctx, per_set * (size_t) chunk + 256);
    if (!base) return GORT_ERR_NOMEM;
    LutWork w;
    w.trig = (double *) base;
    w.vg = w.trig + (size_t) chunk * 4 * LUT_ZW;
    w.tube = w.vg + (size_t) chunk * GORT_NLAYERS * LUT_ZW;
    w.es_all = w.tube + (size_t) chunk * LUT_NSP * LUT_ZW;
    w.shp = w.es_all + (size_t) chunk * GORT_NLAYERS * LUT_ZW;
    w.head = (int *) (w.shp + (size_t) chunk * LUT_SHP);
    w.sub = w.head + chunk;
    w.hl = w.s1 = w.s8 = w.cnt = NULL;                   // no work lists on this path: its kernels walk the sets
    const size_t N = (size_t) n_sets;
    for (int m0 = 0; m0 < n_sets; m0 += chunk) {
        const int n = n_sets - m0 < chunk ? n_sets - m0 : chunk;
        DeadOut o = {vb, fb, t_open, dt_open, dk_open, k_open};
        lut_plan_kernel<<<(n + 127) / 128, 128, 0, s>>>(n, m0, n, cap, structure, N, w);
        lut_prep_kernel<<<(unsigned) (((long) n * LUT_ZW + 127) / 128), 128, 0, s>>>(n, m0, structure, N, w);
        lut_vg_kernel<<<(unsigned) (((long) n * LUT_ZW + LUT_VG_THREADS - 1) / LUT_VG_THREADS), LUT_VG_THREADS, 0, s>>>(n, m0, structure, N, w);
        lut_es_all_kernel<<<(unsigned) (((long) n * LUT_ZW * GORT_NLAYERS + 127) / 128), 128, 0, s>>>(n, m0, structure, N, w);
        lut_dead_kernel<<<(unsigned) n, 32 * LUT_DEAD_WARPS, 0, s>>>(n, m0, structure, N, w, o);
        ctx->launches += 5;
    }
    return check_cuda(ctx, cudaGetLastError(), "gort_lut_intermediates launch");
}

static int launch_lut_impl(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, int method, double *lut,
                           int n_dst, double *const *dst, int multicast, double *dlut);

int launch_lut(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, int method, double *lut)
{
    return launch_lut_out(ctx, s, n_sets, structure, method, lut, 0, NULL, 0);
}

int launch_lut_out(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, int method, double *lut,
                   int n_dst, double *const *dst, int multicast)
{
    return launch_lut_impl(ctx, s, n_sets, structure, method, lut, n_dst, dst, multicast, NULL);
}

int launch_lut_tangent(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, int method, double *lut,
                       double *dlut)
{
    return launch_lut_impl(ctx, s, n_sets, structure, method, lut, 0, NULL, 0, dlut);
}

// dlut != NULL: the tangent kernels, which also write dlut (no further destinations then)
static int launch_lut_impl(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *structure, int method, double *lut,
                           int n_dst, double *const *dst, int multicast, double *dlut)
{
    note_other_work(ctx);
    LutOut out;
    out.local = lut;
    out.n = n_dst;
    out.mc = multicast;
    for (int q = 0; q < GORT_LUT_MAX_DST; q++) out.dst[q] = q < n_dst ? dst[q] : NULL;
    if (method == GORT_LUT_Q08) {
        if (dlut) lut_q08_tangent_kernel<<<n_sets, LUT_THREADS, 0, s>>>(n_sets, structure, lut, dlut);
        else lut_q08_kernel<<<n_sets, LUT_THREADS, 0, s>>>(n_sets, structure, lut);
        ctx->launches++;
        if (n_dst > 0) {
            lut_rows_out_kernel<<<ctx->sm_count * 4, 256, 0, s>>>((size_t) n_sets * GORT_LUT_STRIDE, out);
            ctx->launches++;
        }
        return check_cuda(ctx, cudaGetLastError(), "gort_lut launch");
    }
    // group cap: the geometry is shared by the whole group; with the flat kernels the grid no longer depends on the
    // number of groups, so the cap is simply the largest one (round 1's CTA-per-group kernel shrank it for small
    // batches, which made a 16 384-set shard of the C5 grid do 7x the geometry work).  Results do not depend on it.
    const int cap = LUT_GROUP_CAP;
    if (!ctx->lut_attr_set) {
        cudaError_t e = cudaFuncSetAttribute(lut_crown_kernel<LUT_SUB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) sizeof(CrownSmem<LUT_SUB>));
        if (e != cudaSuccess) return check_cuda(ctx, e, "lut_crown_kernel shared memory");
        ctx->lut_attr_set = 1;
    }
    if (dlut && !ctx->lut_tan_attr_set) {
        cudaError_t e = cudaFuncSetAttribute(lut_crown_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) sizeof(CrownSmemTan<1>));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(lut_crown_kernel<LUT_SUB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) sizeof(CrownSmemTan<LUT_SUB>));
        if (e != cudaSuccess) return check_cuda(ctx, e, "lut_crown_kernel<.., true> shared memory");
        ctx->lut_tan_attr_set = 1;
    }
    const int chunk = n_sets < LUT_CHUNK ? n_sets : LUT_CHUNK;
    const int n_pass = (n_sets + chunk - 1) / chunk;
    // workspace: per-zenith arrays for one pass, the plan (shapes, heads, sub-groups, work lists) for the whole call
    const size_t per_set_pass = sizeof(double) * ((4 + GORT_NLAYERS + LUT_NSP) * LUT_ZW);
    const size_t per_set_plan = sizeof(double) * LUT_SHP + 5 * sizeof(int);
    char *base = (char *) workspace(ctx, per_set_pass * (size_t) chunk + per_set_plan * (size_t) n_sets + sizeof(int) * LUT_NCNT * (size_t) n_pass + 256);
    if (!base) return GORT_ERR_NOMEM;
    LutWork w;
    w.trig = (double *) base;
    w.vg = w.trig + (size_t) chunk * 4 * LUT_ZW;
    w.tube = w.vg + (size_t) chunk * GORT_NLAYERS * LUT_ZW;
    w.es_all = NULL;
    w.shp = w.tube + (size_t) chunk * LUT_NSP * LUT_ZW;
    w.head = (int *) (w.shp + (size_t) n_sets * LUT_SHP);
    w.sub = w.head + n_sets;
    w.hl = w.sub + n_sets;
    w.s1 = w.hl + n_sets;
    w.s8 = w.s1 + n_sets;
    w.cnt = w.s8 + n_sets;
    const size_t N = (size_t) n_sets;
    cudaError_t me = cudaMemsetAsync(w.cnt, 0, sizeof(int) * LUT_NCNT * (size_t) n_pass, s);
    if (me != cudaSuccess) return check_cuda(ctx, me, "gort_lut counters");
    lut_plan_kernel<<<(n_sets + 127) / 128, 128, 0, s>>>(n_sets, 0, chunk, cap, structure, N, w);
    ctx->launches++;
    for (int m0 = 0, c = 0; m0 < n_sets; m0 += chunk, c++) {
        const int n = n_sets - m0 < chunk ? n_sets - m0 : chunk;
        LutWork wc = w;                                  // this pass's slice of the plan
        wc.shp += (size_t) m0 * LUT_SHP; wc.head += m0; wc.sub += m0; wc.hl += m0; wc.s1 += m0; wc.s8 += m0; wc.cnt += LUT_NCNT * c;
        LutOut oc = out;                                 // the crown kernels index rows by the global set index themselves
        lut_prep_kernel<<<(unsigned) (((long) n * LUT_ZW + 127) / 128), 128, 0, s>>>(n, m0, structure, N, wc);
        lut_vg_kernel<<<(unsigned) (((long) n * LUT_ZW + LUT_VG_THREADS - 1) / LUT_VG_THREADS), LUT_VG_THREADS, 0, s>>>(n, m0, structure, N, wc);
        const long tube_ctas = ((long) n * 3 * LUT_NSP + LUT_TUBE_WARPS - 1) / LUT_TUBE_WARPS;
        const long tube_max = (long) ctx->sm_count * LUT_TUBE_OCC;      // 6 .. 12 CTAs per SM measured the same
        lut_tube_kernel<<<(unsigned) (tube_ctas < tube_max ? tube_ctas : tube_max), 32 * LUT_TUBE_WARPS, 0, s>>>(wc);
        const long items = (long) n * 3;
        const long c1 = (long) ctx->sm_count * LUT_CROWN_OCC(1), c8 = (long) ctx->sm_count * LUT_CROWN_OCC(LUT_SUB);
        if (dlut) {
            const long t1 = (long) ctx->sm_count * LUT_CROWN_TAN_OCC(1), t8 = (long) ctx->sm_count * LUT_CROWN_TAN_OCC(LUT_SUB);
            lut_crown_kernel<1, true><<<(unsigned) (items < t1 ? items : t1), 32 * LUT_NSP, sizeof(CrownSmemTan<1>), s>>>(m0, structure, N, wc, oc, dlut);
            lut_crown_kernel<LUT_SUB, true><<<(unsigned) (items < t8 ? items : t8), 32 * LUT_NSP, sizeof(CrownSmemTan<LUT_SUB>), s>>>(m0, structure, N, wc, oc, dlut);
        } else {
            lut_crown_kernel<1, false><<<(unsigned) (items < c1 ? items : c1), 32 * LUT_NSP, sizeof(CrownSmem<1>), s>>>(m0, structure, N, wc, oc, NULL);
            lut_crown_kernel<LUT_SUB, false><<<(unsigned) (items < c8 ? items : c8), 32 * LUT_NSP, sizeof(CrownSmem<LUT_SUB>), s>>>(m0, structure, N, wc, oc, NULL);
        }
        ctx->launches += 5;
    }
    kopen_kernel<<<(unsigned) (((long) n_sets * 32 + 127) / 128), 128, 0, s>>>(n_sets, out);
    ctx->launches++;
    if (dlut) {
        // k_open / k_openep are linear in the rows: the same trapezoid on the tangent rows
        LutOut dout;
        dout.local = dlut; dout.n = 0; dout.mc = 0;
        for (int q = 0; q < GORT_LUT_MAX_DST; q++) dout.dst[q] = NULL;
        kopen_kernel<<<(unsigned) (((long) n_sets * 32 + 127) / 128), 128, 0, s>>>(n_sets, dout);
        ctx->launches++;
    }
    return check_cuda(ctx, cudaGetLastError(), "gort_lut launch");
}

}  // namespace gort
