/* oracle/gort_oracle.c -- TEST INFRASTRUCTURE, not product code.
 *
 * Plain-C CPU restatement of the reference GORT hot path (tquaife/gort): canopy derived
 * parameters, KOpen / P(n) gap probabilities (full and Q08), viewed proportions, two-stream
 * scattering terms, the per-wavelength BRDF loop, hemispherical albedo / fAPAR, Price soil
 * reflectance and the PROSPECT interface.  Every function cites the reference file:line it
 * follows.  Arithmetic keeps the reference's operation order so that this file can be
 * checked BIT-FOR-BIT against the unmodified reference compiled into oracle/_ref
 * (tests/test_oracle_vs_ref.py) and against the golden vectors of SURVEY.md App. E
 * (tests/golden/).  Build: gcc -O2 -ffp-contract=off (oracle/Makefile).
 *
 * PARITY PIN: the reference ships no tests or golden vectors of its own.  This restatement
 * is pinned by (1) bit-equality with oracle/_ref on seeded inputs in the build container and
 * (2) the committed fixtures in tests/golden/ generated from oracle/_ref.  The PROSPECT-D
 * part (prospect_d_oracle.c) is "parity unpinned": see that file's header.
 *
 * Deliberately NOT restated (never read by any output, SURVEY.md 3.3): vb, fb, t_open,
 * dt_open, dk_open, lk_up/down, n_mean, pd_s for h>0 (gortt_pn_kopen.c:928-1078).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may use oracle/.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <stdint.h>
#include "gort_oracle.h"
#include <stdio.h>
#include "../gort_b200/data/gort_tables.h"

#define NTH GORT_ORACLE_NTH
#define NLAY GORT_ORACLE_NLAYERS
#define MAXCROWNS 30
#define NH_ES 20
#define SIMPSON_NOINT 20
#define PD_BUFF 3

/* the reference's macros, include/gortt.h:6-10 */
#define O_DTOR(x) ((x) * M_PI / 180.0)
#define O_SEC(x) ((1.0 / cos((x))))
#define O_MAX(x, y) ((x) > (y) ? (x) : (y))
#define O_MIN(x, y) ((x) < (y) ? (x) : (y))

typedef struct {
    /* inputs */
    double lambda, r, b, h1, h2, favd;
    /* derived, gortt.c:641-697 */
    double ellip, rr, rrr, h, k, elai, tau, z1, z2, lv, favd_p, tau_p, lv_p;
    double z1_p, z2_p, h1_p, h2_p, dz, ds, dz_p, dth;
    double height[NLAY], height_p[NLAY], theta[NTH], theta_p[NTH], factorial[MAXCROWNS + 1];
    /* run-time options */
    int use_beta, use_fd;
    double beta, fd_user;
} canopy_t;

/* gortt.c:641-697, :714, :752-797 (defaults gortt.c:74-93) */
static void canopy_init(canopy_t *c, const double *st6)
{
    memset(c, 0, sizeof *c);
    c->lambda = st6[0]; c->r = st6[1]; c->b = st6[2];
    c->h1 = st6[3]; c->h2 = st6[4]; c->favd = st6[5];
    c->dth = O_DTOR(1);                                          /* gortt.c:76 */
    c->ellip = c->b / c->r;                                      /* :641 */
    c->rr = c->r * c->r;                                         /* :642 */
    c->rrr = c->rr * c->r;                                       /* :643 */
    c->h = 2.0 * c->r * c->ellip + c->h2 - c->h1;                /* :644 */
    c->k = 0.5;                                                  /* :655, LAD_05 -> :622-623 */
    c->elai = c->favd * ((1.333333) * c->lambda * M_PI * c->ellip * c->rrr);   /* :657 */
    c->tau = c->k * c->favd;                                     /* :658 */
    c->z1 = c->h1 - c->r * c->ellip;                             /* :669 */
    c->z2 = c->h2 + c->r * c->ellip;                             /* :670 */
    c->lv = c->lambda / (c->h2 - c->h1);                         /* :671 */
    c->favd_p = c->favd * c->ellip;                              /* :675 */
    c->tau_p = c->k * c->favd_p;                                 /* :676 */
    c->lv_p = c->lv * c->ellip;                                  /* :677 */
    c->z1_p = c->z1 / c->ellip;                                  /* :679-682 */
    c->z2_p = c->z2 / c->ellip;
    c->h1_p = c->h1 / c->ellip;
    c->h2_p = c->h2 / c->ellip;
    c->dz = (double) (c->z2 - c->z1) / ((double) NLAY - 1.0);    /* :695 */
    c->ds = c->dz;                                               /* :696 */
    c->dz_p = c->dz / c->ellip;                                  /* :697 */
    c->factorial[0] = 1;                                         /* :752-754 */
    for (int i = 1; i <= MAXCROWNS; i++) c->factorial[i] = c->factorial[i - 1] * (double) i;
    for (int i = NLAY - 1; i >= 0; i--) {                        /* :778-781 */
        c->height[i] = c->z2 - c->dz * (double) (NLAY - 1 - i);
        c->height_p[i] = c->height[i] / c->ellip;
    }
    for (int i = 0; i < NTH; i++) {                              /* :783-797 */
        c->theta[i] = c->dth * (double) i;
        if (c->theta[i] >= M_PI / 2.0) c->theta[i] = M_PI / 2.0 - 1.0 * M_PI / 180.0;
        c->theta_p[i] = atan(tan(c->theta[i]) * c->ellip);
        if (c->theta_p[i] >= M_PI / 2.0) c->theta_p[i] = M_PI / 2.0 - 1.0 * M_PI / 180.0;
    }
}

/* ---------------------------------------------------------------------------------------
 * P(n=0): crown projection geometry, gortt_pn_kopen.c:149-323
 * ------------------------------------------------------------------------------------- */

/* gortt_pn_kopen.c:285-305 */
static double left_circle_area(double r, double x_cut)
{
    double area_tot = M_PI * r * r;
    double ang_sector = acos(fabs(x_cut) / r) * 2.0;
    double area_sector = area_tot * ang_sector / (2.0 * M_PI);
    double area_triangle = fabs(x_cut) * sqrt(r * r - x_cut * x_cut);
    if (x_cut > 0.0) return area_tot - (area_sector - area_triangle);
    return area_sector - area_triangle;
}

/* gortt_pn_kopen.c:309-323 */
static double right_ellipse_area(double r, double b, double x_cut)
{
    double x_cut_p = x_cut / (b / r);
    double a_p = M_PI * r * r;
    a_p -= left_circle_area(r, x_cut_p);
    return a_p * (b / r);
}

/* gortt_pn_kopen.c:233-282 */
static double weird_cross_section(const canopy_t *c, double t, double h, double z)
{
    double zdiff = h - z;
    double r_p = sqrt(c->rr - zdiff * zdiff);
    double x_cc = zdiff * tan(t);
    double x_p = x_cc / (1.0 - cos(t) * cos(t));
    double a_cp = left_circle_area(r_p, x_p - x_cc);
    double a_ep = right_ellipse_area(c->r, c->r * O_SEC(t), x_p);
    return a_cp + a_ep;
}

/* gortt_pn_kopen.c:170-229 */
static double crown_proj_cross_section(const canopy_t *c, double t, double h, double z)
{
    if (z < h - c->r) return 0.0;
    double h_low = h - c->r * sin(t);
    double h_high = h + c->r * sin(t);
    if (z <= h_low) {
        double a = c->rr - (h - z) * (h - z);
        double r_p = (a <= 0) ? 0 : sqrt(a);
        return M_PI * r_p * r_p;
    } else if (z > h_low && z < h_high) {
        return weird_cross_section(c, t, h, z);
    }
    return M_PI * c->rr * O_SEC(t);
}

/* gortt_pn_kopen.c:149-167: midpoint rule with a running-sum loop variable */
static double crown_proj_volume(const canopy_t *c, double t, double h)
{
    double vol = 0.0;
    for (double z = c->h1_p + c->dz_p / 2.0; z <= c->h2_p; z += c->dz_p)
        vol += crown_proj_cross_section(c, t, h, z) * (c->dz_p);
    return vol;
}

/* ---------------------------------------------------------------------------------------
 * Sphere / cylinder volumes for P(n | s'), gortt_pn_kopen.c:665-924
 * ------------------------------------------------------------------------------------- */

/* gortt_pn_kopen.c:858-872 */
static double triang_fcn(double x, double b, double r, double the)
{
    double a1 = tan(the) * (x - b);
    double a2 = r * r - x * x;
    double a3 = a2 - a1 * a1;
    if (fabs(a3) < 0.0000000001) a3 = 0.0;
    return 2.0 * a1 * sqrt(a3);
}

/* gortt_pn_kopen.c:811-854: composite Simpson rule, noint = 20 */
static double triang(double b, double r, double the, int noint)
{
    double sint = sin(the), cost = cos(the);
    double a1 = r * r - b * b * sint * sint;
    double x0 = b * (sint * sint) + sqrt(a1) * cost;
    int m = noint;
    double h = .50 * (x0 - b) / (float) m;
    double sum1 = 0.0;
    for (int i = 0; i < m; i++) sum1 += triang_fcn(b + (float) (2 * i + 1) * h, b, r, the);
    double volume = 4.0 * sum1;
    double sum2 = 0.0;
    for (int i = 0; i < m - 1; i++) sum2 += triang_fcn(b + (float) (2 * (i + 1)) * h, b, r, the);
    volume += 2.0 * sum2;
    volume += triang_fcn(x0, b, r, the);
    volume += triang_fcn(b, b, r, the);
    volume *= h / 3.0;
    return volume;
}

/* gortt_pn_kopen.c:796-806 */
static double sector(double a1, double a2, double r)
{
    double b1 = r * r * a1 - (a1 * a1 * a1) / 3.0;
    double b2 = r * r * a2 - (a2 * a2 * a2) / 3.0;
    return M_PI * (b2 - b1) / 2.0;
}

/* gortt_pn_kopen.c:771-792 */
static double trisec(double hh, double hh_b, double th, double r)
{
    double tmp = (hh - hh_b);
    /* h_0 (:782) is computed by the reference but never used */
    double x = -1.0 * tmp * sin(th) + sqrt(r * r - tmp * tmp) * cos(th);
    double b = -tmp / sin(th);
    return triang(b, r, th, SIMPSON_NOINT) + sector(x, r, r);
}

/* gortt_pn_kopen.c:876-886 */
static double cylind_fcn(double x, double r)
{
    return .50 * x * sqrt(r * r - x * x) + .50 * r * r * asin(x / r);
}

/* gortt_pn_kopen.c:891-924 */
static double cylind(double r, double h1, double h2, double h)
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

/* gortt_pn_kopen.c:665-768: volume of the beam tube (sphere swept along the path from layer
 * h up to layer h_s at zenith index t) lying below the plane h_b. */
static double tube_vol(const canopy_t *c, int h, int h_s, int t, double h_b)
{
    const double *hp = c->height_p;
    const double th = c->theta_p[t];
    const double r = c->r;
    double V, V_sp1, V_sp2, V_cyln, h_t, h_tt;
    double tmp_s = (hp[h_s] - hp[h]) / cos(th);
    double V_0 = M_PI * c->rr * tmp_s;
    V_0 += (4.0 / 3.0) * M_PI * c->rrr;

    if ((hp[h] - r) >= h_b) {
        V = 0.0;
    } else if ((hp[h] - r * sin(th)) >= h_b) {
        h_t = r - (hp[h] - h_b);
        V = (M_PI / 3.0) * h_t * h_t * (3.0 * r - h_t);
    } else if ((hp[h] + r * sin(th)) >= h_b) {
        V_sp1 = (2.0 / 3.0) * M_PI * c->rrr;
        V_sp1 -= trisec(hp[h], h_b, th, r);
        h_tt = (h_b - (hp[h] - r * sin(th))) / cos(th);
        if (hp[h_s] - r * sin(th) >= h_b) {
            double hh1 = (hp[h] - h_b) / sin(th);
            double hh2 = r;
            double hh = h_tt;
            V_cyln = cylind(r, hh1, hh2, hh);
            V_sp2 = 0.0;
        } else {
            double hh1 = (hp[h] - h_b) / sin(th);
            double hh2 = (hp[h_s] - h_b) / sin(th);
            double hh = (hp[h_s] - hp[h]) / cos(th);
            V_cyln = cylind(r, hh1, hh2, hh);
            V_sp2 = trisec(h_b, hp[h_s], th, r);
        }
        V = V_sp1 + V_cyln + V_sp2;
    } else if (hp[h_s] - r * sin(th) >= h_b) {
        double tmp_h = (h_b - hp[h]) / cos(th);
        V_cyln = M_PI * r * r * tmp_h;
        V_sp1 = (2.0 / 3.0) * M_PI * c->rrr;
        V = V_sp1 + V_cyln;
    } else if (hp[h_s] + r * sin(th) >= h_b) {
        h_tt = (hp[h_s] + r * sin(th) - h_b) / cos(th);
        double hh1 = (h_b - hp[h_s]) / sin(th);
        double hh2 = r;
        double hh = h_tt;
        double tmp_h = (hp[h_s] - hp[h]) / cos(th);
        V_cyln = M_PI * r * r * tmp_h - cylind(r, hh1, hh2, hh);
        V_sp2 = trisec(h_b, hp[h_s], th, r);
        V_sp1 = (2.0 / 3.0) * M_PI * c->rrr;
        V = V_cyln + V_sp2 + V_sp1;
    } else if (hp[h_s] + r >= h_b) {
        h_t = r - (h_b - hp[h_s]);
        V_sp1 = (M_PI / 3.0) * h_t * h_t * (3.0 * r - h_t);
        V = V_0 - V_sp1;
    } else {
        V = V_0;
    }
    return V;
}

/* gortt_pn_kopen.c:566-645 */
static double mean_single_crown_path(const canopy_t *c, int z, double h, int th)
{
    const double hz = c->height_p[z];
    if (hz > h + c->r - 0.0001) return 0.0;
    if (hz < h - c->r + 0.0001) return 4.0 * c->r / 3.0;
    double V_sphere = 4.0 * M_PI * c->rrr / 3.0;
    double zdiff = fabs(h - hz);
    double ht = c->r - zdiff;
    double V_slice = M_PI * ht * ht / 3.0 * (3.0 * c->r - ht);
    double V_tot = (hz > h) ? V_slice : V_sphere - V_slice;
    V_tot /= cos(c->theta_p[th]);
    double proj_area;
    if (h < hz) proj_area = crown_proj_cross_section(c, c->theta_p[th], h, (h - zdiff));
    else proj_area = crown_proj_cross_section(c, c->theta_p[th], h, (h + zdiff));
    return V_tot / proj_area;
}

/* gortt_pn_kopen.c:534-563 (+ :648-659 for the uniform crown-centre density) */
static double expected_single_crown_path(const canopy_t *c, int z, int t)
{
    double ES = 0.0;
    double dh = (c->h2_p - c->h1_p) / (double) NH_ES;
    for (double h = c->h1_p + dh / 2.0; h <= c->h2_p; h += dh)
        ES += mean_single_crown_path(c, z, h, t) * ((1.0 / (c->h2_p - c->h1_p)) * dh);
    return ES;
}

/* gortt_pn_kopen.c:134-139 */
static int s_to_index(const canopy_t *c, double s) { return (int) (s / c->ds + 0.5); }

/* gortt_pn_kopen.c:7-129 restricted to what reaches the outputs (h = 0 for pd_s / epgap);
 * p_n0 and v_g are kept for all layers because p_s0 needs them (:40-45). */
static void gap_probabilities_full(const canopy_t *c, double *v_g /*[NLAY][NTH]*/,
                                   double *p_n0 /*[NLAY][NTH]*/, double *epgap0 /*[NTH]*/,
                                   double *k_open0, double *k_openep0)
{
    for (int t = 0; t < NTH; t++)                                /* :24-32 */
        for (int h = 0; h < NLAY; h++) {
            v_g[h * NTH + t] = crown_proj_volume(c, c->theta_p[t], c->height_p[h]);
            p_n0[h * NTH + t] = exp(-1.0 * c->lv_p * v_g[h * NTH + t]);
        }

    for (int t = 0; t < NTH; t++) epgap0[t] = 0.0;

    for (int t = 0; t < NTH - 1; t++) {                          /* epgap only for t < nth-1, :1099 */
        const int h = 0;
        double p_s0[NLAY];                                       /* :40-45 */
        p_s0[NLAY - 1] = 0.0;
        for (int hh = NLAY - 2; hh >= 0; hh--) p_s0[hh] = p_n0[(hh + 1) * NTH + t] - p_n0[hh * NTH + t];

        int s_max = s_to_index(c, (c->z2_p - c->height_p[h]) / cos(c->theta_p[t]));   /* :57 */
        double *pd = (double *) calloc((size_t) s_max + PD_BUFF, sizeof(double));     /* :64-66 */

        /* gortt_get_pd_s, :400-531 */
        double es = expected_single_crown_path(c, h, t);         /* :445 */
        for (int sp_i = NLAY - 1; sp_i > h; sp_i--) {            /* :457 */
            double s_p = (double) (c->height_p[sp_i] - c->height_p[h]) / cos(c->theta_p[t]);   /* :464 */
            if (sp_i == NLAY - 1) { pd[0] += p_s0[sp_i]; continue; }                        /* :466-475 */
            double P_s_p = p_s0[sp_i];                           /* :482 */
            for (int n = 1; n <= MAXCROWNS; n++) {               /* :489 */
                double temp1 = tube_vol(c, h, sp_i, t, c->h2_p) - tube_vol(c, h, sp_i, t, c->h1_p);  /* :496 */
                temp1 *= c->lv_p;                                /* :497 */
                double P_n = (pow(temp1, (double) n) * exp(-temp1)) /
                             (c->factorial[n] * (1.0 - exp(-temp1)));                        /* :501-502 */
                double s = s_p * (1.0 - exp(-1.0 * (double) n * es / s_p));                  /* :508 */
                pd[s_to_index(c, s)] += P_n * P_s_p;             /* :522 */
            }
        }

        /* gortt_calc_epgap, :1083-1125 with gortt_calc_pgap :1129-1140 */
        double e = 0.0;
        for (int s = 0; s <= s_max; s++) e += exp(-((double) s * c->ds) * c->tau_p) * pd[s];
        epgap0[t] = e;
        free(pd);
    }

    /* gortt_calc_kopen, :351-375 for h = 0 */
    double ko = 0.0, ke = 0.0;
    double tmp1_last = p_n0[0] * sin(2.0 * c->theta[0]);
    double tmp2_last = epgap0[0] * sin(2.0 * c->theta[0]);
    for (int t = 1; t < NTH; t++) {
        double tmp1 = p_n0[t] * sin(2.0 * c->theta[t]);
        ko += (tmp1 + tmp1_last) / 2.0 * c->dth;
        tmp1_last = tmp1;
        double tmp2 = epgap0[t] * sin(2.0 * c->theta[t]);
        ke += (tmp2 + tmp2_last) / 2.0 * c->dth;
        tmp2_last = tmp2;
    }
    *k_open0 = ko;
    *k_openep0 = ke;
}

/* gortt_pn_kopen.c:1144-1200: Lewis's closed-form approximation (Quaife et al. 2008), h = 0 only */
static void gap_probabilities_q08(const canopy_t *c, double *p_n0_0, double *epgap0,
                                  double *k_open0, double *k_openep0)
{
    double cc = M_PI * c->rr * c->lambda;                        /* :1164 */
    double l = c->favd * c->b * 4. / 3. * cc;                    /* :1166 */
    double k2 = 0.348535 * pow(cc, (-1.08069 - 0.0874595 * cc)); /* :1168 */
    double k1 = 0.0014166;                                       /* :1169 */
    double a = cc * (exp(k1 * cc * cc) - exp(-k2 * l));          /* :1171 */
    double ko = 0.0, ke = 0.0;
    /* :1176-1177: the "last" terms are taken before row 0 is filled, from calloc'd zeros */
    double tmp1_last = 0.0 * sin(2.0 * c->theta[0]);
    double tmp2_last = 0.0 * sin(2.0 * c->theta[0]);
    p_n0_0[0] = exp(-cc / (cos(c->theta_p[0])));
    epgap0[0] = exp(-a / (cos(c->theta_p[0]))) - p_n0_0[0];
    for (int t = 1; t < NTH; t++) {
        p_n0_0[t] = exp(-cc / (cos(c->theta_p[t])));
        epgap0[t] = exp(-a / (cos(c->theta_p[t]))) - p_n0_0[t];
        double tmp1 = p_n0_0[t] * sin(2.0 * c->theta[t]);
        ko += (tmp1 + tmp1_last) / 2.0 * c->dth;
        tmp1_last = tmp1;
        double tmp2 = epgap0[t] * sin(2.0 * c->theta[t]);
        ke += (tmp2 + tmp2_last) / 2.0 * c->dth;
        tmp2_last = tmp2;
    }
    *k_open0 = ko;
    *k_openep0 = ke;
}

int gort_oracle_lut(const double *st6, int method, double *lut)
{
    canopy_t c;
    canopy_init(&c, st6);
    if (method == 1) {
        gap_probabilities_q08(&c, lut, lut + NTH, &lut[2 * NTH], &lut[2 * NTH + 1]);
    } else {
        double *v_g = (double *) malloc(sizeof(double) * NLAY * NTH * 2);
        double *p_n0 = v_g + NLAY * NTH;
        gap_probabilities_full(&c, v_g, p_n0, lut + NTH, &lut[2 * NTH], &lut[2 * NTH + 1]);
        memcpy(lut, p_n0, sizeof(double) * NTH);
        free(v_g);
    }
    return 0;
}

/* The histogram bins the crown-count loop of gap_probabilities_full reaches (gortt_pn_kopen.c:457-527, h = 0):
 * umax[t] = the largest s / ds + 0.5 over entry heights sp_i < NLAY - 1 and crown counts n, the value that
 * s_to_index truncates; umax[NTH - 1] = 0 (no epgap there).  s depends on E[S] and s' only, so the tube
 * volumes are not evaluated; the s of each (sp_i, n) is formed exactly as above. */
int gort_oracle_lut_bins(const double *st6, double *umax)
{
    canopy_t c;
    canopy_init(&c, st6);
    for (int t = 0; t < NTH; t++) umax[t] = 0.0;
    for (int t = 0; t < NTH - 1; t++) {
        double es = expected_single_crown_path(&c, 0, t);
        for (int sp_i = NLAY - 2; sp_i > 0; sp_i--) {
            double s_p = (double) (c.height_p[sp_i] - c.height_p[0]) / cos(c.theta_p[t]);
            for (int n = 1; n <= MAXCROWNS; n++) {
                double s = s_p * (1.0 - exp(-1.0 * (double) n * es / s_p));
                double u = s / c.ds + 0.5;
                if (u > umax[t]) umax[t] = u;
            }
        }
    }
    return 0;
}

int gort_oracle_lut_intermediates(const double *st6, double *v_g, double *p_n0, double *derived,
                                  double *theta_p, double *height_p)
{
    canopy_t c;
    double epgap0[NTH], ko, ke;
    canopy_init(&c, st6);
    gap_probabilities_full(&c, v_g, p_n0, epgap0, &ko, &ke);
    derived[0] = c.ellip; derived[1] = c.elai; derived[2] = c.tau; derived[3] = c.tau_p;
    derived[4] = c.lv; derived[5] = c.lv_p; derived[6] = c.z1; derived[7] = c.z2;
    derived[8] = c.dz; derived[9] = c.dz_p; derived[10] = c.h1_p; derived[11] = c.h2_p;
    derived[12] = c.z1_p; derived[13] = c.z2_p; derived[14] = c.h; derived[15] = c.favd_p;
    memcpy(theta_p, c.theta_p, sizeof c.theta_p);
    memcpy(height_p, c.height_p, sizeof c.height_p);
    return 0;
}

/* ---------------------------------------------------------------------------------------
 * Geometry of one input line
 * ------------------------------------------------------------------------------------- */
typedef struct {
    double vza, vaa, sza, saa, raa, vza_p, sza_p, fd;
    double pn0_s, pe_s, pn0_v, pe_v;           /* p_neq0 / p_ngt0 at h=0 for sun and view */
} line_t;

/* gortt.c:581-588 */
static double prime_theta(const canopy_t *c, double za) { return atan((c->b / c->r) * tan(za)); }

/* gortt.c:872-915 */
static void zenith_probabilities(const canopy_t *c, const double *lut, line_t *g)
{
    const double *pn0 = lut, *epg = lut + NTH;
    double pos = fabs(g->sza) / c->dth;
    int ci = ceil(pos), fi = floor(pos);
    double d = pos - fi;
    g->pn0_s = d * pn0[ci] + (1.0 - d) * pn0[fi];
    g->pe_s = d * epg[ci] + (1.0 - d) * epg[fi];
    pos = fabs(g->vza) / c->dth;
    ci = ceil(pos); fi = floor(pos);
    d = pos - fi;
    g->pn0_v = d * pn0[ci] + (1.0 - d) * pn0[fi];
    g->pe_v = d * epg[ci] + (1.0 - d) * epg[fi];
}

/* gortt.c:240-291: degrees in, normalised radians + primes + diffuse fraction out */
static void prepare_line(const canopy_t *c, const double *ang4, line_t *g)
{
    g->vza = O_DTOR(ang4[0]); g->vaa = O_DTOR(ang4[1]); g->sza = O_DTOR(ang4[2]); g->saa = O_DTOR(ang4[3]);
    if (g->sza < 0.0) { g->saa += M_PI; g->sza *= -1.0; }
    if (g->vza < 0.0) { g->vaa += M_PI; g->vza *= -1.0; }
    while (g->saa > 2 * M_PI) g->saa -= 2 * M_PI;
    while (g->vaa > 2 * M_PI) g->vaa -= 2 * M_PI;
    while (g->saa < 0) g->saa += 2 * M_PI;
    while (g->vaa < 0) g->vaa += 2 * M_PI;
    g->raa = g->saa - g->vaa;
    g->raa = fabs((g->raa - 2 * M_PI * (int) (0.5 + g->raa * M_1_PI * 0.5)));      /* :279 */
    g->vza_p = prime_theta(c, g->vza);
    g->sza_p = prime_theta(c, g->sza);
    if (c->use_fd) g->fd = c->fd_user;
    else g->fd = cos(g->sza) / (cos(g->sza) + 0.09);                               /* :291 */
}

/* gortt_brdf.c:23-100 (the live branches: "ambrals style" t2, Li & Strahler '92 t1) */
static double overlap_fn(const canopy_t *c, const line_t *g, double raa)
{
    double ts = tan(g->sza_p), tv = tan(g->vza_p);
    double d = pow(ts, 2) + pow(tv, 2) - 2.0 * ts * tv * cos(raa);
    double D = sqrt(O_MAX(0.0, d));
    double t2 = sqrt(D * D + pow((ts * tv * sin(raa)), 2));
    double t1 = (O_SEC(g->sza_p) + O_SEC(g->vza_p));
    double cos_t = (c->h / c->b) * t2 / t1;
    cos_t = O_MAX(-1.0, cos_t);
    cos_t = O_MIN(1.0, cos_t);
    double t = acos(cos_t);
    return O_MAX(0.0, (t - sin(t) * cos_t) * (O_SEC(g->sza_p) + O_SEC(g->vza_p)) / M_PI);
}

/* gortt_brdf.c:7-20 */
static double kg_fn(const canopy_t *c, const line_t *g, double raa)
{
    double overlap = overlap_fn(c, g, raa);
    return exp(-(c->lambda * pow(c->r, 2) * M_PI * (O_SEC(g->sza_p) + O_SEC(g->vza_p) - overlap)));
}

/* gortt_brdf.c:171-238 */
static void kc_fFbeta(const canopy_t *c, const line_t *g, double raa, double Kg,
                      double *f, double *F, double *beta)
{
    double overlap = overlap_fn(c, g, raa);
    double phase_prime = cos(g->vza_p) * cos(g->sza_p) + sin(g->vza_p) * sin(g->sza_p) * cos(raa);
    double Mi = (1.0 - (1.0 - exp(-c->lambda * M_PI * c->rr * O_SEC(g->sza_p))) / (c->lambda * M_PI * c->rr * O_SEC(g->sza_p)));
    double Mv = (1.0 - (1.0 - exp(-c->lambda * M_PI * c->rr * O_SEC(g->vza_p))) / (c->lambda * M_PI * c->rr * O_SEC(g->vza_p)));
    double Gamma = M_PI * c->rr * (O_SEC(g->sza_p) + O_SEC(g->vza_p) - overlap);
    double Gamma_c = M_PI * c->rr * O_SEC(g->vza_p) * 0.5 * (1.0 + phase_prime);
    double Gamma_v = M_PI * c->rr * O_SEC(g->vza_p);
    *F = Gamma_c / Gamma;
    double M = 1.0 - (1.0 - Kg) / (c->lambda * Gamma);
    double theta_Mi = acos(1.0 - 2.0 * Mi);
    double Gamma_i = Gamma_v;
    double PiMi = (1 - cos(theta_Mi * (1 - (g->sza_p - g->vza_p * cos(raa)) / M_PI))) / 2.0;
    double PvMv = Mv - (1.0 - cos(g->vza_p * cos(raa) - g->sza_p)) / 2.0;
    double Po;
    if ((raa < O_DTOR(270.)) && (raa > O_DTOR(90.))) Po = PvMv;
    else if (fabs(g->vza) > fabs(g->sza)) Po = PiMi;
    else Po = PvMv;
    if (g->sza_p < 0.000000001) {
        *beta = 0.0;
    } else {
        double D = c->r * (1.0 / tan(g->sza_p / 2.0));
        *beta = (c->lambda * Gamma_i) / (c->lambda * Gamma_i + (c->h2 - c->h1) / D)
                * (1.0 - exp(-c->lambda * Gamma_i - (c->h2 - c->h1) / D)) / (1.0 - exp(-c->lambda * Gamma_i));
    }
    *f = *F * (1.0 - Gamma_v * (PvMv + PiMi - Po) / Gamma_c) / (1.0 - M);
}

/* gortt_brdf.c:118-169 */
static double kc_fn(const canopy_t *c, const line_t *g, double Kg)
{
    double f, F, beta, junk, f0, F0, f180, F180;
    kc_fFbeta(c, g, g->raa, Kg, &f, &F, &beta);
    double Kg0 = kg_fn(c, g, O_DTOR(0.));
    kc_fFbeta(c, g, O_DTOR(0.), Kg0, &f0, &F0, &junk);
    double Kg180 = kg_fn(c, g, O_DTOR(180.));
    kc_fFbeta(c, g, O_DTOR(180.), Kg180, &f180, &F180, &junk);
    double frac = g->raa / M_PI;
    if (frac > 1.0) frac = 2.0 - frac;
    if (c->use_beta) beta = c->beta;
    f = (1. - frac) * f0 * F0 + frac * f180 * F180;
    f = beta * f + (1.0 - beta) * F;
    return f * (1.0 - Kg);
}

/* gortt_brdf.c:638-702; k = k_vza = 0.5 (gortt.c:287,655) */
static double kuusk_fn(const canopy_t *c, const line_t *g)
{
    double cos_xi = cos(g->sza) * cos(g->vza) + sin(g->sza) * sin(g->vza) * cos(g->raa);
    double lsza = -log(g->pe_s) / (c->k * c->favd);
    double lvza = -log(g->pe_v) / (0.5 * c->favd);
    double t1, t2;
    if ((lsza * lsza + lvza * lvza - 2. * lsza * lvza * cos_xi) > 0.0) {
        double lsv = sqrt(lsza * lsza + lvza * lvza - 2. * lsza * lvza * cos_xi);
        t2 = (1.0 - exp(-lsv / c->r)) / (lsv / c->r);
    } else {
        t2 = 1.0;
    }
    if ((lsza * lvza) > 0.0) t1 = sqrt(lsza * lvza);
    else t1 = 0.0;
    double H = exp(c->k * c->favd * t1 * t2);
    return g->pe_s * g->pe_v * H;
}

/* gortt.c:385-578 for one prepared line */
static void rsurf_line(const canopy_t *c, const double *lut, const line_t *g, int nw,
                       const double *rleaf, const double *tleaf, const double *rsoil,
                       double *rsurf, double *scomp, double *kprop)
{
    const double k_open0 = lut[2 * NTH], k_openep0 = lut[2 * NTH + 1];
    /* geometric "kernels", gortt.c:424-449 */
    double Kg = kg_fn(c, g, g->raa);
    double Kc = kc_fn(c, g, Kg);
    double Kz = exp(-(c->lambda * M_PI * pow(c->r, 2)) / cos(g->vza_p)) - Kg;
    double Kt = 1.0 - Kc - Kz - Kg;
    Kt = O_MAX(0.0, Kt);
    double Kprime_g = exp(-(c->lambda * M_PI * c->rr) / cos(g->sza_p)) - Kg;
    double Kprime_z = 1.0 - exp(-(c->lambda * M_PI * c->rr) / cos(g->vza_p)) - Kprime_g;
    const double fd = g->fd;
    const double kuusk = kuusk_fn(c, g);                          /* wavelength independent */

    for (int i = 0; i < nw; i++) {                               /* gortt.c:460-567 */
        double omega = rleaf[i] + tleaf[i];                      /* :469 */
        double gam = sqrt(1 - omega);                            /* :470 */
        double rs = rsoil[i];

        /* two-stream terms, gortt_brdf.c */
        double T_inf_ff = exp(-(2.0 * gam * c->k * c->elai));                    /* :492 */
        double R_inf_ff = (1.0 - gam) / (1.0 + gam);                             /* :574 */
        double t_0 = exp(-(c->k * c->elai * O_SEC(g->sza_p)));                   /* :534 */
        double R_inf_df = (1.0 - gam) / (1.0 + 2.0 * cos(g->sza_p) * gam);       /* :552 */
        double T_inf_df = (omega / 2.0);                                         /* :467-471 */
        T_inf_df *= (1. + 2. * cos(g->sza_p)) / (1. - pow((2. * gam * cos(g->sza_p)), 2));
        T_inf_df *= (T_inf_ff - t_0);
        double p_ff = R_inf_ff;                                                  /* :510-512 */
        p_ff *= (1. - pow(T_inf_ff, 2));
        p_ff /= (1. - pow(T_inf_ff * R_inf_ff, 2));
        double t_ff = T_inf_ff;                                                  /* :401-403 */
        t_ff *= (1. - pow(R_inf_ff, 2));
        t_ff /= (1. - pow(R_inf_ff * T_inf_ff, 2));
        double t_df = T_inf_df - p_ff * (t_0 * R_inf_df + T_inf_df * R_inf_ff);  /* :423-424 */
        double p_df = R_inf_df - t_ff * (t_0 * R_inf_df + T_inf_df * R_inf_ff);  /* :628-630 */
        double t_prime_0 = g->pn0_s + g->pe_s;                                   /* :447 */
        double t_prime_df = t_df * (1 - t_prime_0);                              /* :361 */
        double k_open = k_open0 + k_openep0;                                     /* :381 */
        double t_prime_ff = t_ff * (1.0 - k_open) + k_open;                      /* :382 */
        double gfunc = -(4.0 / 9.0) * (rleaf[i] - tleaf[i]) / (omega);           /* :591 */

        /* gortt.c:481-557 */
        double G = fd * rs + (1 - fd) * rs;
        double Zd = (t_prime_df + g->pe_s) * rs;
        double Zf = (t_prime_ff - k_openep0) * rs;
        double Z = fd * Zd + (1 - fd) * Zf;
        double CdC = p_df + ((1.0 - omega) * kuusk * omega * (1.0 - gfunc)) / (2.0 * cos(g->sza_p) * cos(g->vza_p));
        double CfC = p_ff;
        double CdG = (Z * Kprime_z + G * Kprime_g) * k_openep0;
        double CfG = ((k_openep0 + k_open0) * G + (1 - (k_openep0 + k_open0)) * Z) * k_openep0;
        double CdCG = (t_prime_df + t_prime_0) * (rs / (1.0 - rs * p_ff)) * (t_prime_ff - k_open0);
        double CfCG = t_prime_ff * (rs / (1.0 - rs * p_ff)) * (t_prime_ff - k_open0);
        double Cd = CdC + CdG + CdCG;
        double Cf = CfC + CfG + CfCG;
        double C = fd * Cd + (1 - fd) * Cf;
        double Td = CdCG, Tf = CfCG;                             /* :541-547 are the same expressions */
        double T = fd * Td + (1 - fd) * Tf;
        rsurf[i] = Kc * C + Kg * G + Kt * T + Kz * Z;
        if (scomp) { scomp[4 * i] = C; scomp[4 * i + 1] = G; scomp[4 * i + 2] = T; scomp[4 * i + 3] = Z; }
    }
    if (kprop) { kprop[0] = Kc; kprop[1] = Kg; kprop[2] = Kt; kprop[3] = Kz; }
}

static void canopy_options(canopy_t *c, const double *opt)
{
    if (!opt) return;
    if (opt[0] != 0.0) { c->use_beta = 1; c->beta = opt[1]; }
    if (opt[2] != 0.0) { c->use_fd = 1; c->fd_user = opt[3]; }
}

int gort_oracle_brdf(const double *st6, const double *lut, const double *opt,
                     int ngeom, const double *ang, int nw,
                     const double *rleaf, const double *tleaf, const double *rsoil,
                     double *rsurf, double *scomp, double *kprop)
{
    canopy_t c;
    canopy_init(&c, st6);
    canopy_options(&c, opt);
    for (int i = 0; i < ngeom; i++) {
        line_t g;
        prepare_line(&c, ang + 4 * i, &g);
        zenith_probabilities(&c, lut, &g);
        rsurf_line(&c, lut, &g, nw, rleaf, tleaf, rsoil, rsurf + (size_t) i * nw,
                   scomp ? scomp + (size_t) i * nw * 4 : NULL, kprop ? kprop + 4 * i : NULL);
    }
    return 0;
}

long gort_oracle_brdf_repeat(const double *st6, const double *lut, int ngeom, const double *ang, int nw,
                             const double *rleaf, const double *tleaf, const double *rsoil,
                             int reps, double *rsurf_last)
{
    long n = 0;
    double *buf = (double *) malloc(sizeof(double) * (size_t) ngeom * nw);
    for (int r = 0; r < reps; r++) {
        gort_oracle_brdf(st6, lut, NULL, ngeom, ang, nw, rleaf, tleaf, rsoil, buf, NULL, NULL);
        n += (long) ngeom * nw;
    }
    if (rsurf_last) memcpy(rsurf_last, buf, sizeof(double) * (size_t) ngeom * nw);
    free(buf);
    return n;
}

/* ---------------------------------------------------------------------------------------
 * Hemispherical integrals, gortt_albedo.c
 * ------------------------------------------------------------------------------------- */

/* gortt_albedo.c:141-199 (Numerical-Recipes Gauss-Legendre, zero-indexed) */
void gort_oracle_gauleg(int n, double *x, double *w)
{
    const double x1 = -1., x2 = 1.;
    int m = (n + 1) / 2;
    double xm = 0.5 * (x2 + x1), xl = 0.5 * (x2 - x1);
    for (int i = 0; i < m; i++) {
        double z = cos(3.141592654 * (i + 0.75) / (n + 0.5)), z1, pp;
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
        } while (fabs(z - z1) > 3.0e-11);
        x[i] = xm - xl * z;
        x[n - 1 - i] = xm + xl * z;
        w[i] = 2.0 * xl / ((1.0 - z * z) * pp * pp);
        w[n - 1 - i] = w[i];
    }
}

/* gortt_albedo.c:62-138 then :7-60, for one sun geometry; nw is unrestricted here (the
 * reference's scratch overflow for nw > 32, gortt_albedo.c:79-88, is not inherited) */
static void energy_line(const canopy_t *c, const double *lut, const double *ang4, int nw,
                        const double *rleaf, const double *tleaf, const double *rsoil,
                        const double *absc, const double *wts, int npoints,
                        double *albedo, double *favegt, double *fasoil)
{
    line_t g;
    prepare_line(c, ang4, &g);
    zenith_probabilities(c, lut, &g);
    double *sum_y = (double *) calloc(nw, sizeof(double));
    double *sum_x = (double *) calloc(nw, sizeof(double));
    double *rs = (double *) malloc(sizeof(double) * nw);
    double *sc = (double *) malloc(sizeof(double) * nw * 4);
    const double xm = 0.5 * (1. - 1.), xr = 0.5 * (1. + 1.);
    const double ym = 0.5 * (2. * M_PI - 0.), yr = 0.5 * (2. * M_PI + 0.);
    for (int k = 0; k < nw; k++) sum_y[k] = 0.;
    for (int i = 0; i < npoints; i++) {
        double y = ym + yr * absc[i];
        g.vaa = y;
        while (g.vaa > 2 * M_PI) g.vaa -= 2 * M_PI;
        g.raa = g.saa - g.vaa;
        g.raa = fabs((g.raa - 2 * M_PI * (int) (0.5 + g.raa * M_1_PI * 0.5)));
        for (int k = 0; k < nw; k++) sum_x[k] = 0.;
        for (int j = npoints / 2.; j < npoints; j++) {
            double x = xm + xr * absc[j];
            g.vza = acos(x);
            if (g.vza < 0.0) { g.vaa += M_PI; g.vza *= -1.0; }
            g.vza_p = prime_theta(c, g.vza);
            g.sza_p = prime_theta(c, g.sza);
            zenith_probabilities(c, lut, &g);
            rsurf_line(c, lut, &g, nw, rleaf, tleaf, rsoil, rs, sc, NULL);
            for (int k = 0; k < nw; k++) sum_x[k] = sum_x[k] + rs[k] * wts[j] * fabs(x) * xr;
        }
        for (int k = 0; k < nw; k++) sum_y[k] = sum_y[k] + sum_x[k] * wts[i] * yr;
    }
    for (int k = 0; k < nw; k++) albedo[k] = sum_y[k] / M_PI;

    /* gortt_energy, gortt_albedo.c:37-52 */
    const double Fd1 = 1., Pn0 = g.pn0_s;
    for (int k = 0; k < nw; k++) {
        double Fu1 = albedo[k];
        double G = sc[4 * k + 1], Z = sc[4 * k + 3];
        double Fu2 = G * Pn0 + Z * (1. - Pn0);
        double Fd2 = Pn0 + Z * (1. - Pn0) / rsoil[k];
        favegt[k] = Fd1 - Fu1 - Fd2 + Fu2;
        fasoil[k] = Fd2 - Fu2;
    }
    free(sum_x); free(sum_y); free(rs); free(sc);
}

int gort_oracle_energy(const double *st6, const double *lut, const double *opt,
                       int ngeom, const double *ang, int nw,
                       const double *rleaf, const double *tleaf, const double *rsoil,
                       double *albedo, double *favegt, double *fasoil)
{
    canopy_t c;
    double absc[32], wts[32];
    canopy_init(&c, st6);
    canopy_options(&c, opt);
    gort_oracle_gauleg(32, absc, wts);                           /* gortt.c:93,209 */
    for (int i = 0; i < ngeom; i++)
        energy_line(&c, lut, ang + 4 * i, nw, rleaf, tleaf, rsoil, absc, wts, 32,
                    albedo + (size_t) i * nw, favegt + (size_t) i * nw, fasoil + (size_t) i * nw);
    return 0;
}

/* ---------------------------------------------------------------------------------------
 * Spectra: Price soil (gortt.c:1286-1328) and the PROSPECT interface (gortt.c:1331-1374)
 * ------------------------------------------------------------------------------------- */
static double f64bits(uint64_t u) { double d; memcpy(&d, &u, sizeof d); return d; }

static double soil_eof_sum(const double *w, int idx)
{
    /* one-past-the-end read at 2500 nm (gortt.c:1311,1318) is multiplied by a zero fraction
     * in the reference; return 0 instead of reading out of bounds */
    if (idx >= GORT_SOIL_NW) return 0.0;
    return w[0] * f64bits(gort_tab_soil_eof1_f64[idx]) + w[1] * f64bits(gort_tab_soil_eof2_f64[idx])
         + w[2] * f64bits(gort_tab_soil_eof3_f64[idx]) + w[3] * f64bits(gort_tab_soil_eof4_f64[idx]);
}

int gort_oracle_spectra(const double *leaf7, const double *soil4, double user_leaf, double user_soil,
                        int nw, const double *wl, double *rleaf, double *tleaf, double *rsoil)
{
    static double refl[GORT_PROSPECT_NW + 1], tran[GORT_PROSPECT_NW + 1];
    for (int i = 0; i < nw; i++)
        if (wl[i] < 400 || wl[i] > 2500) return 1;               /* gortt.c:1299-1302, :1350-1353 */
    for (int i = 0; i < nw; i++) {                               /* gortt.c:1297-1324 */
        if (user_soil >= 0.0) { rsoil[i] = user_soil; continue; }
        int upper = 1. + (wl[i] - 400) / 5.0;
        int lower = (wl[i] - 400) / 5.0;
        double fraction = (double) (wl[i] - 400.) / 5.0 - lower;
        double rs_lower = soil_eof_sum(soil4, lower);
        double rs_upper = soil_eof_sum(soil4, upper);
        rsoil[i] = rs_lower * (1 - fraction) + rs_upper * fraction;
    }
    if (user_leaf < 0.0) {
        gort_oracle_prospect_full(leaf7, refl, tran);
        refl[GORT_PROSPECT_NW] = 0.0; tran[GORT_PROSPECT_NW] = 0.0;   /* see soil_eof_sum note */
    }
    for (int i = 0; i < nw; i++) {                               /* gortt.c:1349-1371 */
        if (user_leaf >= 0.0) {
            rleaf[i] = user_leaf / 2.0;
            tleaf[i] = user_leaf / 2.0;
        } else {
            int upper = 1 + (wl[i] - 400.0) / 1.0;
            int lower = (wl[i] - 400.0) / 1.0;
            float fraction = (float) (wl[i] - 400.0) / 1.0 - lower;   /* float, gortt.c:1338,1364 */
            rleaf[i] = refl[lower] * (1 - fraction) + refl[upper] * fraction;
            tleaf[i] = tran[lower] * (1 - fraction) + tran[upper] * fraction;
        }
    }
    return 0;
}

/* ---------------------------------------------------------------------------------------
 * Soil spectrum file: gortt_read_soil_lut, gortt.c:1388-1451 (the reference stops after building the
 * table -- it prints it and exits; the interpolation loop :1404-1433 is what is restated here) and the
 * lookup gortt_get_rsoil_lut (declared include/gortt.h:296, never defined) in the form DESIGN.md gives
 * it: gortt_price_soil's index / fraction arithmetic (gortt.c:1311-1321) on the 1-nm table.
 * Return: 0 ok, 1 cannot open, 2 unparsable line, 3 first wavelength > 400, 4 last wavelength < 2500;
 * *where receives the line number / wavelength the reference's message would print.
 * ------------------------------------------------------------------------------------- */
int gort_oracle_soil_table(const char *path, double *table, double *where)
{
    FILE *fp;
    char line[1000];                                             /* MAX_LINE_LEN, include/gortt.h:28 */
    int n = 0, i, index;
    double this_wl, this_rs, last_wl = 0, last_rs = 0;
    for (i = 0; i <= 2100; i++) table[i] = 0.0;
    if ((fp = fopen(path, "r")) == NULL) return 1;               /* :1399 */
    while (fgets(line, 1000, fp) != NULL) {                      /* :1404 */
        n++;
        if (sscanf(line, "%lf %lf", &this_wl, &this_rs) != 2) { *where = n + 1; fclose(fp); return 2; }   /* :1407 */
        if (n == 1 && this_wl > 400) { *where = this_wl; fclose(fp); return 3; }                          /* :1412 */
        if (n > 1) {
            for (i = ceil(last_wl); i <= floor(this_wl); i++) {  /* :1420 */
                index = i - 400;
                if ((index >= 0) && (index <= 2100))
                    table[index] = last_rs + (i - last_wl) / (this_wl - last_wl) * (this_rs - last_rs);   /* :1425 */
            }
        }
        last_wl = this_wl;
        last_rs = this_rs;
    }
    fclose(fp);
    if (last_wl < 2500) { *where = last_wl; return 4; }          /* :1435 */
    return 0;
}

int gort_oracle_soil_lookup(const double *table, int nw, const double *wl, double *rsoil)
{
    for (int i = 0; i < nw; i++)
        if (wl[i] < 400 || wl[i] > 2500) return 1;
    for (int i = 0; i < nw; i++) {
        int upper = 1. + (wl[i] - 400) / 1.0;
        int lower = (wl[i] - 400) / 1.0;
        double fraction = (double) (wl[i] - 400.) / 1.0 - lower;
        double rs_lower = table[lower];
        double rs_upper = upper <= 2100 ? table[upper] : 0.0;   /* zero weight at 2500 nm, as soil_eof_sum */
        rsoil[i] = rs_lower * (1 - fraction) + rs_upper * fraction;
    }
    return 0;
}

/* ---------------------------------------------------------------------------------------
 * The intermediates of the gap-probability code that never reach the BRDF (SURVEY.md 8f row 1):
 * gortt_calc_vb :925-972, gortt_calc_fb :975-1006, gortt_calc_t_open :1010-1078 and the dk_open /
 * k_open[h] rows of gortt_calc_kopen :351-375.  Outputs: vb[15], fb[15][91], t_open[15][15],
 * dt_open[15][15], dk_open[15], k_open[15].
 * ------------------------------------------------------------------------------------- */
#include <float.h>
int gort_oracle_lut_dead(const double *st6, double *vb, double *fb, double *t_open, double *dt_open,
                         double *dk_open, double *k_open)
{
    canopy_t c;
    canopy_init(&c, st6);
    double *v_g = (double *) malloc(sizeof(double) * NLAY * NTH * 2);
    double *p_n0 = v_g + NLAY * NTH;
    double epgap0[NTH], ko0, ke0;
    gap_probabilities_full(&c, v_g, p_n0, epgap0, &ko0, &ke0);

    for (int i = 0; i < NLAY; i++) {                             /* gortt_calc_vb, :938-970 */
        double Vol = 4.0 * M_PI * c.rrr / 3.0, tmp;
        if (c.height_p[i] + c.r > c.h2_p) {
            tmp = c.height_p[i] + c.r - c.h2_p;
            Vol -= M_PI * tmp * tmp * (3.0 * c.r - tmp) / 3.0;
        }
        if (c.height_p[i] - c.r < c.h1_p) {
            tmp = c.h1_p - (c.height_p[i] - c.r);
            Vol -= M_PI * tmp * tmp * (3.0 * c.r - tmp) / 3.0;
        }
        if (Vol < -0.0000001) { free(v_g); return 1; }           /* the reference exits here */
        if (Vol < 0) Vol = 0.0;
        vb[i] = Vol;
    }
    for (int t = 0; t < NTH; t++)                                /* gortt_calc_fb, :981-1003 */
        for (int i = 0; i < NLAY; i++) {
            double d = (1.0 - p_n0[i * NTH + t]);
            if (d < DBL_MIN * 2.) d = DBL_MIN * 2.;
            fb[i * NTH + t] = (1.0 - exp(-c.lv_p * vb[i])) / d;
        }
    for (int i = 0; i < NLAY * NLAY; i++) { t_open[i] = 0.0; dt_open[i] = 0.0; }
    for (int z = 0; z < NLAY; z++)                               /* gortt_calc_t_open, :1033-1075 */
        for (int h = NLAY - 1; h >= z; h--) {
            t_open[h * NLAY + z] = 0.0;
            dt_open[h * NLAY + z] = 0.0;
            if (z != h) {
                for (int t = 0; t < NTH; t++) {
                    double T = 0.0, dT = 0.0;
                    double s_p = fabs(c.height_p[z] - c.height_p[h]) / cos(c.theta_p[t]);
                    for (int n = 1; n <= MAXCROWNS; n++) {
                        double s = s_p * (1.0 - exp(-n * expected_single_crown_path(&c, z, t) / s_p));
                        double temp1 = c.lv_p * M_PI * c.r * c.r * s_p;
                        double P_n = (pow(temp1, (double) n) * exp(-temp1)) / (c.factorial[n] * (1.0 - exp(-temp1)));
                        T += P_n * exp(-s * c.tau_p);
                        double ds = (1.0 - exp(c.lv_p * vb[z])) * c.dz_p / cos(c.theta_p[t]);      /* sic: + exponent */
                        dT += P_n * exp(-s * c.tau_p) * (1.0 - exp(c.tau_p * ds));
                    }
                    t_open[h * NLAY + z] += sin(2.0 * c.theta[t]) * T * c.dth;
                    dt_open[h * NLAY + z] += sin(2.0 * c.theta[t]) * dT * c.dth;
                    t_open[z * NLAY + h] = t_open[h * NLAY + z];
                    dt_open[z * NLAY + h] = dt_open[h * NLAY + z];
                }
            } else {
                for (int t = 0; t < NTH; t++) {
                    double ds = 0.5 * (1.0 - exp(-c.lv_p * vb[z])) * c.dz_p / cos(c.theta_p[t]);
                    double dT = 1.0 - exp(-c.tau_p * ds);
                    dt_open[h * NLAY + z] += sin(2.0 * c.theta[t]) * dT * c.dth;
                }
            }
        }
    for (int h = 0; h < NLAY; h++) {                             /* gortt_calc_kopen, :351-375 */
        double ko = 0.0, dk = 0.0;
        double ps_last = (h == NLAY - 1 ? 0.0 : p_n0[(h + 1) * NTH] - p_n0[h * NTH]);
        double tmp1_last = p_n0[h * NTH] * sin(2.0 * c.theta[0]);
        double tmp3_last = ps_last * sin(2.0 * c.theta[0]);
        for (int t = 1; t < NTH; t++) {
            double tmp1 = p_n0[h * NTH + t] * sin(2.0 * c.theta[t]);
            ko += (tmp1 + tmp1_last) / 2.0 * c.dth;
            tmp1_last = tmp1;
            double ps = (h == NLAY - 1 ? 0.0 : p_n0[(h + 1) * NTH + t] - p_n0[h * NTH + t]);     /* p_s0, :40-45 */
            double tmp3 = ps * sin(2.0 * c.theta[t]);
            dk += (tmp3 + tmp3_last) / 2.0 * c.dth;
            tmp3_last = tmp3;
        }
        k_open[h] = ko;
        dk_open[h] = dk;
    }
    free(v_g);
    return 0;
}
