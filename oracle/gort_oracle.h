/* oracle/gort_oracle.h -- TEST INFRASTRUCTURE, not product code.
 * Plain-C CPU restatement of the reference GORT hot path (tquaife/gort), used only as the
 * parity checker by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg.
 * Entry points have the same signatures as oracle/ref_harness.c so tests can run either.
 */
#ifndef GORT_ORACLE_H
#define GORT_ORACLE_H

#define GORT_ORACLE_NTH 91
#define GORT_ORACLE_NLAYERS 15
#define GORT_ORACLE_LUT_LEN (2 * GORT_ORACLE_NTH + 2)

/* st6 = lambda, r, b, h1, h2, favd.  lut = p_n0[0][0..90], epgap[0][0..90], k_open[0], k_openep[0]. */
int gort_oracle_lut(const double *st6, int method, double *lut);
int gort_oracle_lut_intermediates(const double *st6, double *v_g, double *p_n0, double *derived,
                                  double *theta_p, double *height_p);
/* umax[t] = largest s/ds + 0.5 the crown-count loop of the full method reaches at zenith t (the value truncated to a
 * histogram bin); umax[NTH - 1] = 0 */
int gort_oracle_lut_bins(const double *st6, double *umax);
int gort_oracle_brdf(const double *st6, const double *lut, const double *opt,
                     int ngeom, const double *ang, int nw,
                     const double *rleaf, const double *tleaf, const double *rsoil,
                     double *rsurf, double *scomp, double *kprop);
int gort_oracle_energy(const double *st6, const double *lut, const double *opt,
                       int ngeom, const double *ang, int nw,
                       const double *rleaf, const double *tleaf, const double *rsoil,
                       double *albedo, double *favegt, double *fasoil);
int gort_oracle_spectra(const double *leaf7, const double *soil4, double user_leaf, double user_soil,
                        int nw, const double *wl, double *rleaf, double *tleaf, double *rsoil);
void gort_oracle_gauleg(int n, double *x, double *w);
long gort_oracle_brdf_repeat(const double *st6, const double *lut, int ngeom, const double *ang, int nw,
                             const double *rleaf, const double *tleaf, const double *rsoil,
                             int reps, double *rsurf_last);

/* intermediates that never reach the BRDF (gortt_calc_vb / _fb / _t_open, dk_open; gortt_pn_kopen.c:925-1078, :351-375) */
int gort_oracle_lut_dead(const double *st6, double *vb, double *fb, double *t_open, double *dt_open,
                         double *dk_open, double *k_open);

/* soil spectrum file (gortt_read_soil_lut, gortt.c:1388-1451) and the 1-nm lookup */
int gort_oracle_soil_table(const char *path, double *table, double *where);
int gort_oracle_soil_lookup(const double *table, int nw, const double *wl, double *rsoil);

/* from prospect_d_oracle.c */
void gort_oracle_prospect_full(const double *leaf7, double *refl2101, double *tran2101);
double gort_oracle_tav_abs(double theta_deg, double nr);
double gort_oracle_plate_tau(double k);

#endif
