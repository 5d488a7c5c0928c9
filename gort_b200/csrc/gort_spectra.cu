// gort_spectra.cu -- PROSPECT-D leaf optics and Price soil reflectance (sm_100a, FP64).
//
// Replaces gortt_price_soil (gortt.c:1286-1328), gortt_prospect_interface (gortt.c:1331-1374) and
// the Fortran prospect_DB / tav_abs (PROSPECT-D/prospect_DB.f90:72-191, tav_abs.f90:16-60).
//
// gfortran semantics of the reference build are kept (SURVEY.md App. B4): the spectral tables are
// binary32 constants widened to FP64 (gort_tables.h), tav_abs's pi is single-precision pi, real
// exponents (**2., **3.) go through pow(), integer exponents are repeated products.
//
//   tav_kernel       once per context: tav_abs(90 deg) and tav_abs(40 deg) for the 2101-entry
//                    refractive-index table -- they depend on no leaf parameter.
//   spectra_kernel   one thread per (parameter set, requested wavelength): evaluates PROSPECT-D only
//                    at the two table rows the reference's linear interpolation touches (1 at 2500 nm)
//                    and the Price EOF sum.  Coalesced [M][W] stores.
//   prospect_full_kernel  the whole 2101-band RT array of prospect_DB_, [M][2101].
#include <string.h>
#include "gort_internal.h"
#include "../data/gort_tables.h"

#define NWP GORT_PROSPECT_NW

namespace gort {

// table rows inside ctx->d_prospect
enum { T_NR = 0, T_CAB, T_CAR, T_ANTH, T_BROWN, T_CW, T_CM, T_TAV90, T_TAV40, T_ROWS };

// tav_abs.f90:16-60
__device__ double tav_abs_dev(double theta, double nr)
{
    const double pi = (double) 3.14159274101257324f;       // :30  atan(1.)*4. in REAL(4)
    const double rd = pi / 180.0;                           // :31
    const double n2 = pow(nr, 2.0);                         // :32
    const double np = n2 + 1.0;
    const double nm = n2 - 1.0;
    const double a = ((nr + 1.0) * (nr + 1.0)) / 2.0;       // :35
    const double k = -(((n2 - 1.0) * (n2 - 1.0)) / 4.0);    // :36
    const double sa = sin(theta * rd);                      // :37
    double b1;
    if (theta == 90.0) b1 = 0.0;                            // :39-43
    else b1 = sqrt((sa * sa - np / 2.0) * (sa * sa - np / 2.0) + k);
    const double b2 = sa * sa - np / 2.0;
    const double b = b1 - b2;
    const double b3 = (b * b) * b;
    const double a3 = (a * a) * a;
    const double ts = ((pow(k, 2.0) / (6.0 * b3) + k / b) - b / 2.0)
                    - ((pow(k, 2.0) / (6.0 * a3) + k / a) - a / 2.0);            // :49
    const double tp1 = -(((2.0 * n2) * (b - a)) / (np * np));
    const double tp2 = -((((2.0 * n2) * np) * log(b / a)) / (nm * nm));
    const double tp3 = (n2 * (1.0 / b - 1.0 / a)) / 2.0;
    const double tp4 = (((16.0 * pow(n2, 2.0)) * (n2 * n2 + 1.0))
                        * log(((2.0 * np) * b - nm * nm) / ((2.0 * np) * a - nm * nm)))
                       / (pow(np, 3.0) * (nm * nm));
    const double tp5 = ((16.0 * pow(n2, 3.0))
                        * (1.0 / ((2.0 * np) * b - nm * nm) - 1.0 / ((2.0 * np) * a - nm * nm)))
                       / ((np * np) * np);
    const double tp = (((tp1 + tp2) + tp3) + tp4) + tp5;
    return (ts + tp) / (2.0 * (sa * sa));
}

__global__ void tav_kernel(double* __restrict__ tab)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= NWP) return;
    double nr = tab[T_NR * NWP + i];
    tab[T_TAV90 * NWP + i] = tav_abs_dev(90.0, nr);          // prospect_DB.f90:145-146
    tab[T_TAV40 * NWP + i] = tav_abs_dev(40.0, nr);          // :147-148
}

// prospect_DB.f90:104-141
__device__ double plate_tau_dev(double k)
{
    double xx, yy;
    if (k <= 0.0) return 1.0;
    if (k <= 4.0) {
        xx = 0.5 * k - 1.0;
        yy = (((((((((((((((-3.60311230482612224e-13
            * xx + 3.46348526554087424e-12) * xx - 2.99627399604128973e-11)
            * xx + 2.57747807106988589e-10) * xx - 2.09330568435488303e-9)
            * xx + 1.59501329936987818e-8) * xx - 1.13717900285428895e-7)
            * xx + 7.55292885309152956e-7) * xx - 4.64980751480619431e-6)
            * xx + 2.63830365675408129e-5) * xx - 1.37089870978830576e-4)
            * xx + 6.47686503728103400e-4) * xx - 2.76060141343627983e-3)
            * xx + 1.05306034687449505e-2) * xx - 3.57191348753631956e-2)
            * xx + 1.07774527938978692e-1) * xx - 2.96997075145080963e-1;
        yy = (yy * xx + 8.64664716763387311e-1) * xx + 7.42047691268006429e-1;
        yy = yy - log(k);
        return (1.0 - k) * exp(-k) + (k * k) * yy;
    }
    if (k <= 85.0) {
        xx = 14.5 / (k + 3.25) - 1.0;
        yy = (((((((((((((((-1.62806570868460749e-12
            * xx - 8.95400579318284288e-13) * xx - 4.08352702838151578e-12)
            * xx - 1.45132988248537498e-11) * xx - 8.35086918940757852e-11)
            * xx - 2.13638678953766289e-10) * xx - 1.10302431467069770e-9)
            * xx - 3.67128915633455484e-9) * xx - 1.66980544304104726e-8)
            * xx - 6.11774386401295125e-8) * xx - 2.70306163610271497e-7)
            * xx - 1.05565006992891261e-6) * xx - 4.72090467203711484e-6)
            * xx - 1.95076375089955937e-5) * xx - 9.16450482931221453e-5)
            * xx - 4.05892130452128677e-4) * xx - 2.14213055000334718e-3;
        yy = ((yy * xx - 1.06374875116569657e-2) * xx - 8.50699154984571871e-2) * xx
             + 9.23755307807784058e-1;
        yy = (exp(-k) * yy) / k;
        return (1.0 - k) * exp(-k) + (k * k) * yy;
    }
    return 0.0;
}

struct Leaf7 { double N, Cab, Car, Anth, Cbrown, Cw, Cm; };

// prospect_DB.f90:94-189 for table row i
__device__ void prospect_row(const double* __restrict__ tab, const Leaf7& p, int i, double& refl, double& tran)
{
    const double nr = tab[T_NR * NWP + i];
    const double k = (((((p.Cab * tab[T_CAB * NWP + i] + p.Car * tab[T_CAR * NWP + i])
                         + p.Anth * tab[T_ANTH * NWP + i]) + p.Cbrown * tab[T_BROWN * NWP + i])
                       + p.Cw * tab[T_CW * NWP + i]) + p.Cm * tab[T_CM * NWP + i]) / p.N;   // :94
    const double tau = plate_tau_dev(k);
    const double t12 = tab[T_TAV90 * NWP + i];
    const double talf = tab[T_TAV40 * NWP + i];
    const double ralf = 1.0 - talf;                      // :149
    const double r12 = 1.0 - t12;
    const double t21 = t12 / (nr * nr);
    const double r21 = 1.0 - t21;
    double denom = 1.0 - (r21 * r21) * (tau * tau);      // :154
    const double Ta = ((talf * tau) * t21) / denom;
    const double Ra = ralf + (r21 * tau) * Ta;
    const double t = ((t12 * tau) * t21) / denom;
    const double r = r12 + (r21 * tau) * t;
    const double D = sqrt(((((1.0 + r) + t) * ((1.0 + r) - t)) * ((1.0 - r) + t)) * ((1.0 - r) - t));   // :167
    const double rq = r * r, tq = t * t;
    const double a = (((1.0 + rq) - tq) + D) / (2.0 * r);
    const double b = (((1.0 - rq) + tq) + D) / (2.0 * t);
    const double bNm1 = pow(b, p.N - 1.0);               // :172
    const double bN2 = bNm1 * bNm1;
    const double a2 = a * a;
    denom = a2 * bN2 - 1.0;
    double Rsub = (a * (bN2 - 1.0)) / denom;
    double Tsub = (bNm1 * (a2 - 1.0)) / denom;
    if (r + t >= 1.0) {                                  // :181-184
        Tsub = t / (t + (1.0 - t) * (p.N - 1.0));
        Rsub = 1.0 - Tsub;
    }
    denom = 1.0 - Rsub * r;                              // :187
    tran = (Ta * Tsub) / denom;
    refl = Ra + (((Ta * Rsub) * t) / denom);
}

__device__ __forceinline__ double soil_sum(const double* __restrict__ eof, const double* w4, int idx)
{
    // the reference reads one past the tables at 2500 nm and multiplies by a zero fraction
    // (gortt.c:1311,1318): contribute 0 instead
    if (idx >= GORT_SOIL_NW) return 0.0;
    return w4[0] * eof[0 * GORT_SOIL_NW + idx] + w4[1] * eof[1 * GORT_SOIL_NW + idx]
         + w4[2] * eof[2 * GORT_SOIL_NW + idx] + w4[3] * eof[3 * GORT_SOIL_NW + idx];
}

__global__ void __launch_bounds__(128)
spectra_kernel(int n_sets, int n_wl, const double* __restrict__ leaf, const double* __restrict__ soil,
               double user_leaf, double user_soil, const double* __restrict__ wl,
               const double* __restrict__ tab, const double* __restrict__ eof,
               double* __restrict__ rleaf, double* __restrict__ tleaf, double* __restrict__ rsoil)
{
    long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long) n_sets * n_wl) return;
    const int m = (int) (e / n_wl), i = (int) (e - (long) m * n_wl);
    const double wv = wl[i];
    if (!(wv >= GORT_WL_MIN && wv <= GORT_WL_MAX)) {
        // the reference exits on an out-of-range wavelength (gortt.c:1299-1302, :1350-1353); the
        // host entry points reject it before launch, device callers get NaN instead of a wild read
        const double qnan = __longlong_as_double(0x7ff8000000000000LL);
        rleaf[e] = qnan; tleaf[e] = qnan; rsoil[e] = qnan;
        return;
    }

    // gortt_price_soil, gortt.c:1297-1324
    if (user_soil >= 0.0) {
        rsoil[e] = user_soil;
    } else {
        double w4[4] = { soil[0 * (size_t) n_sets + m], soil[1 * (size_t) n_sets + m],
                         soil[2 * (size_t) n_sets + m], soil[3 * (size_t) n_sets + m] };
        int upper = (int) (1. + (wv - 400) / 5.0);
        int lower = (int) ((wv - 400) / 5.0);
        double fraction = (double) (wv - 400.) / 5.0 - lower;
        double rs_lower = soil_sum(eof, w4, lower);
        double rs_upper = soil_sum(eof, w4, upper);
        rsoil[e] = rs_lower * (1 - fraction) + rs_upper * fraction;
    }

    // gortt_prospect_interface, gortt.c:1349-1371
    if (user_leaf >= 0.0) {
        rleaf[e] = user_leaf / 2.0;
        tleaf[e] = user_leaf / 2.0;
    } else {
        Leaf7 p = { leaf[0 * (size_t) n_sets + m], leaf[1 * (size_t) n_sets + m], leaf[2 * (size_t) n_sets + m],
                    leaf[3 * (size_t) n_sets + m], leaf[4 * (size_t) n_sets + m], leaf[5 * (size_t) n_sets + m],
                    leaf[6 * (size_t) n_sets + m] };
        int upper = (int) (1 + (wv - 400.0) / 1.0);
        int lower = (int) ((wv - 400.0) / 1.0);
        float fraction = (float) ((float) (wv - 400.0) / 1.0 - lower);            // float: gortt.c:1338,1364
        float omf = 1 - fraction;
        double rl, tl, ru = 0.0, tu = 0.0;
        prospect_row(tab, p, lower, rl, tl);
        // the upper row is evaluated even when the fraction is 0: y*0 is NaN for a NaN row (N > 1 and k > 85:
        // tau = 0, b = inf, Rsub = inf/inf), and the reference's interpolation propagates it.  At 2500 nm the
        // reference's upper row is one past the array and its fraction is 0: it contributes 0
        if (upper < NWP) prospect_row(tab, p, upper, ru, tu);
        rleaf[e] = rl * omf + ru * fraction;
        tleaf[e] = tl * omf + tu * fraction;
    }
}

__global__ void __launch_bounds__(128)
prospect_full_kernel(int n_sets, const double* __restrict__ leaf, const double* __restrict__ tab,
                     double* __restrict__ refl, double* __restrict__ tran)
{
    long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long) n_sets * NWP) return;
    const int m = (int) (e / NWP), i = (int) (e - (long) m * NWP);
    Leaf7 p = { leaf[0 * (size_t) n_sets + m], leaf[1 * (size_t) n_sets + m], leaf[2 * (size_t) n_sets + m],
                leaf[3 * (size_t) n_sets + m], leaf[4 * (size_t) n_sets + m], leaf[5 * (size_t) n_sets + m],
                leaf[6 * (size_t) n_sets + m] };
    double r, t;
    prospect_row(tab, p, i, r, t);
    refl[e] = r;
    tran[e] = t;
}

int launch_tav_tables(gort_ctx *ctx, cudaStream_t s, double *d_prospect)
{
    // widen the binary32 tables to FP64 on the host (a data conversion, not model arithmetic)
    static const uint32_t *src[7] = { gort_tab_refractive_f32, gort_tab_k_cab_f32, gort_tab_k_car_f32,
                                      gort_tab_k_anth_f32, gort_tab_k_brown_f32, gort_tab_k_cw_f32,
                                      gort_tab_k_cm_f32 };
    double *h = (double *) malloc(sizeof(double) * 7 * NWP);
    if (!h) return set_error(ctx, GORT_ERR_NOMEM, "out of host memory");
    for (int t = 0; t < 7; t++)
        for (int i = 0; i < NWP; i++) {
            float f;
            memcpy(&f, &src[t][i], sizeof f);
            h[t * NWP + i] = (double) f;
        }
    cudaError_t e = cudaMemcpyAsync(d_prospect, h, sizeof(double) * 7 * NWP, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    free(h);
    if (e != cudaSuccess) return check_cuda(ctx, e, "upload PROSPECT tables");
    tav_kernel<<<(NWP + 127) / 128, 128, 0, s>>>(d_prospect);
    ctx->launches++;
    return check_cuda(ctx, cudaGetLastError(), "tav_kernel launch");
}

// rsoil from a 1-nm soil table read from a file (gort_soil_table_read): the lookup the reference declares as
// gortt_get_rsoil_lut (include/gortt.h:296) and never defines.  Same index / fraction arithmetic as gortt_price_soil
// (gortt.c:1311-1321) with a 1-nm step; the row past 2500 nm is never read (its weight is zero).
__global__ void __launch_bounds__(128)
soil_table_kernel(int n_sets, int n_wl, const double* __restrict__ table, const double* __restrict__ wl,
                  double* __restrict__ rsoil)
{
    long e = (long) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long) n_sets * n_wl) return;
    const int i = (int) (e % n_wl);
    const double wv = wl[i];
    if (!(wv >= GORT_WL_MIN && wv <= GORT_WL_MAX)) { rsoil[e] = __longlong_as_double(0x7ff8000000000000LL); return; }
    int upper = (int) (1. + (wv - 400) / 1.0);
    int lower = (int) ((wv - 400) / 1.0);
    double fraction = (double) (wv - 400.) / 1.0 - lower;
    double rs_lower = table[lower];
    double rs_upper = upper < GORT_SOIL_TABLE_NW ? table[upper] : 0.0;
    rsoil[e] = rs_lower * (1 - fraction) + rs_upper * fraction;
}

int launch_soil_table(gort_ctx *ctx, cudaStream_t s, const double *table, int n_sets, int n_wl, const double *wl, double *rsoil)
{
    note_other_work(ctx);
    long total = (long) n_sets * n_wl;
    soil_table_kernel<<<(unsigned) ((total + 127) / 128), 128, 0, s>>>(n_sets, n_wl, table, wl, rsoil);
    ctx->launches++;
    return check_cuda(ctx, cudaGetLastError(), "soil_table_kernel launch");
}

int upload_soil_tables(gort_ctx *ctx, cudaStream_t s, double *d_soil)
{
    static const uint64_t *src[4] = { gort_tab_soil_eof1_f64, gort_tab_soil_eof2_f64,
                                      gort_tab_soil_eof3_f64, gort_tab_soil_eof4_f64 };
    for (int t = 0; t < 4; t++) {
        cudaError_t e = cudaMemcpyAsync(d_soil + (size_t) t * GORT_SOIL_NW, src[t], sizeof(double) * GORT_SOIL_NW,
                                        cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) return check_cuda(ctx, e, "upload soil tables");
    }
    return check_cuda(ctx, cudaStreamSynchronize(s), "upload soil tables");
}

int launch_spectra(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *leaf, const double *soil,
                   double user_leaf, double user_soil, int n_wl, const double *wl,
                   double *rleaf, double *tleaf, double *rsoil)
{
    note_other_work(ctx);
    if (n_sets <= 0 || n_wl <= 0) return set_error(ctx, GORT_ERR_INVALID, "gort_spectra: n_sets and n_wl must be positive");
    if (user_leaf < 0.0 && !leaf) return set_error(ctx, GORT_ERR_INVALID, "gort_spectra: leaf parameters missing");
    if (user_soil < 0.0 && !soil) return set_error(ctx, GORT_ERR_INVALID, "gort_spectra: soil weights missing");
    long total = (long) n_sets * n_wl;
    spectra_kernel<<<(unsigned) ((total + 127) / 128), 128, 0, s>>>(n_sets, n_wl, leaf, soil, user_leaf, user_soil, wl,
                                                                    ctx->d_prospect, ctx->d_soil, rleaf, tleaf, rsoil);
    ctx->launches++;
    return check_cuda(ctx, cudaGetLastError(), "gort_spectra launch");
}

int launch_prospect_full(gort_ctx *ctx, cudaStream_t s, int n_sets, const double *leaf, double *refl, double *tran)
{
    note_other_work(ctx);
    if (n_sets <= 0 || !leaf) return set_error(ctx, GORT_ERR_INVALID, "gort_prospect: bad arguments");
    long total = (long) n_sets * NWP;
    prospect_full_kernel<<<(unsigned) ((total + 127) / 128), 128, 0, s>>>(n_sets, leaf, ctx->d_prospect, refl, tran);
    ctx->launches++;
    return check_cuda(ctx, cudaGetLastError(), "gort_prospect launch");
}

}  // namespace gort
