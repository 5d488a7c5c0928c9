"""ctypes bindings for the CHECKERS (test infrastructure only).

  oracle()  -> oracle/libgort_oracle.so   our plain-C restatement
  ref()     -> oracle/_ref/libgortt_ref.so the unmodified reference compiled in the build container
               (None if it was not built / did not travel)

Both expose the same call signatures (oracle/gort_oracle.h, oracle/ref_harness.c) through the
`Checker` wrapper below, which takes and returns numpy arrays.
"""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
NTH = 91
LUT_LEN = 2 * NTH + 2

_dp = C.POINTER(C.c_double)


def _p(a):
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dp)


class Checker:
    def __init__(self, lib, prefix):
        self.lib = lib
        self.prefix = prefix
        f = lambda n: getattr(lib, prefix + n)
        self._lut = f("lut")
        self._lut.argtypes = [_dp, C.c_int, _dp]
        self._lut_i = f("lut_intermediates")
        self._lut_i.argtypes = [_dp] * 6
        self._brdf = f("brdf")
        self._brdf.argtypes = [_dp, _dp, _dp, C.c_int, _dp, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp]
        self._energy = f("energy")
        self._energy.argtypes = [_dp, _dp, _dp, C.c_int, _dp, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp]
        self._spectra = f("spectra")
        self._spectra.argtypes = [_dp, _dp, C.c_double, C.c_double, C.c_int, _dp, _dp, _dp, _dp]
        self._spectra.restype = C.c_int
        self._gauleg = f("gauleg")
        self._gauleg.argtypes = [C.c_int, _dp, _dp]
        self._repeat = f("brdf_repeat")
        self._repeat.argtypes = [_dp, _dp, C.c_int, _dp, C.c_int, _dp, _dp, _dp, C.c_int, _dp]
        self._repeat.restype = C.c_long

    @staticmethod
    def _st(st6):
        st = np.ascontiguousarray(st6, dtype=np.float64)
        assert st.shape == (6,)
        return st

    def lut(self, st6, method=0):
        out = np.empty(LUT_LEN)
        self._lut(_p(self._st(st6)), method, _p(out))
        return out

    def lut_intermediates(self, st6):
        v_g = np.empty((15, NTH)); p_n0 = np.empty((15, NTH)); der = np.empty(16)
        th = np.empty(NTH); hp = np.empty(15)
        self._lut_i(_p(self._st(st6)), _p(v_g), _p(p_n0), _p(der), _p(th), _p(hp))
        return dict(v_g=v_g, p_n0=p_n0, derived=der, theta_p=th, height_p=hp)

    @staticmethod
    def _opt(beta=None, fd=None):
        if beta is None and fd is None:
            return None
        return np.array([beta is not None, beta or 0.0, fd is not None, fd or 0.0], dtype=np.float64)

    def brdf(self, st6, lut, ang, rleaf, tleaf, rsoil, beta=None, fd=None, want_scomp=True):
        ang = np.ascontiguousarray(ang, dtype=np.float64).reshape(-1, 4)
        rleaf, tleaf, rsoil = (np.ascontiguousarray(a, dtype=np.float64) for a in (rleaf, tleaf, rsoil))
        ng, nw = ang.shape[0], rleaf.shape[0]
        rsurf = np.empty((ng, nw)); scomp = np.empty((ng, nw, 4)) if want_scomp else None
        kprop = np.empty((ng, 4))
        self._brdf(_p(self._st(st6)), _p(np.ascontiguousarray(lut)), _p(self._opt(beta, fd)), ng, _p(ang), nw,
                   _p(rleaf), _p(tleaf), _p(rsoil), _p(rsurf), _p(scomp), _p(kprop))
        return rsurf, scomp, kprop

    def energy(self, st6, lut, ang, rleaf, tleaf, rsoil, beta=None, fd=None):
        ang = np.ascontiguousarray(ang, dtype=np.float64).reshape(-1, 4)
        rleaf, tleaf, rsoil = (np.ascontiguousarray(a, dtype=np.float64) for a in (rleaf, tleaf, rsoil))
        ng, nw = ang.shape[0], rleaf.shape[0]
        alb = np.empty((ng, nw)); fv = np.empty((ng, nw)); fs = np.empty((ng, nw))
        self._energy(_p(self._st(st6)), _p(np.ascontiguousarray(lut)), _p(self._opt(beta, fd)), ng, _p(ang), nw,
                     _p(rleaf), _p(tleaf), _p(rsoil), _p(alb), _p(fv), _p(fs))
        return alb, fv, fs

    def spectra(self, leaf7, soil4, wl, user_leaf=-1.0, user_soil=-1.0):
        leaf7 = np.ascontiguousarray(leaf7, dtype=np.float64); soil4 = np.ascontiguousarray(soil4, dtype=np.float64)
        wl = np.ascontiguousarray(wl, dtype=np.float64)
        nw = wl.shape[0]
        rl = np.empty(nw); tl = np.empty(nw); rs = np.empty(nw)
        self._spectra(_p(leaf7), _p(soil4), user_leaf, user_soil, nw, _p(wl), _p(rl), _p(tl), _p(rs))
        return rl, tl, rs

    def lut_dead(self, st6):
        """vb[15], fb[15][91], t_open[15][15], dt_open[15][15], dk_open[15], k_open[15] (gortt_pn_kopen.c:925-1078)."""
        rc, out = self.lut_dead_rc(st6)
        assert rc == 0, "negative sphere volume: the reference exits on this structure"
        return out

    def lut_dead_rc(self, st6):
        """(rc, outputs of lut_dead): rc = 1 where the reference exits on a negative sphere volume (gortt_calc_vb);
        the outputs are then undefined."""
        fn = getattr(self.lib, self.prefix + "lut_dead")
        fn.argtypes = [_dp] * 7
        fn.restype = C.c_int
        out = dict(vb=np.empty(15), fb=np.empty((15, NTH)), t_open=np.empty((15, 15)), dt_open=np.empty((15, 15)),
                   dk_open=np.empty(15), k_open=np.empty(15))
        rc = fn(_p(self._st(st6)), *[_p(out[k]) for k in ("vb", "fb", "t_open", "dt_open", "dk_open", "k_open")])
        return rc, out

    def lut_bins(self, st6):
        """(restatement only) umax[91]: per zenith, the largest s/ds + 0.5 the full method's crown-count loop reaches,
        i.e. the largest histogram bin is int(umax[t]) (gortt_pn_kopen.c:457-527, :134-139)."""
        fn = getattr(self.lib, self.prefix + "lut_bins")
        fn.argtypes = [_dp, _dp]
        fn.restype = C.c_int
        out = np.empty(NTH)
        rc = fn(_p(self._st(st6)), _p(out))
        assert rc == 0
        return out

    def soil_table(self, path):
        """(restatement only) -> (rc, table[2101], where): the reference's soil-file interpolation loop."""
        fn = self.lib.gort_oracle_soil_table
        fn.argtypes = [C.c_char_p, _dp, _dp]
        tab = np.empty(2101); where = np.zeros(1)
        rc = fn(os.fsencode(str(path)), _p(tab), _p(where))
        return rc, tab, float(where[0])

    def soil_lookup(self, table, wl):
        fn = self.lib.gort_oracle_soil_lookup
        fn.argtypes = [_dp, C.c_int, _dp, _dp]
        wl = np.ascontiguousarray(wl, dtype=np.float64)
        out = np.empty(wl.shape[0])
        rc = fn(_p(np.ascontiguousarray(table, dtype=np.float64)), wl.shape[0], _p(wl), _p(out))
        assert rc == 0
        return out

    def gauleg(self, n=32):
        x = np.empty(n); w = np.empty(n)
        self._gauleg(n, _p(x), _p(w))
        return x, w

    def brdf_repeat(self, st6, lut, ang, rleaf, tleaf, rsoil, reps):
        ang = np.ascontiguousarray(ang, dtype=np.float64).reshape(-1, 4)
        ng, nw = ang.shape[0], rleaf.shape[0]
        return self._repeat(_p(self._st(st6)), _p(np.ascontiguousarray(lut)), ng, _p(ang), nw,
                            _p(np.ascontiguousarray(rleaf)), _p(np.ascontiguousarray(tleaf)),
                            _p(np.ascontiguousarray(rsoil)), reps, None)


_cache = {}


def build_checkers():
    """(Re)build the checkers with oracle/Makefile. Building the checker is not using it."""
    subprocess.run(["make", "-s", "-C", str(ROOT / "oracle")], check=True,
                   stdout=subprocess.DEVNULL)


def oracle():
    if "oracle" not in _cache:
        so = ROOT / "oracle" / "libgort_oracle.so"
        if not so.exists():
            build_checkers()
        _cache["oracle"] = Checker(C.CDLL(str(so)), "gort_oracle_")
    return _cache["oracle"]


class UlpOracle(Checker):
    """The oracle restatement linked against a 1-ULP-noisy libm (oracle/ulp_libm_shim.c)."""

    def __init__(self, lib):
        super().__init__(lib, "gort_oracle_")
        lib.gort_oracle_ulp_seed.argtypes = [C.c_uint64]

    def seed(self, s):
        self.lib.gort_oracle_ulp_seed(s)


def oracle_ulp():
    if "ulp" not in _cache:
        so = ROOT / "oracle" / "libgort_oracle_ulp.so"
        if not so.exists():
            build_checkers()
        _cache["ulp"] = UlpOracle(C.CDLL(str(so)))
    return _cache["ulp"]


def sensitivity(fn, ref_value, seeds=(1, 2, 3)):
    """Element-wise max |f_ulp(seed) - ref| over a few seeds: how far the reference algorithm itself
    moves under a 1-ULP libm.  `fn(checker)` must return an array (or tuple of arrays) like ref_value."""
    u = oracle_ulp()
    single = not isinstance(ref_value, tuple)
    refs = (ref_value,) if single else ref_value
    sens = [np.zeros_like(np.asarray(r, dtype=np.float64)) for r in refs]
    for sd in seeds:
        u.seed(sd)
        out = fn(u)
        outs = (out,) if single else out
        for k, (a, r) in enumerate(zip(outs, refs)):
            if r is None:
                continue
            d = np.abs(np.asarray(a) - np.asarray(r))
            d = np.where(np.isnan(d), np.inf, d)
            sens[k] = np.maximum(sens[k], d)
    return sens[0] if single else tuple(sens)


# ---- comparison with the oracle (BASELINE.json north_star / SURVEY.md 8d) ----------------------
#        |x - ref| <= 1e-9 * max(|ref|, 1e-12),  NaN positions must coincide.
RTOL = 1e-9
FLOOR = 1e-12
COND_FACTOR = 32.0


def rel_err(x, ref):
    x = np.asarray(x); ref = np.asarray(ref)
    assert x.shape == ref.shape, (x.shape, ref.shape)
    nx, nr = np.isnan(x), np.isnan(ref)
    assert np.array_equal(nx, nr), "NaN positions differ: %d vs %d" % (nx.sum(), nr.sum())
    ok = ~nr
    if not ok.any():
        return 0.0
    return float(np.max(np.abs(x[ok] - ref[ok]) / np.maximum(np.abs(ref[ok]), FLOOR)))


def assert_close(x, ref, what, rtol=RTOL):
    e = rel_err(x, ref)
    assert e <= rtol, "%s: max rel err %.3e > %.1e" % (what, e, rtol)
    return e


def assert_close_cond(x, ref, sens, what, rtol=RTOL):
    """Strict bound first.  An entry that misses it must be explained by the reference algorithm's own
    conditioning: |x - ref| <= COND_FACTOR * (how far the oracle itself moves under a 1-ULP libm,
    sensitivity below).  Returns (strict worst rel err, number of entries excused)."""
    x = np.asarray(x); ref = np.asarray(ref)
    nx, nr = np.isnan(x), np.isnan(ref)
    assert np.array_equal(nx, nr), "%s: NaN positions differ" % what
    ok = ~nr
    err = np.abs(x[ok] - ref[ok])
    strict = err <= rtol * np.maximum(np.abs(ref[ok]), FLOOR)
    excused = ~strict & (err <= COND_FACTOR * sens[ok])
    bad = ~strict & ~excused
    rel = err / np.maximum(np.abs(ref[ok]), FLOOR)
    assert not bad.any(), "%s: %d entries miss 1e-9 and are not explained by conditioning; worst rel %.3e (sens %.3e, err %.3e)" % (
        what, bad.sum(), rel[bad].max(), sens[ok][bad][rel[bad].argmax()], err[bad][rel[bad].argmax()])
    return (float(rel.max()) if rel.size else 0.0), int(excused.sum())


DEAD_KEYS = ("vb", "fb", "t_open", "dt_open", "dk_open", "k_open")


def check_set(got, st6, oracle, what):
    """One set's gort_lut_intermediates outputs against the oracle's lut_dead.  fb = (1 - exp(-lv' vb)) / (1 - p_n0) is
    rounding noise wherever p_n0 rounds to 1 (the reference divides by DBL_MIN * 2 there, gortt_pn_kopen.c:990) and
    wherever vb is itself a cancelled ~1e-16 (a sphere centred on the lowest layer touches the h1 plane): those entries
    are compared for finiteness only.  Everything else: 1e-9, conditioning-aware like the LUT tests."""
    import parity_audit as pa                      # imports this module: deferred
    KEYS = DEAD_KEYS
    want = oracle.lut_dead(st6)
    lut = oracle.lut_intermediates(st6)
    sens = None
    worst = {}
    for k in KEYS:
        x, r = got[k], want[k]
        mask = np.ones(r.shape, dtype=bool)
        if k == "fb":
            mask = (1.0 - lut["p_n0"] >= 1e-12) & (want["vb"][:, None] > 1e-9)      # see the docstring
            assert np.isfinite(x).all()
        if k == "vb":
            mask = r > 1e-9
            assert np.all(np.abs(x[~mask] - r[~mask]) < 1e-12)
        s = pa.compare(x[mask], r[mask])
        if s["n_beyond_tol"]:
            if sens is None:
                sens = dict(zip(KEYS, sensitivity(lambda c: tuple(c.lut_dead(st6)[q] for q in KEYS), tuple(want[q] for q in KEYS))))
            s = pa.compare(x[mask], r[mask], sens[k][mask])
        assert pa.passed(s), "%s %s: %r" % (what, k, s)
        worst[k] = s["max_rel_err"]
    return worst


def ref():
    if "ref" not in _cache:
        so = ROOT / "oracle" / "_ref" / "libgortt_ref.so"
        if not so.exists() and os.path.exists("/root/reference/gortt.c"):
            build_checkers()
        _cache["ref"] = Checker(C.CDLL(str(so)), "ref_") if so.exists() else None
    return _cache["ref"]


def ref_makefile_flags():
    """the unmodified reference built with its own makefile's CFLAGS (-g, no optimisation): for timing only"""
    if "ref_g" not in _cache:
        so = ROOT / "oracle" / "_ref" / "libgortt_ref_g.so"
        if not so.exists() and os.path.exists("/root/reference/gortt.c"):
            build_checkers()
        _cache["ref_g"] = Checker(C.CDLL(str(so)), "ref_") if so.exists() else None
    return _cache["ref_g"]


REF_BIN = ROOT / "oracle" / "_ref" / "gortt_ref"


# ---- structure helpers shared by tests -------------------------------------------------------
def structure_from_cli(lambda_=0.405, r=0.76, b=None, h1=3.0, h2=8.5, favd=0.858,
                       hb=None, br=None, pcc=None, lai=None):
    """Mirror of the reference CLI's parameter derivation (gortt.c:67-72, :1014, :1117-1131),
    including the float-typed -HB/-BR/-PCC/-LAI values."""
    if b is None:
        b = 3.55263 * r
    if hb is not None or br is not None or pcc is not None:
        hb = np.float32(2.0 if hb is None else hb); br = np.float32(1.0 if br is None else br)
        pcc = np.float32(0.5 if pcc is None else pcc)
        r = 10.0
        b = float(br) * r
        h1 = b * 2.0
        h2 = float(hb) * b + h1
        lambda_ = float(pcc) / (r * r * np.pi)
    if lai is not None:
        lai = float(np.float32(lai))
        favd = lai * 3.0 / (lambda_ * r * r * np.pi * b * 4.0)
    return np.array([lambda_, r, b, h1, h2, favd], dtype=np.float64)
