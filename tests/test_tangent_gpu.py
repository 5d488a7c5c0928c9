"""GPU tests of the exact favd / LAI tangent (gort_lut_tangent_batch_dev, gort_brdf_tangent_batch_dev,
gort_lai_tangent_batch).

Reference: the CPU checker's chain (LUT -> spectra -> BRDF) differenced centrally in favd at relative steps h = 1e-3, h/2
and h/4 and Richardson-extrapolated, R(h) = (4 D(h/2) - D(h)) / 3.  Each member is compared with the reference's own
error bar: max|tangent - R(h)| <= max(1e-9 max|R(h)|, 10 max|R(h) - R(h/2)|).  The bar matters where the reference
itself converges slowly (a Q08 epgap that is a near-cancelling difference of two exponentials)."""
import ctypes as C

import numpy as np
import pytest
import torch

import gort_b200
import lut_catalogue as lc
from gort_b200 import workloads as wk

pytestmark = pytest.mark.gpu
FULL, Q08 = gort_b200.LUT_FULL, gort_b200.LUT_Q08
H = 1e-3


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda:0"))


def richardson(f, x0):
    """(R(h), |R(h) - R(h/2)|) of f at x0 for the relative step H"""
    def D(h):
        return (f(x0 * (1.0 + h)) - f(x0 * (1.0 - h))) / (2.0 * h * x0)
    d1, d2, d4 = D(H), D(H / 2), D(H / 4)
    r1, r2 = (4.0 * d2 - d1) / 3.0, (4.0 * d4 - d2) / 3.0
    return r1, np.abs(r1 - r2)


def assert_within_bar(got, ref, bar, what):
    err = np.max(np.abs(got - ref))
    bound = max(1e-9 * np.max(np.abs(ref)), 10.0 * np.max(bar))
    assert err <= bound, "%s: |tangent - R| = %.3e above %.3e (max|R| %.3e)" % (what, err, bound, np.max(np.abs(ref)))
    return err / bound


def lai_factor(st):
    """d favd / d LAI at fixed crown geometry (gortt.c:1129)"""
    return 3.0 / (st[0] * st[1] * st[1] * np.pi * st[2] * 4.0)


# ---- 1. LUT tangent ----------------------------------------------------------------------------------------------------
def lut_sets(style):
    if style == "c3":
        return wk.random_structures(np.random.Generator(np.random.PCG64(41)), 10)
    if style == "c4b":
        return wk.c4_enkf(n_members=10, seed=42)["structure"]
    if style == "c5":             # favd fastest: two sub-groups of 8 members sharing shape and stem density
        return wk.c5_lut_grid(n=(1, 2, 1, 1, 1, 8))["structure"]
    if style == "beyond_single":
        return lc.beyond_table_singles()[:, :8]
    if style == "beyond_sub":
        return lc.beyond_table_subgroups()[:, :13]
    raise ValueError(style)


@pytest.mark.parametrize("method", [FULL, Q08])
@pytest.mark.parametrize("style", ["c3", "c4b", "c5", "beyond_single", "beyond_sub"])
def test_lut_tangent_against_oracle(gort, oracle, method, style):
    st = lut_sets(style)
    M = st.shape[1]
    subs = lc.sub_groups(lc.plan(st)[1])
    if style in ("c5", "beyond_sub"):
        assert max(n for _, n in subs) == 8                    # lut_crown_kernel<8, true>
    if style in ("c3", "beyond_single"):
        assert all(n == 1 for _, n in subs)                    # lut_crown_kernel<1, true>
    d_st = dev(st)
    lut = torch.full((M, gort_b200.LUT_STRIDE), np.nan, dtype=torch.float64, device="cuda:0")
    dlut = torch.full_like(lut, np.nan)
    torch.cuda.synchronize()
    gort.lut_tangent_dev(d_st, lut, dlut, method=method)
    gort.synchronize()
    lut, dlut = lut.cpu().numpy(), dlut.cpu().numpy()
    assert np.array_equal(lut, gort.lut(st, method), equal_nan=True)
    NTH = gort_b200.NTH
    assert np.all(dlut[:, :NTH] == 0.0) and np.all(dlut[:, 2 * NTH] == 0.0)
    worst = 0.0
    for m in range(M):
        def rec(favd, m=m):
            s = st[:, m].copy()
            s[5] = favd
            return oracle.lut(s, method)
        ref, bar = richardson(rec, st[5, m])
        worst = max(worst, assert_within_bar(dlut[m], ref, bar, "%s member %d" % (style, m)))
    print("%s method %d: worst error / bound %.3f" % (style, method, worst))


# ---- 2. ensemble entry point against the oracle ------------------------------------------------------------------------
_ref_cache = {}


def oracle_tangent(oracle, w, method):
    """per member: (R, bar) of d rsurf / d favd through the checker's chain, or None where rsurf is not finite"""
    key = (id(w), method)
    if key not in _ref_cache:
        st, ang, wl = w["structure"], w["angles"], w["wavelength"]
        out = []
        for m in range(st.shape[1]):
            a = np.ascontiguousarray(ang[:, m, :].T)
            rl, tl, rs = oracle.spectra(w["leaf"][:, m], w["soil"][:, m], wl)

            def chain(favd, m=m, a=a, rl=rl, tl=tl, rs=rs):
                s = st[:, m].copy()
                s[5] = favd
                return oracle.brdf(s, oracle.lut(s, method), a, rl, tl, rs, want_scomp=False)[0]
            out.append(richardson(chain, st[5, m]) if np.isfinite(chain(st[5, m])).all() else None)
        _ref_cache[key] = out
    return _ref_cache[key]


W24 = wk.c4_enkf(n_members=24, seed=31)


@pytest.mark.parametrize("method", [FULL, Q08])
@pytest.mark.parametrize("param", [gort_b200.JAC_FAVD, gort_b200.JAC_LAI])
def test_lai_tangent_against_oracle(gort, oracle, method, param):
    w = W24
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    jac, rsurf = gort.lai_tangent(st, w["leaf"], w["soil"], wl, ang, param=param, method=method, want_rsurf=True)
    assert np.array_equal(rsurf, gort.forward(st, w["leaf"], w["soil"], wl, ang, method=method), equal_nan=True)
    refs = oracle_tangent(oracle, w, method)
    worst, n = 0.0, 0
    for m, r in enumerate(refs):
        if r is None:
            continue
        f = lai_factor(st[:, m]) if param == gort_b200.JAC_LAI else 1.0
        worst = max(worst, assert_within_bar(jac[m], r[0] * f, r[1] * f, "member %d" % m))
        n += 1
    assert n >= 20
    print("method %d param %d: worst error / bound %.3f over %d members" % (method, param, worst, n))


@pytest.mark.parametrize("method", [FULL, Q08])
def test_lai_is_favd_times_map(gort, method):
    w = W24
    st = w["structure"]
    args = (st, w["leaf"], w["soil"], w["wavelength"], w["angles"])
    jf = gort.lai_tangent(*args, param=gort_b200.JAC_FAVD, method=method)
    jl = gort.lai_tangent(*args, param=gort_b200.JAC_LAI, method=method)
    lai = st[5] * (st[0] * st[1] ** 2 * np.pi * st[2] * 4.0) / 3.0
    want = jf * (st[5] / lai)[:, None, None]
    ok = np.isfinite(want)
    assert np.array_equal(ok, np.isfinite(jl))
    assert np.max(np.abs(jl[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1e-300)) <= 1e-12


# ---- 3. against the existing central difference ------------------------------------------------------------------------
def grazing(w, n=6):
    """w with the first n members' last two geometries at grazing sun / view zeniths"""
    w = {k: v.copy() for k, v in w.items()}
    w["angles"][0, :n, -1] = 89.999
    w["angles"][2, :n, -2] = 89.999
    w["angles"][0, :n, -2] = 90.0
    return w


@pytest.mark.parametrize("method", [FULL, Q08])
def test_tangent_against_central_difference(gort, oracle, method):
    """gort.jacobian at h = 1e-4 agrees with the tangent to 1e-7 of the member's largest entry.  A member where it does
    not is one where the difference quotient's own truncation error is larger (Q08's near-cancelling epgap): there the
    tangent must match the checker's extrapolated reference and the difference quotient must be the farther of the two."""
    w = grazing(wk.c4_enkf(n_members=300, seed=32))
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    for param in (gort_b200.JAC_LAI, gort_b200.JAC_FAVD):
        cd = gort.jacobian(st, w["leaf"], w["soil"], wl, ang, param=param, rel_step=1e-4, method=method)
        tg = gort.lai_tangent(st, w["leaf"], w["soil"], wl, ang, param=param, method=method)
        assert np.array_equal(np.isfinite(cd), np.isfinite(tg))
        ok = np.isfinite(cd).all(axis=(1, 2))
        assert ok.mean() > 0.95
        scale = np.max(np.abs(cd[ok]), axis=(1, 2), keepdims=True)
        err = np.max(np.abs(cd[ok] - tg[ok]) / scale, axis=(1, 2))
        far = np.nonzero(ok)[0][err > 1e-7]
        print("method %d param %d: max |CD - tangent| / max|J| = %.3e, members above 1e-7: %s" % (method, param, err.max(), far))
        assert far.size <= 3
        for m in far:
            a = np.ascontiguousarray(ang[:, m, :].T)
            rl, tl, rs = oracle.spectra(w["leaf"][:, m], w["soil"][:, m], wl)

            def chain(favd, m=m, a=a, rl=rl, tl=tl, rs=rs):
                s = st[:, m].copy()
                s[5] = favd
                return oracle.brdf(s, oracle.lut(s, method), a, rl, tl, rs, want_scomp=False)[0]
            ref, bar = richardson(chain, st[5, m])
            f = lai_factor(st[:, m]) if param == gort_b200.JAC_LAI else 1.0
            assert_within_bar(tg[m], ref * f, bar * f, "member %d" % m)
            assert np.max(np.abs(cd[m] - ref * f)) > np.max(np.abs(tg[m] - ref * f))


# ---- 4. dispatch -------------------------------------------------------------------------------------------------------
def c2_lines(n_lines=48, step=1):
    w = wk.c2_hemisphere(wl_step=step)
    idx = (np.arange(n_lines) * 211) % w["angles"].shape[1]
    w["angles"] = np.ascontiguousarray(w["angles"][:, idx])
    return w


def dev_tangent(gort, st, lut, dlut, ang, rl, tl, rs, **kw):
    M, G, W = st.shape[1], ang.shape[-1], rl.shape[-1]
    out = torch.full((M, G, W), np.nan, dtype=torch.float64, device="cuda:0")
    torch.cuda.synchronize()
    gort.brdf_tangent_dev(dev(st), dev(lut), dev(dlut), dev(ang), dev(rl), dev(tl), dev(rs), out, **kw)
    gort.synchronize()
    return out.cpu().numpy()


def dev_lut_tangent(gort, st, method):
    M = st.shape[1]
    lut = torch.empty((M, gort_b200.LUT_STRIDE), dtype=torch.float64, device="cuda:0")
    dlut = torch.empty_like(lut)
    gort.lut_tangent_dev(dev(st), lut, dlut, method=method)
    gort.synchronize()
    return lut.cpu().numpy(), dlut.cpu().numpy()


@pytest.mark.parametrize("grid", ["w7", "w97", "w2101"])
def test_dispatch_layouts_and_dev_pair(gort, grid):
    """shared / per-set angles and spectra give the same bits, and the _dev pair gives the host entry point's bits"""
    if grid == "w2101":
        w = c2_lines()
        st = np.repeat(w["structure"], 3, axis=1) * np.array([1.0, 1, 1, 1, 1, 1.0])[:, None]
        st[5] *= np.array([1.0, 0.8, 1.3])
        w["leaf"] = np.repeat(w["leaf"], 3, axis=1)
        w["soil"] = np.repeat(w["soil"], 3, axis=1)
    else:
        w = wk.c4_enkf(n_members=40, seed=33)
        st = w["structure"]
        if grid == "w97":
            w["wavelength"] = np.arange(400.0, 2320.0 + 0.5, 20.0)
    M, wl = st.shape[1], w["wavelength"]
    ang = w["angles"] if w["angles"].ndim == 3 else np.repeat(w["angles"][:, None, :], M, axis=1)
    G = ang.shape[-1]
    host = gort.lai_tangent(st, w["leaf"], w["soil"], wl, ang, param=gort_b200.JAC_FAVD)
    lut, dlut = dev_lut_tangent(gort, st, FULL)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], wl)
    got = dev_tangent(gort, st, lut, dlut, ang, rl, tl, rs)
    assert np.array_equal(got, host, equal_nan=True)
    # shared angles (every member the same lines) and shared spectra
    sh_ang = np.ascontiguousarray(ang[:, 0, :])
    per = dev_tangent(gort, st, lut, dlut, np.ascontiguousarray(np.repeat(sh_ang[:, None, :], M, axis=1)),
                      np.repeat(rl[:1], M, axis=0), np.repeat(tl[:1], M, axis=0), np.repeat(rs[:1], M, axis=0))
    shared = dev_tangent(gort, st, lut, dlut, sh_ang, rl[0], tl[0], rs[0])
    assert np.array_equal(per, shared, equal_nan=True)
    assert np.isfinite(shared).mean() > 0.9 and G * wl.size > 0
    # against the central difference of the same layout
    cd = gort.jacobian(st, w["leaf"], w["soil"], wl, ang, param=gort_b200.JAC_FAVD, rel_step=1e-4)
    ok = np.isfinite(cd).all(axis=(1, 2))
    scale = np.max(np.abs(cd[ok]), axis=(1, 2), keepdims=True)
    assert np.max(np.abs(cd[ok] - host[ok]) / scale) <= 1e-7


@pytest.mark.parametrize("opts", [dict(beta=0.4), dict(fd=0.3), dict(beta=0.0, fd=1.0)])
def test_options(gort, opts):
    w = wk.c4_enkf(n_members=60, seed=34)
    args = (w["structure"], w["leaf"], w["soil"], w["wavelength"], w["angles"])
    tg, rsurf = gort.lai_tangent(*args, want_rsurf=True, **opts)
    assert np.array_equal(rsurf, gort.forward(*args, **opts), equal_nan=True)
    cd = gort.jacobian(*args, rel_step=1e-4, **opts)
    ok = np.isfinite(cd).all(axis=(1, 2))
    assert ok.mean() > 0.95
    scale = np.max(np.abs(cd[ok]), axis=(1, 2), keepdims=True)
    assert np.max(np.abs(cd[ok] - tg[ok]) / scale) <= 1e-7


def test_member_bits_do_not_depend_on_the_batch(gort):
    """2500 members run in three chunks; a member alone, in a slice, or at a chunk boundary gets the same bits"""
    w = wk.c4_enkf(n_members=2500, seed=35)
    st, ang = w["structure"], w["angles"]
    args = (w["leaf"], w["soil"], w["wavelength"])
    full, rsurf = gort.lai_tangent(st, *args, ang, want_rsurf=True)
    assert np.array_equal(rsurf, gort.forward(st, *args, ang), equal_nan=True)
    for lo, hi in ((0, 1), (1020, 1030), (1023, 1025), (2047, 2049), (2400, 2500)):
        part = gort.lai_tangent(st[:, lo:hi], w["leaf"][:, lo:hi], w["soil"][:, lo:hi], w["wavelength"], ang[:, lo:hi])
        assert np.array_equal(part, full[lo:hi], equal_nan=True), (lo, hi)


def test_one_slot_walk_over_contiguous_hemisphere(gort, oracle):
    """The whole C2 hemisphere (11 664 lines in runs of 36 that share a sun) for three forests of different favd at
    W = 421, in one call.  With W > 128 a CTA of rsurf_tangent_kernel has one line slot: its threads walk a range of
    consecutive lines (tens of them on a B200, across several 32-line record tiles and, for some CTAs, across a set
    boundary), keep their leaf terms while the set stays and rebuild their sun terms only where the record flags a new
    sun.  The result must have the bits of the same lines run 400 at a time (then every CTA holds one line and rebuilds
    everything), match the central difference to 1e-7 of each forest's largest entry, and match the checker's
    extrapolated reference on sampled lines."""
    w = wk.c2_hemisphere(wl_step=5, sets=3)
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    M, G, W = st.shape[1], ang.shape[1], wl.size
    assert W > 128 and len(set(st[5])) == M == 3
    assert np.mean(np.abs(np.diff(ang[2])) == 0) > 0.9          # most consecutive lines share the sun
    lut, dlut = dev_lut_tangent(gort, st, FULL)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], wl)
    full = dev_tangent(gort, st, lut, dlut, ang, rl, tl, rs)
    host = gort.lai_tangent(st, w["leaf"], w["soil"], wl, ang, param=gort_b200.JAC_FAVD)
    assert np.array_equal(full, host, equal_nan=True)
    assert np.isfinite(full).all()
    for m in range(M):
        for g0 in range(0, G, 400):
            a = np.ascontiguousarray(ang[:, g0:g0 + 400])
            part = dev_tangent(gort, st[:, m:m + 1], lut[m:m + 1], dlut[m:m + 1], a, rl[m:m + 1], tl[m:m + 1], rs[m:m + 1])
            assert np.array_equal(part[0], full[m, g0:g0 + 400]), (m, g0)
    cd = gort.jacobian(st, w["leaf"], w["soil"], wl, ang, param=gort_b200.JAC_FAVD, rel_step=1e-4)
    for m in range(M):
        err = np.max(np.abs(cd[m] - full[m])) / np.max(np.abs(cd[m]))
        print("forest %d: max |CD - tangent| / max|J| = %.3e" % (m, err))
        assert err <= 1e-7
    idx = np.concatenate([np.arange(35, 11664, 997), [0, 1, 36 * 18 + 1]])   # ends and starts of sun runs
    for m in range(M):
        a = np.ascontiguousarray(ang[:, idx].T)

        def chain(favd, m=m, a=a):
            s = st[:, m].copy()
            s[5] = favd
            return oracle.brdf(s, oracle.lut(s, FULL), a, rl[m], tl[m], rs[m], want_scomp=False)[0]
        ref, bar = richardson(chain, st[5, m])
        assert_within_bar(full[m, idx], ref, bar, "forest %d" % m)


# ---- 5. contracts ------------------------------------------------------------------------------------------------------
def test_refusals_enqueue_nothing(gort):
    w = wk.c4_enkf(n_members=8, seed=36)
    st, ang = w["structure"], w["angles"]
    args = (st, w["leaf"], w["soil"], w["wavelength"], ang)
    good = gort.lai_tangent(*args)
    for bad in (gort_b200.JAC_LAMBDA, gort_b200.JAC_R, 9, -1):
        n0 = gort.launch_count()
        with pytest.raises(gort_b200.GortError) as e:
            gort.lai_tangent(*args, param=bad)
        assert e.value.code == 1 and gort.launch_count() == n0
    lut, dlut = dev_lut_tangent(gort, st, FULL)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], w["wavelength"])
    M, G, W = st.shape[1], ang.shape[-1], rl.shape[-1]
    out = torch.full((M, G, 16), np.nan, dtype=torch.float64, device="cuda:0")
    ins = [dev(a) for a in (st, lut, dlut, ang, rl, tl, rs)]
    torch.cuda.synchronize()
    sh = gort._shape(M, G, W, True, True, out_pitch=16)
    n0 = gort.launch_count()
    rc = gort._lib.gort_brdf_tangent_batch_dev(gort._h, None, C.byref(sh), *[t.data_ptr() for t in ins], out.data_ptr())
    assert rc == 1 and gort.launch_count() == n0
    gort.synchronize()
    assert torch.isnan(out).all()
    assert np.array_equal(gort.lai_tangent(*args), good, equal_nan=True)


_streams = []                     # kept alive for the context (include/gort_b200.h)


def test_tangent_after_overlapped_brdf_calls():
    """overlap-mode brdf_dev calls on one stream, then a tangent call on another: the same bits as with overlap off"""
    ctx = gort_b200.Gort(0)
    try:
        w = c2_lines(n_lines=400, step=5)
        st = w["structure"]
        lut, dlut = dev_lut_tangent(ctx, st, FULL)
        rl, tl, rs = ctx.spectra(w["leaf"], w["soil"], w["wavelength"])
        ins = [dev(a) for a in (st, lut, w["angles"], rl, tl, rs)]
        d_dlut = dev(dlut)
        G, W = w["angles"].shape[1], rl.shape[1]
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        _streams.extend([s1, s2])

        def run(overlap):
            ctx.set_overlap(overlap)
            X = torch.full((1, G, W), np.nan, dtype=torch.float64, device="cuda:0")
            T = torch.full((1, G, W), np.nan, dtype=torch.float64, device="cuda:0")
            torch.cuda.synchronize()
            for _ in range(3):
                ctx.brdf_dev(*ins, X, stream=s1.cuda_stream)
            ctx.brdf_tangent_dev(ins[0], ins[1], d_dlut, *ins[2:], T, stream=s2.cuda_stream)
            ctx.brdf_dev(*ins, X, stream=s1.cuda_stream)
            ctx.synchronize()
            return X.cpu().numpy(), T.cpu().numpy()

        plain = run(False)
        over = run(True)
        for p, q in zip(plain, over):
            assert np.array_equal(p, q, equal_nan=True)
        assert np.isfinite(plain[1]).mean() > 0.9
    finally:
        ctx.close()
