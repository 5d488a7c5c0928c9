"""Sensor-band entry points (gort_brdf_band_batch[_dev], gort_energy_band_batch[_dev], gort_forward_band_batch) against
the definition in include/gort_b200.h applied to the per-wavelength entry points on the same inputs:
|band - band_mean(x)| <= 1e-12 max_{i in S_b} |x_i|, NaN positions equal (tests/band_ref.py).

The inputs: random crowns and PROSPECT leaves, lines in runs of two that share a sun, two grids -- 40 columns (the
per-wavelength reference is rsurf_flat_kernel) and 211 columns (rsurf_wide_kernel) -- and five bands on each: a boxcar
touching the first column, a Gaussian, an overlapping boxcar with a sloped response, a single column, and a comb whose
zero-weight columns lie inside the band and which touches the last column."""
import ctypes as C

import numpy as np
import pytest
import torch

import gort_b200
from gort_b200 import workloads as wk
from band_ref import MODIS_EDGES, band_mean, close_to_band_mean

pytestmark = pytest.mark.gpu

M, G = 5, 6
SENT = -7.0
GRIDS = {"w40": np.arange(600.0, 1000.0, 10.0), "w211": np.arange(400.0, 2500.5, 10.0)}
GRID_1NM = np.arange(400.0, 2500.5, 1.0)


@pytest.fixture(scope="module")
def g():
    ctx = gort_b200.Gort(0)
    yield ctx
    ctx.close()


def bands_for(grid):
    W, lo, hi = len(grid), grid[0], grid[-1]
    span = hi - lo
    rows = [gort_b200.band_weights(grid, [lo, lo + 0.2 * span], [1.0, 1.0])]
    x = np.linspace(lo + 0.3 * span, lo + 0.6 * span, 41)
    rows.append(gort_b200.band_weights(grid, x, np.exp(-0.5 * ((x - x.mean()) / ((x[-1] - x[0]) / 6.0)) ** 2)))
    rows.append(gort_b200.band_weights(grid, [lo + 0.5 * span, lo + 0.7 * span], [2.0, 0.5]))
    single = np.zeros((1, W))
    single[0, W // 3] = 0.7
    comb = np.zeros((1, W))
    comb[0, W - 1:W - 1 - 2 * (W // 8):-2] = 1.3
    rows += [single, comb]
    w = np.vstack(rows)
    assert w[0, 0] > 0 and w[4, W - 1] > 0 and w[4, W - 2] == 0 and np.count_nonzero(w[3]) == 1
    return w


def make(g, seed, grid, per_set_geom, per_set_spectra, n_sets=M, n_geom=G):
    rng = np.random.Generator(np.random.PCG64(seed))
    st = wk.random_structures(rng, n_sets)
    leaf = wk.random_leaves(rng, n_sets)
    soil = np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), n_sets, axis=1)
    lead = (n_sets,) if per_set_geom else ()
    vza = rng.uniform(0.0, 70.0, lead + (n_geom,))
    vaa = rng.uniform(0.0, 360.0, lead + (n_geom,))
    sza = np.repeat(rng.uniform(15.0, 70.0, lead + ((n_geom + 1) // 2,)), 2, axis=-1)[..., :n_geom]
    saa = rng.uniform(0.0, 360.0, lead + (n_geom,))
    ang = np.stack([vza, vaa, sza, saa])
    lut = g.lut(st)
    rl, tl, rs = g.spectra(leaf, soil, grid)
    if not per_set_spectra:
        rl, tl, rs = rl[0], tl[0], rs[0]
    return dict(st=st, leaf=leaf, soil=soil, ang=ang, lut=lut, sp=(rl, tl, rs), grid=grid)


def assert_band(got, x, w):
    ok, worst = close_to_band_mean(got, x, w)
    assert ok, "worst |error| / (1e-12 max|x|) = %g" % worst


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda:0"))


LAYOUTS = [(gps, sps) for gps in (False, True) for sps in (False, True)]


# ---- BRDF ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("gps,sps", LAYOUTS, ids=["shared", "spectra_per_set", "angles_per_set", "both_per_set"])
def test_brdf_band_is_the_mean_of_brdf(g, grid, gps, sps):
    x = make(g, 11, GRIDS[grid], gps, sps)
    w = bands_for(x["grid"])
    rsurf = g.brdf(x["st"], x["lut"], x["ang"], *x["sp"])
    assert np.isfinite(rsurf).all()
    rb = g.brdf_band(x["st"], x["lut"], x["ang"], *x["sp"], w)
    assert rb.shape == (M, G, w.shape[0])
    assert_band(rb, rsurf, w)


@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("opt", [dict(beta=0.35), dict(fd=0.3), dict(beta=1.2, fd=0.85)], ids=["beta", "fd", "beta_fd"])
def test_brdf_band_options(g, grid, opt):
    x = make(g, 12, GRIDS[grid], True, True)
    w = bands_for(x["grid"])
    rsurf = g.brdf(x["st"], x["lut"], x["ang"], *x["sp"], **opt)
    assert_band(g.brdf_band(x["st"], x["lut"], x["ang"], *x["sp"], w, **opt), rsurf, w)


@pytest.mark.parametrize("grid", sorted(GRIDS))
def test_nan_spectra_outside_the_support_do_not_propagate(g, grid):
    x = make(g, 13, GRIDS[grid], True, True)
    w = bands_for(x["grid"])
    W = w.shape[1]
    rl, tl, rs = (a.copy() for a in x["sp"])
    rl[:, W - 2] = np.nan         # a zero-weight column inside the comb band, outside every other band
    assert not (w[:, W - 2] > 0).any()
    rs[0, 1] = np.nan             # inside band 0, set 0 only
    rsurf = g.brdf(x["st"], x["lut"], x["ang"], rl, tl, rs)
    rb = g.brdf_band(x["st"], x["lut"], x["ang"], rl, tl, rs, w)
    assert_band(rb, rsurf, w)
    assert np.isnan(rb[0, :, 0]).all() and np.isfinite(rb[1:, :, 0]).all() and np.isfinite(rb[:, :, 1:]).all()


@pytest.mark.parametrize("grid", sorted(GRIDS))
def test_grazing_lines_give_nan_bands(g, grid):
    x = make(g, 14, GRIDS[grid], True, True)
    ang = x["ang"].copy()
    ang[0, 1, 2] = 90.0            # view at the horizon
    ang[2, 3, 4] = 90.0            # sun at the horizon
    ang[2, 3, 5] = 90.0
    w = bands_for(x["grid"])
    rsurf = g.brdf(x["st"], x["lut"], ang, *x["sp"])
    rb = g.brdf_band(x["st"], x["lut"], ang, *x["sp"], w)
    assert np.isnan(rsurf).any()
    assert_band(rb, rsurf, w)
    assert np.isnan(rb[3, 4]).all() and np.isnan(rb[1, 2]).all()


def test_sixty_four_bands_and_sets_split_over_ctas(g):
    """GORT_MAX_BANDS random bands (more (run, band) pairs than a CTA has threads) and 20 lines per set (a set's lines
    over two CTAs), every line its own sun"""
    x = make(g, 15, GRIDS["w211"], True, True, n_geom=20)
    x["ang"][2] = np.random.Generator(np.random.PCG64(16)).uniform(15.0, 70.0, (M, 20))
    rng = np.random.Generator(np.random.PCG64(17))
    W = x["grid"].size
    w = np.zeros((gort_b200.MAX_BANDS, W))
    for b in range(gort_b200.MAX_BANDS):
        lo = int(rng.integers(0, W - 1))
        hi = int(rng.integers(lo, min(W, lo + 40)))
        w[b, lo:hi + 1] = rng.uniform(0.0, 1.0, hi + 1 - lo)
        w[b, lo] = 0.5
    rsurf = g.brdf(x["st"], x["lut"], x["ang"], *x["sp"])
    assert_band(g.brdf_band(x["st"], x["lut"], x["ang"], *x["sp"], w), rsurf, w)
    ref = g.energy(x["st"], x["lut"], x["ang"], *x["sp"])
    for a, b in zip(g.energy_band(x["st"], x["lut"], x["ang"], *x["sp"], w), ref):
        assert_band(a, b, w)


def test_many_lines_take_the_line_per_thread_geometry_kernel(g):
    """2500 sets x 16 geometries = 40 000 lines: above the 256 x SMs lines at which the geometry records come from
    geom_lines_kernel (C4's chunks run there)"""
    n, ng = 2500, 16
    assert n * ng >= 256 * torch.cuda.get_device_properties(0).multi_processor_count
    x = make(g, 18, GRIDS["w40"], True, True, n_sets=n, n_geom=ng)
    w = bands_for(x["grid"])
    rsurf = g.brdf(x["st"], x["lut"], x["ang"], *x["sp"])
    assert np.isfinite(rsurf).mean() > 0.99
    assert_band(g.brdf_band(x["st"], x["lut"], x["ang"], *x["sp"], w), rsurf, w)


# ---- energy ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("gps,sps", LAYOUTS, ids=["shared", "spectra_per_set", "angles_per_set", "both_per_set"])
def test_energy_band_is_the_mean_of_energy(g, grid, gps, sps):
    x = make(g, 21, GRIDS[grid], gps, sps)
    w = bands_for(x["grid"])
    ref = g.energy(x["st"], x["lut"], x["ang"], *x["sp"])
    got = g.energy_band(x["st"], x["lut"], x["ang"], *x["sp"], w)
    for a, b in zip(got, ref):
        assert np.isfinite(b).all()
        assert_band(a, b, w)


@pytest.mark.parametrize("opt", [dict(beta=0.35), dict(fd=0.3)], ids=["beta", "fd"])
def test_energy_band_options(g, opt):
    x = make(g, 22, GRIDS["w211"], True, True)
    w = bands_for(x["grid"])
    ref = g.energy(x["st"], x["lut"], x["ang"], *x["sp"], **opt)
    for a, b in zip(g.energy_band(x["st"], x["lut"], x["ang"], *x["sp"], w, **opt), ref):
        assert_band(a, b, w)


# ---- device entry points, determinism --------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", sorted(GRIDS))
def test_dev_entry_points_equal_host_ones(g, grid):
    x = make(g, 31, GRIDS[grid], True, True)
    w = bands_for(x["grid"])
    B = w.shape[0]
    host_rb = g.brdf_band(x["st"], x["lut"], x["ang"], *x["sp"], w)
    host_en = g.energy_band(x["st"], x["lut"], x["ang"], *x["sp"], w)
    d_in = [dev(a) for a in (x["st"], x["lut"], x["ang"])] + [dev(a) for a in x["sp"]]
    d_w = dev(w)
    rb = torch.full((M, G, B), SENT, dtype=torch.float64, device="cuda:0")
    en = [torch.full((M, G, B), SENT, dtype=torch.float64, device="cuda:0") for _ in range(3)]
    torch.cuda.synchronize()        # the fills above ran on torch's stream; the calls run on the context's
    g.brdf_band_dev(*d_in, d_w, rb)
    g.energy_band_dev(*d_in, d_w, *en)
    g.synchronize()
    assert np.array_equal(rb.cpu().numpy(), host_rb)
    for a, b in zip(en, host_en):
        assert np.array_equal(a.cpu().numpy(), b)


def test_identical_calls_give_identical_bits(g):
    x = make(g, 32, GRIDS["w211"], True, True)
    w = bands_for(x["grid"])
    a = g.brdf_band(x["st"], x["lut"], x["ang"], *x["sp"], w)
    e = g.energy_band(x["st"], x["lut"], x["ang"], *x["sp"], w)
    assert np.array_equal(a, g.brdf_band(x["st"], x["lut"], x["ang"], *x["sp"], w))
    for p, q in zip(e, g.energy_band(x["st"], x["lut"], x["ang"], *x["sp"], w)):
        assert np.array_equal(p, q)
    f1 = g.forward_band(x["st"], x["leaf"], x["soil"], x["grid"], w, x["ang"])
    assert np.array_equal(f1, g.forward_band(x["st"], x["leaf"], x["soil"], x["grid"], w, x["ang"]))


# ---- forward operator ------------------------------------------------------------------------------------------------
def modis_1nm():
    return np.concatenate([gort_b200.band_weights(GRID_1NM, [lo, hi], [1.0, 1.0]) for lo, hi in MODIS_EDGES])


def test_forward_band_full_grid_several_chunks(g):
    """2500 members (chunks of 1024, 1024, 452) on the full 2101-column grid with the 7 MODIS land bands: equal to
    brdf_band on LUTs and spectra from separate calls, and to the band mean of forward(); lut_out equals lut()."""
    n, ng = 2500, 4
    x = make(g, 41, GRID_1NM, True, True, n_sets=n, n_geom=ng)
    w = modis_1nm()
    rb, lut = g.forward_band(x["st"], x["leaf"], x["soil"], GRID_1NM, w, x["ang"], want_lut=True)
    assert rb.shape == (n, ng, 7)
    assert np.array_equal(lut, x["lut"])
    sep = g.brdf_band(x["st"], x["lut"], x["ang"], *x["sp"], w)
    fin = np.isfinite(sep)
    assert fin.mean() > 0.99               # a few random crowns give NaN lines, as they do per wavelength
    assert np.array_equal(np.isfinite(rb), fin)
    assert np.all(np.abs(rb[fin] - sep[fin]) <= 1e-12 * np.abs(sep[fin]))
    rsurf = g.forward(x["st"], x["leaf"], x["soil"], GRID_1NM, x["ang"])
    assert_band(rb, rsurf, w)


@pytest.mark.parametrize("case", ["user_leaf", "user_soil", "q08", "shared_angles_fd"])
def test_forward_band_variants(g, case):
    n = 1100                       # above one chunk (1024) and not a multiple of it
    x = make(g, 42, GRIDS["w211"], case != "shared_angles_fd", True, n_sets=n, n_geom=3)
    w = bands_for(x["grid"])
    kw = dict(user_leaf=0.12) if case == "user_leaf" else dict(user_soil=0.08) if case == "user_soil" else \
        dict(method=gort_b200.LUT_Q08) if case == "q08" else dict(fd=0.4)
    leaf = None if case == "user_leaf" else x["leaf"]
    soil = None if case == "user_soil" else x["soil"]
    rb = g.forward_band(x["st"], leaf, soil, x["grid"], w, x["ang"], **kw)
    rsurf = g.forward(x["st"], leaf, soil, x["grid"], x["ang"], **kw)
    assert np.isfinite(rsurf).mean() > 0.99
    assert_band(rb, rsurf, w)


# ---- stream switches in overlap mode ---------------------------------------------------------------------------------
_streams = []                     # kept alive for the context (include/gort_b200.h)


def test_band_call_between_overlap_mode_brdf_calls():
    """overlap-mode brdf_dev, a band call on another stream, then brdf_dev calls back on the first stream: every result
    equals that of the same calls in plain order"""
    ctx = gort_b200.Gort(0)
    try:
        xa = make(ctx, 51, GRIDS["w211"], True, True)
        xb = make(ctx, 52, GRIDS["w211"], True, True)
        w = bands_for(xa["grid"])
        B = w.shape[0]
        ins = {k: [dev(a) for a in (x["st"], x["lut"], x["ang"])] + [dev(a) for a in x["sp"]] for k, x in (("a", xa), ("b", xb))}
        d_w = dev(w)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        _streams.extend([s1, s2])

        def run(overlap):
            ctx.set_overlap(overlap)
            X = torch.full((M, G, w.shape[1]), SENT, dtype=torch.float64, device="cuda:0")
            Y = torch.empty_like(X)
            RB = torch.full((M, G, B), SENT, dtype=torch.float64, device="cuda:0")
            torch.cuda.synchronize()
            ctx.brdf_dev(*ins["b"], X, stream=s1.cuda_stream)
            ctx.brdf_dev(*ins["a"], X, stream=s1.cuda_stream)
            with torch.cuda.stream(s1):
                Y.copy_(X)
            ctx.brdf_band_dev(*ins["a"], d_w, RB, stream=s2.cuda_stream)
            ctx.brdf_dev(*ins["b"], X, stream=s1.cuda_stream)
            ctx.brdf_dev(*ins["a"], X, stream=s1.cuda_stream)
            ctx.synchronize()
            return Y.cpu().numpy(), RB.cpu().numpy(), X.cpu().numpy()

        plain = run(False)
        over = run(True)
        for p, q in zip(plain, over):
            assert np.array_equal(p, q)
        assert np.array_equal(plain[0], plain[2])
        assert_band(plain[1], plain[0], w)
    finally:
        ctx.close()


# ---- validation ------------------------------------------------------------------------------------------------------
def _raw_calls(g, x, w, n_bands, out_pitch=0):
    """the three host entry points through ctypes with sentinel-filled outputs -> [(rc, outputs)]"""
    st, lut, ang = (np.ascontiguousarray(a) for a in (x["st"], x["lut"], x["ang"]))
    rl, tl, rs = x["sp"]
    W = rl.shape[-1]
    w = None if w is None else np.ascontiguousarray(w, dtype=np.float64)
    sh = g._shape(M, G, W, ang.ndim == 3, rl.ndim == 2, out_pitch=out_pitch)
    p = lambda a: None if a is None else a.ctypes.data
    res = []
    o = np.full((M, G, 8), SENT)
    rc = g._lib.gort_brdf_band_batch(g._h, C.byref(sh), n_bands, p(w), p(st), p(lut), p(ang), p(rl), p(tl), p(rs), p(o))
    res.append((rc, [o]))
    e = [np.full((M, G, 8), SENT) for _ in range(3)]
    rc = g._lib.gort_energy_band_batch(g._h, C.byref(sh), n_bands, p(w), p(st), p(lut), p(ang), p(rl), p(tl), p(rs),
                                       *[p(a) for a in e])
    res.append((rc, e))
    f = np.full((M, G, 8), SENT)
    fl = np.full((M, gort_b200.LUT_STRIDE), SENT)
    rc = g._lib.gort_forward_band_batch(g._h, C.byref(sh), 0, p(st), p(x["leaf"]), p(x["soil"]), -1.0, -1.0,
                                        p(np.ascontiguousarray(x["grid"])), n_bands, p(w), p(ang), p(f), p(fl))
    res.append((rc, [f, fl]))
    return res


def _bad_weights(w, kind):
    w = w.copy()
    if kind == "nan":
        w[2, 5] = np.nan
    elif kind == "inf":
        w[1, 0] = np.inf
    elif kind == "negative":
        w[4, 3] = -1e-3
    elif kind == "empty_row":
        w[3] = 0.0
    return w


@pytest.mark.parametrize("kind", ["nan", "inf", "negative", "empty_row", "zero_bands", "too_many_bands", "out_pitch",
                                  "null_weights"])
def test_host_validation_errors_enqueue_nothing(g, kind):
    x = make(g, 61, GRIDS["w40"], True, True)
    w = bands_for(x["grid"])
    n_bands = {"zero_bands": 0, "too_many_bands": gort_b200.MAX_BANDS + 1}.get(kind, w.shape[0])
    if kind == "too_many_bands":
        w = np.tile(w, (14, 1))[:n_bands]
    w = None if kind == "null_weights" else _bad_weights(w, kind)
    for rc, outs in _raw_calls(g, x, w, n_bands, out_pitch=64 if kind == "out_pitch" else 0):
        assert rc == 1, g._lib.gort_last_error(g._h)
        for o in outs:
            assert (o == SENT).all()


def test_forward_band_range_error_covers_every_wavelength(g):
    x = make(g, 62, GRIDS["w40"], True, True)
    grid = x["grid"].copy()
    grid[-1] = 2501.0                                     # outside 400-2500, and outside every band
    w = bands_for(x["grid"])
    w[:, -1] = 0.0
    x = dict(x, grid=grid)
    rc, outs = _raw_calls(g, x, w, w.shape[0])[2]
    assert rc == 3
    for o in outs:
        assert (o == SENT).all()


@pytest.mark.parametrize("kind", ["zero_bands", "too_many_bands", "out_pitch"])
def test_dev_validation_errors_enqueue_nothing(g, kind):
    x = make(g, 63, GRIDS["w40"], True, True)
    w = bands_for(x["grid"])
    d_in = [dev(a) for a in (x["st"], x["lut"], x["ang"])] + [dev(a) for a in x["sp"]]
    out = torch.full((M, G, 8), SENT, dtype=torch.float64, device="cuda:0")
    n_bands = {"zero_bands": 0, "too_many_bands": gort_b200.MAX_BANDS + 1}.get(kind, w.shape[0])
    d_w = dev(np.tile(w, (14, 1)))
    sh = g._shape(M, G, w.shape[1], True, True, out_pitch=64 if kind == "out_pitch" else 0)
    ptrs = [C.c_void_p(t.data_ptr()) for t in d_in]
    rc = g._lib.gort_brdf_band_batch_dev(g._h, None, C.byref(sh), n_bands, C.c_void_p(d_w.data_ptr()), *ptrs,
                                         C.c_void_p(out.data_ptr()))
    assert rc == 1
    rc = g._lib.gort_energy_band_batch_dev(g._h, None, C.byref(sh), n_bands, C.c_void_p(d_w.data_ptr()), *ptrs,
                                           *[C.c_void_p(out.data_ptr())] * 3)
    assert rc == 1
    rc = g._lib.gort_brdf_band_batch_dev(g._h, None, C.byref(sh), w.shape[0], None, *ptrs, C.c_void_p(out.data_ptr()))
    assert rc == 1
    g.synchronize()
    assert (out == SENT).all()


@pytest.mark.parametrize("grid", sorted(GRIDS))
def test_defective_device_rows_give_nan_in_their_band_only(g, grid):
    x = make(g, 64, GRIDS[grid], True, True)
    w = bands_for(x["grid"])
    bad = w.copy()
    bad[0, 2] = np.nan
    bad[2, 4] = -0.5
    bad[3] = 0.0
    good = [1, 4]
    d_in = [dev(a) for a in (x["st"], x["lut"], x["ang"])] + [dev(a) for a in x["sp"]]
    B = w.shape[0]
    rb = torch.full((M, G, B), SENT, dtype=torch.float64, device="cuda:0")
    en = [torch.full((M, G, B), SENT, dtype=torch.float64, device="cuda:0") for _ in range(3)]
    d_bad = dev(bad)
    torch.cuda.synchronize()
    g.brdf_band_dev(*d_in, d_bad, rb)
    g.energy_band_dev(*d_in, d_bad, *en)
    g.synchronize()
    rsurf = g.brdf(x["st"], x["lut"], x["ang"], *x["sp"])
    ref_en = g.energy(x["st"], x["lut"], x["ang"], *x["sp"])
    for got, ref in [(rb, rsurf)] + list(zip(en, ref_en)):
        got = got.cpu().numpy()
        assert np.isnan(got[..., [0, 2, 3]]).all()
        assert_band(got[..., good], ref, w[good])


# ---- the oracle ------------------------------------------------------------------------------------------------------
def test_small_case_against_the_oracle(g, oracle):
    x = make(g, 71, GRIDS["w40"], True, True, n_sets=2, n_geom=3)
    w = bands_for(x["grid"])
    luts = np.stack([oracle.lut(x["st"][:, m]) for m in range(2)])
    sp = [np.stack(a) for a in zip(*[oracle.spectra(x["leaf"][:, m], x["soil"][:, m], x["grid"]) for m in range(2)])]
    rb = g.brdf_band(x["st"], luts, x["ang"], *sp, w)
    en = g.energy_band(x["st"], luts, x["ang"], *sp, w)
    ref_b = np.stack([band_mean(oracle.brdf(x["st"][:, m], luts[m], x["ang"][:, m, :].T, sp[0][m], sp[1][m], sp[2][m])[0], w)
                      for m in range(2)])
    ref_e = [np.stack(r) for r in zip(*[[band_mean(a, w) for a in oracle.energy(x["st"][:, m], luts[m], x["ang"][:, m, :].T,
                                                                                sp[0][m], sp[1][m], sp[2][m])]
                                        for m in range(2)])]

    def rel(a, b):
        return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-12)))

    assert rel(rb, ref_b) <= 1e-9
    for a, b in zip(en, ref_e):
        assert rel(a, b) <= 1e-9
