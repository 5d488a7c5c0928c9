"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle on the same seeded
inputs.  Tolerance (BASELINE.json north_star / SURVEY.md 8d):
        |x - ref| <= 1e-9 * max(|ref|, 1e-12),  NaN positions must coincide.
"""
import numpy as np
import pytest

from gort_b200 import workloads as wk
import gort_b200
from checkers import assert_close, assert_close_cond, sensitivity

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------
def test_c1_readme_end_to_end(gort, oracle):
    w = wk.c1_readme()
    st = w["structure"]
    lut = gort.lut(st)
    lut_o = oracle.lut(st[:, 0])
    assert_close(lut[0], lut_o, "lut")
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], w["wavelength"])
    rl_o, tl_o, rs_o = oracle.spectra(w["leaf"][:, 0], w["soil"][:, 0], w["wavelength"])
    assert_close(rl[0], rl_o, "rleaf"); assert_close(tl[0], tl_o, "tleaf"); assert_close(rs[0], rs_o, "rsoil")
    rsurf, scomp, kprop = gort.brdf(st, lut, w["angles"], rl[0], tl[0], rs[0], want_scomp=True, want_kprop=True)
    r_o, s_o, k_o = oracle.brdf(st[:, 0], lut_o, w["angles"].T, rl_o, tl_o, rs_o)
    assert_close(rsurf[0], r_o, "rsurf"); assert_close(scomp[0], s_o, "scomp"); assert_close(kprop[0], k_o, "kprop")


def test_golden_e1_alb_leaf(gort):
    """SURVEY.md App. E1: -LAI 4.0 -alb_leaf 0.5, full-precision values captured from the reference."""
    st = gort_b200.structure_from_options(lai=4.0).reshape(6, 1)
    wl = np.array([450.0, 600.0, 800.0, 1000.0])
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(None, wk.DEFAULT_SOIL.reshape(4, 1), wl, user_leaf=0.5)
    rsurf, kprop = gort.brdf(st, lut, np.array([[10.0], [0.0], [30.0], [20.0]]), rl[0], tl[0], rs[0], want_kprop=True)
    gold = np.array([0.050996023726925049, 0.056904932488151413, 0.063793005449302428, 0.068538876965779413])
    assert_close(rsurf[0, 0], gold, "E1 rsurf")
    assert_close(kprop[0, 0], np.array([0.24500453130170924, 0.078537903246602814, 0.33486586946440577,
                                        0.34159169598728212]), "E1 K")
    alb, fv, fs = gort.energy(st, lut, np.array([[10.0], [0.0], [30.0], [20.0]]), rl[0], tl[0], rs[0])
    assert_close(np.array([alb[0, 0, 0], fv[0, 0, 0], fs[0, 0, 0]]),
                 np.array([0.063777031489123184, 0.68728814305278241, 0.24893482545809434]), "E1 energy")


def test_golden_e4_lut_rows(gort):
    st = gort_b200.structure_from_options(lai=4.0).reshape(6, 1)
    lut = gort.lut(st)[0]
    assert_close(np.array([lut[0], lut[91], lut[30], lut[91 + 30], lut[60], lut[91 + 60], lut[182], lut[183]]),
                 np.array([0.4827649653877204, 0.049784714005155141, 0.18980914239271468, 0.054402229555638691,
                           0.010675513076152983, 0.017277579752321828, 0.11690037154524389, 0.0348709390952388]),
                 "E4 LUT rows")


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", [gort_b200.LUT_FULL, gort_b200.LUT_Q08])
def test_lut_random_structures(gort, oracle, method):
    rng = np.random.Generator(np.random.PCG64(11))
    st = wk.random_structures(rng, 48)
    lut = gort.lut(st, method)
    worst, excused = 0.0, 0
    for m in range(st.shape[1]):
        lo = oracle.lut(st[:, m], method)
        sens = sensitivity(lambda c: c.lut(st[:, m], method), lo)
        e, n = assert_close_cond(lut[m], lo, sens, "lut set %d %r" % (m, st[:, m]))
        worst = max(worst, e); excused += n
    print("lut method %d: worst strict rel err %.3e, %d of %d entries excused by conditioning" % (
        method, worst, excused, lut.size))


def test_lut_c5_grid_corners(gort, oracle):
    """corners + a stride through the C5 structural grid (extreme crown shapes)."""
    st = wk.c5_lut_grid()["structure"]
    idx = np.unique(np.concatenate([np.arange(0, st.shape[1], 4099), [0, st.shape[1] - 1]]))
    sub = np.ascontiguousarray(st[:, idx])
    lut = gort.lut(sub)
    for k in range(sub.shape[1]):
        assert_close(lut[k], oracle.lut(sub[:, k]), "C5 grid point %d %r" % (idx[k], sub[:, k]))


def test_spectra_prospect_price(gort, oracle):
    rng = np.random.Generator(np.random.PCG64(12))
    leaf = wk.random_leaves(rng, 16)
    soil = np.stack([rng.uniform(0.05, 0.4, 16), rng.uniform(-0.1, 0.1, 16), rng.uniform(-0.05, 0.05, 16),
                     rng.uniform(-0.04, 0.04, 16)])
    wl = np.concatenate([np.array([400.0, 2500.0, 858.5, 469.25, 1240.75, 2499.999]), rng.uniform(400, 2500, 40),
                         wk.MODIS_BANDS])
    rl, tl, rs = gort.spectra(leaf, soil, wl)
    for m in range(16):
        rl_o, tl_o, rs_o = oracle.spectra(leaf[:, m], soil[:, m], wl)
        assert_close(rl[m], rl_o, "rleaf"); assert_close(tl[m], tl_o, "tleaf"); assert_close(rs[m], rs_o, "rsoil")
    # full 2101-band table
    r, t = gort.prospect(leaf[:, :3])
    for m in range(3):
        rl_o, tl_o, _ = oracle.spectra(leaf[:, m], soil[:, m], np.arange(400.0, 2501.0))
        assert_close(r[m], rl_o, "prospect refl"); assert_close(t[m], tl_o, "prospect tran")
    # user overrides (-alb_leaf / -alb_soil)
    rl, tl, rs = gort.spectra(None, None, wl, user_leaf=0.5, user_soil=0.2, n_sets=2)
    assert np.all(rl == 0.25) and np.all(tl == 0.25) and np.all(rs == 0.2)


def test_spectra_wavelength_out_of_range(gort):
    with pytest.raises(gort_b200.GortError) as ei:
        gort.spectra(wk.DEFAULT_LEAF.reshape(7, 1), wk.DEFAULT_SOIL.reshape(4, 1), np.array([399.0, 500.0]))
    assert ei.value.code == 3


# ---------------------------------------------------------------------------------------------
def _spectra_for(oracle, leaf, soil, wl):
    return oracle.spectra(leaf, soil, wl)


@pytest.mark.parametrize("nw", [7, 211])
def test_brdf_random_shared_geometry(gort, oracle, nw):
    """wide (W >= 64) and flat (W < 64) kernels; LUT from the oracle so only the BRDF path is compared."""
    rng = np.random.Generator(np.random.PCG64(13 + nw))
    M, G = 5, 97
    st = wk.random_structures(rng, M)
    leaf = wk.random_leaves(rng, M)
    wl = wk.MODIS_BANDS if nw == 7 else np.arange(400.0, 2501.0, 10.0)
    ang = np.stack([rng.uniform(-80, 89, G), rng.uniform(-400, 400, G), rng.uniform(-80, 89, G), rng.uniform(-400, 400, G)])
    ang[2, 10:40] = 35.0; ang[3, 10:40] = 100.0            # a run of lines sharing the sun (cached sun terms)
    ang[:, 0] = [0.0, 0.0, 0.0, 0.0]                       # nadir / overhead sun: beta = 0 branch
    lut = np.stack([oracle.lut(st[:, m]) for m in range(M)])
    sp = [oracle.spectra(leaf[:, m], wk.DEFAULT_SOIL, wl) for m in range(M)]
    rl = np.stack([s[0] for s in sp]); tl = np.stack([s[1] for s in sp]); rs = np.stack([s[2] for s in sp])
    rsurf, scomp, kprop = gort.brdf(st, lut, ang, rl, tl, rs, want_scomp=True, want_kprop=True)
    for m in range(M):
        r_o, s_o, k_o = oracle.brdf(st[:, m], lut[m], ang.T, rl[m], tl[m], rs[m])
        assert_close(rsurf[m], r_o, "rsurf set %d" % m)
        assert_close(scomp[m], s_o, "scomp set %d" % m)
        # Kt = max(0, 1 - Kc - Kz - Kg) is a difference of O(1) areal proportions: conditioning-aware
        ks = sensitivity(lambda c: c.brdf(st[:, m], lut[m], ang.T, rl[m], tl[m], rs[m])[2], k_o)
        assert_close_cond(kprop[m], k_o, ks, "kprop set %d" % m)
    # shared spectra + options (-beta, -diffuse)
    rsurf = gort.brdf(st, lut, ang, rl[0], tl[0], rs[0], beta=0.3, fd=0.8)
    for m in range(M):
        r_o, _, _ = oracle.brdf(st[:, m], lut[m], ang.T, rl[0], tl[0], rs[0], beta=0.3, fd=0.8)
        assert_close(rsurf[m], r_o, "rsurf(opt) set %d" % m)


def test_brdf_per_set_geometry_c4_sample(gort, oracle):
    w = wk.c4_enkf(n_members=64, seed=1002)
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    M = st.shape[1]
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], wl)
    rsurf = gort.brdf(st, lut, ang, rl, tl, rs)
    worst = 0.0
    for m in range(M):
        lut_o = oracle.lut(st[:, m])
        sp = oracle.spectra(w["leaf"][:, m], w["soil"][:, m], wl)
        r_o, _, _ = oracle.brdf(st[:, m], lut_o, ang[:, m, :].T, *sp)
        worst = max(worst, assert_close(rsurf[m], r_o, "C4 member %d" % m))
    print("C4 sample worst rel err %.3e" % worst)


def test_brdf_grazing_nan_parity(gort, oracle):
    """zenith > 89 deg: epgap row 90 is 0 -> -log(0) in the hotspot -> the reference yields NaN / Inf
    by design (SURVEY.md App. B6); positions must coincide."""
    st = gort_b200.structure_from_options(lai=4.0)
    lut = oracle.lut(st)
    wl = np.array([450.0, 800.0])
    rl, tl, rs = oracle.spectra(wk.DEFAULT_LEAF, wk.DEFAULT_SOIL, wl)
    ang = np.array([[89.5, 10.0, 30.0, 89.9], [0.0, 20.0, 0.0, 0.0], [30.0, 89.7, 89.2, 10.0], [0.0, 0.0, 180.0, 90.0]])
    rsurf = gort.brdf(st.reshape(6, 1), lut.reshape(1, -1), ang, rl, tl, rs)
    r_o, _, _ = oracle.brdf(st, lut, ang.T, rl, tl, rs)
    assert np.array_equal(np.isnan(rsurf[0]), np.isnan(r_o))
    assert_close(rsurf[0], r_o, "grazing")


def test_brdf_q08_lut_and_read_lut(gort, oracle, tmp_path):
    """E2: -q08_pn_kopen; and a "-P" LUT (rows 0..89 only, row 90 = 0) through the text layout."""
    st = gort_b200.structure_from_options(lai=4.0)
    wl = np.array([450.0, 600.0, 800.0, 1000.0])
    lut = gort.lut(st.reshape(6, 1), gort_b200.LUT_Q08)
    rl, tl, rs = gort.spectra(None, wk.DEFAULT_SOIL.reshape(4, 1), wl, user_leaf=0.5)
    ang = np.array([[10.0], [0.0], [30.0], [20.0]])
    rsurf = gort.brdf(st.reshape(6, 1), lut, ang, rl[0], tl[0], rs[0])
    assert_close(rsurf[0, 0], np.array([0.050742404003082275, 0.056485203146758124, 0.063178656471069655,
                                        0.067789806911394482]), "E2")
    full = gort.lut(st.reshape(6, 1))
    p = tmp_path / "lut.txt"
    gort_b200.lut_write_text(full[0], str(p))
    back = gort_b200.lut_read_text(str(p))
    assert back[90] == 0.0 and back[91 + 90] == 0.0
    keep = np.r_[0:90, 91:181, 182, 183]
    assert_close(back[keep], full[0][keep], "LUT text round trip", rtol=1e-15)
    r1 = gort.brdf(st.reshape(6, 1), back.reshape(1, -1), ang, rl[0], tl[0], rs[0])
    r_o, _, _ = oracle.brdf(st, back, ang.T, rl[0], tl[0], rs[0])
    assert_close(r1[0], r_o, "-P LUT")


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nw", [5, 70, 300])
def test_energy_random(gort, oracle, nw):
    rng = np.random.Generator(np.random.PCG64(14 + nw))
    M = 3
    st = wk.random_structures(rng, M)
    leaf = wk.random_leaves(rng, M)
    wl = np.sort(rng.uniform(400, 2500, nw))
    ang = np.array([[0.0, 10.0, 0.0, 0.0], [0.0, 0.0, 0.0, 0.0], [0.0, 30.0, 60.0, 75.0], [0.0, 40.0, 180.0, 300.0]])
    lut = np.stack([oracle.lut(st[:, m]) for m in range(M)])
    sp = [oracle.spectra(leaf[:, m], wk.DEFAULT_SOIL, wl) for m in range(M)]
    rl = np.stack([s[0] for s in sp]); tl = np.stack([s[1] for s in sp]); rs = np.stack([s[2] for s in sp])
    alb, fv, fs = gort.energy(st, lut, ang, rl, tl, rs)
    for m in range(M):
        a_o, v_o, s_o = oracle.energy(st[:, m], lut[m], ang.T, rl[m], tl[m], rs[m])
        assert_close(alb[m], a_o, "albedo set %d" % m)
        assert_close(fv[m], v_o, "favegt set %d" % m, rtol=1e-8)   # 1 - albedo - Fd2 + Fu2: cancellation, see DESIGN.md
        assert_close(fs[m], s_o, "fasoil set %d" % m)


def test_gauleg_nodes(gort, oracle):
    x, w = gort.gauleg()
    xo, wo = oracle.gauleg(32)
    assert_close(x, xo, "abscissa", rtol=1e-14); assert_close(w, wo, "weights", rtol=1e-13)


# ---------------------------------------------------------------------------------------------
def test_c2_full_size_properties(gort, oracle):
    """BASELINE config 2 at full size (11 664 lines x 2101 bands): oracle on a line subsample +
    size-independent properties (azimuth mirror symmetry, K proportions sum, device == host API)."""
    import torch
    w = wk.c2_hemisphere()
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], wl)
    rsurf, kprop = gort.brdf(st, lut, ang, rl[0], tl[0], rs[0], want_kprop=True)
    assert rsurf.shape == (1, 11664, 2101)
    assert np.isfinite(rsurf).all()
    # oracle on every 97th line
    idx = np.arange(0, ang.shape[1], 97)
    lut_o = oracle.lut(st[:, 0])
    sp_o = oracle.spectra(w["leaf"][:, 0], w["soil"][:, 0], wl)
    r_o, _, k_o = oracle.brdf(st[:, 0], lut_o, ang[:, idx].T, *sp_o)
    e = assert_close(rsurf[0, idx], r_o, "C2 subsample")
    print("C2 subsample worst rel err %.3e" % e)
    # mirror symmetry in relative azimuth: raz and 360 - raz give the same reflectance
    R = rsurf[0].reshape(18, 18, 36, 2101)
    for a in (1, 7, 17):
        assert_close(R[:, :, a], R[:, :, 36 - a], "azimuth mirror %d" % a, rtol=1e-12)
    # Kc + Kg + Kt + Kz == 1 wherever Kt was not clamped at 0
    ks = kprop[0].sum(axis=1)
    free = kprop[0][:, 2] > 0
    assert np.max(np.abs(ks[free] - 1.0)) < 1e-12
    # device-pointer API gives the same bits as the host-pointer API
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    out = torch.empty((1, 11664, 2101), dtype=torch.float64, device=dev)
    gort.brdf_dev(t(st), t(lut), t(ang), t(rl[0]), t(tl[0]), t(rs[0]), out)
    gort.synchronize()
    assert np.array_equal(out.cpu().numpy(), rsurf)
    # padded row pitch (line-aligned warp stores): same bits in the first W columns; the padding up to the end
    # of the row's last 128-byte line belongs to the call and receives copies of the last column
    outp = torch.full((1, 11664, 2112), -7.0, dtype=torch.float64, device=dev)
    gort.brdf_dev(t(st), t(lut), t(ang), t(rl[0]), t(tl[0]), t(rs[0]), outp)
    gort.synchronize()
    hp = outp.cpu().numpy()
    assert np.array_equal(hp[:, :, :2101], rsurf) and np.array_equal(hp[:, :, 2101:], np.repeat(rsurf[:, :, 2100:], 11, axis=2))
    # a pitch beyond that line: the extra columns are not touched
    outq = torch.full((1, 64, 2144), -7.0, dtype=torch.float64, device=dev)
    gort.brdf_dev(t(st), t(lut), t(ang[:, :64]), t(rl[0]), t(tl[0]), t(rs[0]), outq)
    gort.synchronize()
    hq = outq.cpu().numpy()
    assert np.array_equal(hq[:, :, :2101], rsurf[:, :64]) and np.all(hq[:, :, 2112:] == -7.0)
    # repeated calls into the same buffer overlap across calls (geometry kernel of call i+1 under the stores of
    # call i): results must still be those of the last call
    ang2 = ang.copy(); ang2[0] = (ang2[0] + 2.5) % 85.0
    d_a1, d_a2 = t(ang), t(ang2)
    d_in = (t(st), t(lut), t(rl[0]), t(tl[0]), t(rs[0]))
    ref2 = gort.brdf(st, lut, ang2, rl[0], tl[0], rs[0])
    gort.set_overlap(True)
    try:
        for k in range(6):
            gort.brdf_dev(d_in[0], d_in[1], d_a2 if k % 2 else d_a1, d_in[2], d_in[3], d_in[4], outp)
        gort.synchronize()
        assert np.array_equal(outp.cpu().numpy()[:, :, :2101], ref2)
        # the same through the chunked kernel (a dense, unaligned pitch cannot take the full-spectrum kernel)
        for k in range(6):
            gort.brdf_dev(d_in[0], d_in[1], d_a2 if k % 2 else d_a1, d_in[2], d_in[3], d_in[4], out)
        gort.synchronize()
        assert np.array_equal(out.cpu().numpy(), ref2)
    finally:
        gort.set_overlap(False)


def test_overlap_mode_sees_other_gort_work_between_calls(gort):
    """Overlap mode (gort_set_overlap): a LUT / spectra call of this context between two same-shape BRDF calls rewrites
    inputs of the second one; the library must order the calls completely (ADVICE r1: the geometry kernel of the second
    call must not become a programmatic dependent of kopen_kernel / spectra_kernel)."""
    import torch
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    w = wk.c2_hemisphere(wl_step=1)
    ang, wl = w["angles"][:, :3000], w["wavelength"]
    G, W = ang.shape[1], wl.shape[0]
    sts = [gort_b200.structure_from_options(lai=lai).reshape(6, 1) for lai in (1.0, 2.0, 3.0, 4.0, 5.0, 6.0)]
    leaves = [wk.DEFAULT_LEAF.reshape(7, 1) * np.array([1, 1 + 0.2 * k, 1, 1, 1, 1, 1]).reshape(7, 1) for k in range(6)]
    d_ang, d_wl, d_soil = t(ang), t(wl), t(wk.DEFAULT_SOIL.reshape(4, 1))
    d_st = torch.empty((6, 1), dtype=torch.float64, device=dev)
    d_lut = torch.empty((1, gort_b200.LUT_STRIDE), dtype=torch.float64, device=dev)
    d_rl, d_tl, d_rs = (torch.empty((1, W), dtype=torch.float64, device=dev) for _ in range(3))
    out = torch.empty((1, G, 2112), dtype=torch.float64, device=dev)
    results = []
    ts = torch.cuda.Stream(device=dev)
    gort.set_overlap(True)
    try:
        with torch.cuda.stream(ts):
            for k in range(6):
                d_st.copy_(t(sts[k]), non_blocking=True)
                gort.lut_dev(d_st, d_lut, stream=ts.cuda_stream)                         # rewrites the LUT the BRDF reads
                gort.spectra_dev(t(leaves[k]), d_soil, d_wl, d_rl, d_tl, d_rs, stream=ts.cuda_stream)   # and the spectra
                gort.brdf_dev(d_st, d_lut, d_ang, d_rl[0], d_tl[0], d_rs[0], out, stream=ts.cuda_stream)
                results.append(out.clone())
        ts.synchronize()
        gort.synchronize()
    finally:
        gort.set_overlap(False)
    for k in range(6):
        lut = gort.lut(sts[k])
        rl, tl, rs = gort.spectra(leaves[k], wk.DEFAULT_SOIL.reshape(4, 1), wl)
        ref = gort.brdf(sts[k], lut, ang, rl[0], tl[0], rs[0])
        assert np.array_equal(results[k].cpu().numpy()[:, :, :W], ref), "step %d" % k


# ---------------------------------------------------------------------------------------------
# BASELINE.json configs 3-5 at FULL size: oracle on a subsample + size-independent properties
def test_c5_full_grid_properties_and_group_invariance(gort, oracle):
    """131 072 LUTs.  Consecutive grid points share the crown shape (cover and favd vary fastest), so the kernel
    computes the shape-only part once per group of sets; a set must get the same BITS whether it is computed
    inside a group, at a chunk boundary, or alone (this is also what makes the result independent of how the
    grid is sharded over GPUs)."""
    st = wk.c5_lut_grid()["structure"]
    M = st.shape[1]
    lut = gort.lut(st)
    assert lut.shape == (M, gort_b200.LUT_STRIDE)
    nan_sets = np.isnan(lut).any(axis=1)
    ok = ~nan_sets
    pn0, epg = lut[ok, :91], lut[ok, 91:182]
    assert np.all((pn0 >= 0) & (pn0 <= 1)) and np.all(epg >= -1e-15) and np.all(epg[:, 90] == 0.0)
    assert np.all(np.diff(pn0[:, :90], axis=1) <= 1e-12)            # gap probability falls with zenith
    assert np.all(lut[ok, 182] >= 0) and np.all(lut[ok, 182] <= 1.01)      # trapezoid of p_n0 sin(2 theta) over the clamped theta grid
    # same bits alone, in a different batch composition, and across chunk boundaries
    rng = np.random.Generator(np.random.PCG64(5))
    pick = np.unique(np.concatenate([rng.integers(0, M, 40), [0, 63, 64, 65, 127, 128, 16383, 16384, 16385, 7 * 16384 - 1, 7 * 16384, M - 1]]))   # group and pass boundaries
    for k in pick:
        alone = gort.lut(np.ascontiguousarray(st[:, k:k + 1]))[0]
        assert np.array_equal(alone, lut[k], equal_nan=True), "set %d differs when computed alone" % k
    lo = 777
    part = gort.lut(np.ascontiguousarray(st[:, lo:lo + 500]))
    assert np.array_equal(part, lut[lo:lo + 500], equal_nan=True)
    # NaN sets: the reference yields NaN for the same sets and entries (oracle on a sample of them + neighbours)
    idx = np.flatnonzero(nan_sets)
    print("C5: %d of %d LUTs contain NaN" % (idx.size, M))
    for k in np.concatenate([idx[:: max(1, idx.size // 6)][:6], idx[:1] - 1 if idx.size and idx[0] > 0 else []]).astype(int):
        lo_ = oracle.lut(st[:, k])
        sens = sensitivity(lambda c: c.lut(st[:, k]), lo_)
        assert_close_cond(lut[k], lo_, sens, "C5 grid point %d %r" % (k, st[:, k]))


def test_c4_full_size(gort, oracle):
    """10^5 members x 16 geometries x 7 bands, everything varying (LUT + spectra + BRDF on the GPU)."""
    w = wk.c4_enkf()
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    M = st.shape[1]
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], wl)
    rsurf = gort.brdf(st, lut, ang, rl, tl, rs)
    assert rsurf.shape == (M, 16, 7)
    bad_lut = np.isnan(lut).any(axis=1)
    # non-finite reflectances are part of the reference's behaviour (a zero within-crown gap probability in the
    # interpolated LUT row gives -log(0) in the hotspot, SURVEY.md App. B6): they must be rare and must coincide
    # with the reference's, which the sampled comparison below checks on some of them explicitly
    nonfin = ~np.isfinite(rsurf).all(axis=(1, 2))
    assert nonfin.mean() < 0.01
    fin = rsurf[~nonfin]
    assert fin.min() >= 0.0 and fin.max() < 1.5
    worst = 0.0
    sample = list(range(0, M, 4001)) + list(np.flatnonzero(nonfin & ~bad_lut)[:4]) + list(np.flatnonzero(bad_lut)[:2])
    for m in sample:
        lut_o = oracle.lut(st[:, m])
        sens = sensitivity(lambda c: c.lut(st[:, m]), lut_o)
        assert_close_cond(lut[m], lut_o, sens, "C4 LUT member %d" % m)
        sp = oracle.spectra(w["leaf"][:, m], w["soil"][:, m], wl)
        r_o, _, _ = oracle.brdf(st[:, m], lut[m], ang[:, m, :].T, *sp)      # same LUT: isolates the BRDF path
        worst = max(worst, assert_close(rsurf[m], r_o, "C4 member %d" % m))
    print("C4 full size: worst rel err %.3e over %d sampled members, %d members with NaN LUT, %d with non-finite output" % (
        worst, len(sample), bad_lut.sum(), nonfin.sum()))
    # 4a: structure shared, LAI only varying -> every member shares the crown shape (one LUT group per 64 members)
    wa = wk.c4_enkf(n_members=1000, vary_structure=False)
    luta = gort.lut(wa["structure"])
    for m in (0, 63, 64, 500, 999):
        assert np.array_equal(gort.lut(np.ascontiguousarray(wa["structure"][:, m:m + 1]))[0], luta[m], equal_nan=True)
        assert_close(luta[m], oracle.lut(wa["structure"][:, m]), "C4a LUT member %d" % m)


def test_c3_full_size(gort, oracle):
    """10^4 parameter sets x 3 sun angles x 211 bands x 512 quadrature nodes."""
    w = wk.c3_albedo()
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    M = st.shape[1]
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], wl)
    alb, fv, fs = gort.energy(st, lut, ang, rl, tl, rs)
    assert alb.shape == (M, 3, 211)
    # non-finite results are part of the reference's behaviour (zero within-crown gap probability in a LUT row
    # -> -log(0) in the hotspot): rare, and compared against the oracle on some of them below
    good = np.isfinite(alb).all(axis=(1, 2)) & np.isfinite(fv).all(axis=(1, 2)) & np.isfinite(fs).all(axis=(1, 2))
    assert good.mean() > 0.99
    a, v, s = alb[good], fv[good], fs[good]
    assert a.min() > 0.0 and a.max() < 1.0
    # energy balance: favegt = 1 - albedo - Fd2 + Fu2, fasoil = Fd2 - Fu2  (gortt_albedo.c:48-52)
    assert np.max(np.abs(a + v + s - 1.0)) < 1e-12
    print("C3 full size: %d of %d sets with non-finite results" % ((~good).sum(), M))
    for m in list(range(0, M, 1777)) + list(np.flatnonzero(~good)[:3]):
        sp = oracle.spectra(w["leaf"][:, m], w["soil"][:, m], wl)
        a_o, v_o, s_o = oracle.energy(st[:, m], lut[m], ang.T, *sp)
        assert_close(alb[m], a_o, "C3 albedo set %d" % m)
        assert_close(fv[m], v_o, "C3 favegt set %d" % m, rtol=1e-8)
        assert_close(fs[m], s_o, "C3 fasoil set %d" % m)


# ---------------------------------------------------------------------------------------------
# Shapes that exercise the per-wavelength kernel's control flow: several record stages per CTA, runs that cross
# stage and CTA boundaries, parameter-set changes inside a CTA's line range, every chunking of the spectrum.
@pytest.mark.parametrize("nw,pitch", [(64, 0), (65, 80), (96, 96), (127, 128), (333, 336), (700, 704), (1153, 1168), (2101, 0)])
def test_wide_kernel_shapes_partition_invariance(gort, oracle, nw, pitch):
    import torch
    rng = np.random.Generator(np.random.PCG64(100 + nw))
    M = 3
    G = 16000 if nw <= 128 else (4000 if nw < 1000 else 1500)      # M*G lines: up to ~160 lines per CTA -> 2 stages
    st = wk.random_structures(rng, M)
    leaf = wk.random_leaves(rng, M)
    wl = np.sort(rng.uniform(400, 2500, nw))
    # runs of random length (1..300 lines) sharing the sun, random views
    sza = np.empty(G); saa = np.empty(G)
    k = 0
    while k < G:
        n = int(rng.integers(1, 300))
        sza[k:k + n] = rng.uniform(0, 80); saa[k:k + n] = rng.uniform(0, 360)
        k += n
    ang = np.stack([rng.uniform(0, 85, G), rng.uniform(0, 360, G), sza, saa])
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(leaf, np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), M, axis=1), wl)
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    P = pitch if pitch else nw
    out = torch.full((M, G, P), -3.0, dtype=torch.float64, device=dev)
    gort.brdf_dev(t(st), t(lut), t(ang), t(rl), t(tl), t(rs), out)
    gort.synchronize()
    full = out.cpu().numpy()
    # columns beyond the padded line are untouched; padding inside the last 128-byte line copies the last band
    ncol = min(P, (nw + 15) // 16 * 16) if P % 16 == 0 else nw
    assert np.all(full[:, :, ncol:] == -3.0)
    if ncol > nw:
        assert np.array_equal(full[:, :, nw:ncol], np.repeat(full[:, :, nw - 1:nw], ncol - nw, axis=2))
    full = full[:, :, :nw]
    # same bits when the lines are evaluated in separate calls, one set at a time, cut at arbitrary places
    cuts = [0, 1, 130, 131, 5000 if G > 5000 else G // 2, G]
    for m in range(M):
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            part = gort.brdf(st[:, m:m + 1], lut[m:m + 1], ang[:, lo:hi], rl[m], tl[m], rs[m])
            assert np.array_equal(part[0], full[m, lo:hi], equal_nan=True), "set %d lines %d:%d differ from the batched call" % (m, lo, hi)
    # oracle on a subsample of lines of every set
    idx = np.unique(np.concatenate([np.arange(0, G, max(1, G // 25)), [0, 127, 128, 129, G - 1]]))
    for m in range(M):
        lut_o = oracle.lut(st[:, m])
        r_o, _, _ = oracle.brdf(st[:, m], lut[m], ang[:, idx].T, rl[m], tl[m], rs[m])
        assert_close(full[m, idx], r_o, "set %d" % m)
    # component signatures through the scomp variant of the kernel: rsurf must agree with the fast path to rounding
    r2, sc = gort.brdf(st, lut, ang[:, :600], rl, tl, rs, want_scomp=True)
    assert_close(r2, full[:, :600], "scomp-path rsurf vs fast path", rtol=1e-12)
    for m in range(M):
        _, s_o, _ = oracle.brdf(st[:, m], lut[m], ang[:, :40].T, rl[m], tl[m], rs[m])
        assert_close(sc[m, :40], s_o, "scomp set %d" % m)


def test_small_and_degenerate_shapes(gort, oracle):
    """one line, one band, one set; band-set kernel boundary at W = 63 / 64."""
    st = gort_b200.structure_from_options(lai=2.5).reshape(6, 1)
    lut = gort.lut(st)
    for nw in (1, 2, 63, 64):
        wl = np.linspace(400.0, 2500.0, nw)
        rl, tl, rs = gort.spectra(wk.DEFAULT_LEAF.reshape(7, 1), wk.DEFAULT_SOIL.reshape(4, 1), wl)
        for ang in (np.array([[12.0], [40.0], [33.0], [250.0]]), np.array([[0.0, 60.0], [0.0, 10.0], [0.0, 60.0], [0.0, 10.0]])):
            r = gort.brdf(st, lut, ang, rl[0], tl[0], rs[0])
            r_o, _, _ = oracle.brdf(st[:, 0], lut[0], ang.T, rl[0], tl[0], rs[0])
            assert_close(r[0], r_o, "nw %d" % nw)
            a, v, s = gort.energy(st, lut, ang, rl[0], tl[0], rs[0])
            a_o, v_o, s_o = oracle.energy(st[:, 0], lut[0], ang.T, rl[0], tl[0], rs[0])
            assert_close(a[0], a_o, "albedo nw %d" % nw); assert_close(v[0], v_o, "favegt", rtol=1e-8); assert_close(s[0], s_o, "fasoil")
    with pytest.raises(gort_b200.GortError):
        gort.brdf(st, lut, np.zeros((4, 0)), np.zeros(3), np.zeros(3), np.zeros(3))


def test_wide_kernel_many_lines_multiwave_geometry(gort, oracle):
    """300 000 lines x 64 bands: the geometry kernel needs several waves of CTAs while the per-wavelength kernel,
    launched as its programmatic dependent, waits on the per-tile flags -- results must not depend on it."""
    rng = np.random.Generator(np.random.PCG64(321))
    M, G, nw = 2, 150000, 64
    st = wk.random_structures(rng, M)
    leaf = wk.random_leaves(rng, M)
    wl = np.sort(rng.uniform(400, 2500, nw))
    sza = np.repeat(rng.uniform(0, 75, G // 50), 50); saa = np.repeat(rng.uniform(0, 360, G // 50), 50)
    ang = np.stack([rng.uniform(0, 80, G), rng.uniform(0, 360, G), sza, saa])
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(leaf, np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), M, axis=1), wl)
    full = gort.brdf(st, lut, ang, rl, tl, rs)
    assert full.shape == (M, G, nw) and np.isfinite(full).all()
    for m in range(M):
        for lo, hi in ((0, 777), (74990, 75100), (G - 513, G)):
            part = gort.brdf(st[:, m:m + 1], lut[m:m + 1], ang[:, lo:hi], rl[m], tl[m], rs[m])
            assert np.array_equal(part[0], full[m, lo:hi])
        idx = np.arange(0, G, 2999)
        r_o, _, _ = oracle.brdf(st[:, m], lut[m], ang[:, idx].T, rl[m], tl[m], rs[m])
        assert_close(full[m, idx], r_o, "set %d" % m)


def test_forward_batch_equals_the_three_calls(gort):
    """gort_forward_batch (chunked: LUT -> spectra -> BRDF on the GPU, copies under kernels) returns the bits of
    gort_lut_batch + gort_spectra_batch + gort_brdf_batch; several chunks, ragged last chunk, both angle layouts."""
    w = wk.c4_enkf(n_members=5003, seed=77)
    st, ang, wl = w["structure"], w["angles"], w["wavelength"]
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], wl)
    want = gort.brdf(st, lut, ang, rl, tl, rs)
    got, lut2 = gort.forward(st, w["leaf"], w["soil"], wl, ang, want_lut=True)
    assert np.array_equal(got, want, equal_nan=True) and np.array_equal(lut2, lut, equal_nan=True)
    # shared geometry, options, -alb_leaf / -alb_soil style overrides
    shared = np.ascontiguousarray(ang[:, 0, :])
    want = gort.brdf(st, lut, shared, *gort.spectra(None, w["soil"], wl, user_leaf=0.4), beta=0.3, fd=0.7)
    got = gort.forward(st, None, w["soil"], wl, shared, user_leaf=0.4, beta=0.3, fd=0.7)
    assert np.array_equal(got, want, equal_nan=True)
    # a batch smaller than one chunk, Q08 LUTs
    small = np.ascontiguousarray(st[:, :7])
    lq = gort.lut(small, gort_b200.LUT_Q08)
    sp = gort.spectra(w["leaf"][:, :7], w["soil"][:, :7], wl)
    assert np.array_equal(gort.forward(small, w["leaf"][:, :7], w["soil"][:, :7], wl, shared, method=gort_b200.LUT_Q08),
                          gort.brdf(small, lq, shared, *sp), equal_nan=True)
    with pytest.raises(gort_b200.GortError) as ei:
        gort.forward(small, w["leaf"][:, :7], w["soil"][:, :7], np.array([399.0, 500.0]), shared)
    assert ei.value.code == 3


@pytest.mark.parametrize("nw,pitch", [(2101, 2112), (700, 704), (64, 64), (333, 352)])
def test_component_signatures_through_the_bulk_store_ring(gort, nw, pitch):
    """-prnspec with 128-byte aligned rows: rsurf and the { C, G, T, Z } quadruples leave through the shared-memory ring
    and cp.async.bulk; same bits as the per-thread store path (dense host arrays), padding columns hold copies of the
    last band, columns beyond the padded line are untouched."""
    import torch
    rng = np.random.Generator(np.random.PCG64(500 + nw))
    M, G = 2, 1500
    st = wk.random_structures(rng, M)
    leaf = wk.random_leaves(rng, M)
    wl = np.sort(rng.uniform(400, 2500, nw))
    sza = np.repeat(rng.uniform(0, 80, G // 30), 30); saa = np.repeat(rng.uniform(0, 360, G // 30), 30)
    ang = np.stack([rng.uniform(0, 85, G), rng.uniform(0, 360, G), sza, saa])
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(leaf, np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), M, axis=1), wl)
    r_ref, s_ref = gort.brdf(st, lut, ang, rl, tl, rs, want_scomp=True)          # dense rows: per-thread stores
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    d_r = torch.full((M, G, pitch), -9.0, dtype=torch.float64, device=dev)
    d_s = torch.full((M, G, pitch, 4), -9.0, dtype=torch.float64, device=dev)
    gort.brdf_dev(t(st), t(lut), t(ang), t(rl), t(tl), t(rs), d_r, scomp=d_s)
    gort.synchronize()
    r, sc = d_r.cpu().numpy(), d_s.cpu().numpy()
    assert np.array_equal(r[:, :, :nw], r_ref) and np.array_equal(sc[:, :, :nw], s_ref)
    ncol = min(pitch, (nw + 15) // 16 * 16)
    if ncol > nw:
        assert np.array_equal(r[:, :, nw:ncol], np.repeat(r[:, :, nw - 1:nw], ncol - nw, axis=2))
        assert np.array_equal(sc[:, :, nw:ncol], np.repeat(sc[:, :, nw - 1:nw], ncol - nw, axis=2))
    assert np.all(r[:, :, ncol:] == -9.0) and np.all(sc[:, :, ncol:] == -9.0)


def test_host_api_leaves_padding_columns_of_pitched_rows_alone(gort):
    """gort_brdf_batch with out_pitch > n_wl (host arrays): only the n_wl columns of every row are written."""
    import ctypes as C
    from gort_b200 import api
    w = wk.c1_readme()
    st, wl = w["structure"], np.arange(400.0, 2500.0, 30.0)              # 70 bands
    ang = np.stack([np.linspace(0, 60, 50), np.zeros(50), np.full(50, 30.0), np.linspace(0, 300, 50)])
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(w["leaf"], w["soil"], wl)
    dense, sc_dense = gort.brdf(st, lut, ang, rl[0], tl[0], rs[0], want_scomp=True)
    P = 96
    out = np.full((1, 50, P), -4.0); sc = np.full((1, 50, P, 4), -4.0)
    sh = gort._shape(1, 50, wl.size, False, False, out_pitch=P)
    a = [np.ascontiguousarray(x) for x in (st, lut, ang, rl[0], tl[0], rs[0])]
    rc = gort._lib.gort_brdf_batch(gort._h, C.byref(sh), *[api._ptr(x) for x in a], api._ptr(out), api._ptr(sc), None)
    assert rc == 0
    assert np.array_equal(out[:, :, :70], dense) and np.all(out[:, :, 70:] == -4.0)
    assert np.array_equal(sc[:, :, :70], sc_dense) and np.all(sc[:, :, 70:] == -4.0)
