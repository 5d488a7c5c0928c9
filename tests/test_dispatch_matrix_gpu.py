"""The BRDF and energy kernels on the variants, layouts and options that the workload tests do not reach.

launch_brdf (gort_b200/csrc/gort_brdf.cu) picks its kernels from the shape of each call: geom_kernel, or geom_lines_kernel
once there are at least 256 lines per SM; then rsurf_flat_kernel (W < 64) or one of the
rsurf_wide_kernel<LPT, SCOMP, TMAB> instantiations, chosen by the row pitch, the alignment of rsurf and scomp
and the wavelengths per thread that waste the fewest columns.  Every BRDF case below first asserts, from a torch.profiler
trace of the call, which kernels ran, so that a later change of the heuristic cannot quietly move a case off the path it
was written for.  Then it compares with the oracle on sampled lines and checks that the same sets computed alone, or as a
slice of another batch (other CTA line ranges, the other geometry kernel), give the same bits.

The angles contain what the wide kernel's run detection has to get right: runs of one line, long runs sharing the sun,
consecutive lines with sza = +x / -x (one run by design: every sun term depends on |sza| and the set only), set
boundaries between two lines with the same sun, and vza < 0, vaa > 360, saa < 0.
"""
import re

import numpy as np
import pytest

import gort_b200
from gort_b200 import workloads as wk
from checkers import assert_close, assert_close_cond, sensitivity
from test_jacobian_gpu import H, oracle_jacobian

pytestmark = pytest.mark.gpu

SENT = -5.0                                   # what output buffers hold before a call
OPTIONS = [{}, {"beta": 0.3, "fd": 0.8}]      # -beta / -diffuse


# ---- which kernels ran ----------------------------------------------------------------------------------------------
def kernel_key(name):
    """A kernel name as the profiler reports it -> 'geom_kernel', 'rsurf_wide_kernel<2,0,0>', ...  Accepts the
    demangled spellings '<2, false, 0>' and '<(int)2, (bool)0, ...>' and the mangled one."""
    m = re.search(r"([a-z_]+_kernel)I((?:L[ib]\d+E)+)E", name) if name.startswith("_Z") else None
    if m:
        return "%s<%s>" % (m.group(1), ",".join(re.findall(r"L[ib](\d+)E", m.group(2))))
    m = re.search(r"(\w+_kernel)(?:<([^>]*)>)?", name)
    if not m:
        return name
    if m.group(2) is None:
        return m.group(1)
    args = [re.sub(r"^\((int|bool)\)", "", a.strip()).replace("true", "1").replace("false", "0") for a in m.group(2).split(",")]
    return "%s<%s>" % (m.group(1), ",".join(args))


def test_kernel_key_spellings():
    want = "rsurf_wide_kernel<2,0,0>"
    assert kernel_key("void gort::rsurf_wide_kernel<2, false, 0>(gort::WideArgs)") == want
    assert kernel_key("void gort::rsurf_wide_kernel<(int)2, (bool)0, (int)0>(gort::WideArgs)") == want
    assert kernel_key("_ZN4gort17rsurf_wide_kernelILi2ELb0ELi0EEEvNS_8WideArgsE") == want
    assert kernel_key("gort::geom_lines_kernel(int, int, int, gort_options, const double *)") == "geom_lines_kernel"


@pytest.fixture
def traced():
    """traced(fn) -> (fn(), set of kernel_key of every gort kernel that ran inside fn), from torch.profiler with CUDA
    activity only."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    def run(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        names = {e.name() for e in prof.profiler.kineto_results.events() if e.device_type() == DeviceType.CUDA}
        got = {kernel_key(n) for n in names if "gort" in n}
        assert got, "the profiler recorded no gort kernel (CUDA kernels seen: %r)" % sorted(names)[:8]
        return out, got
    return run


def by_line_threshold():
    """lines from which launch_brdf takes geom_lines_kernel: 256 per SM"""
    import torch
    return 64 * 4 * torch.cuda.get_device_properties(0).multi_processor_count


# ---- inputs ---------------------------------------------------------------------------------------------------------
def sun_sequence(rng, n):
    """sza, saa of n consecutive lines: lines with a sun of their own, runs of 2..199 lines sharing one, and pairs of
    lines with sza = +x / -x (the second with the same or another saa).  Returns sza, saa, first lines of the pairs."""
    sza = np.empty(n); saa = np.empty(n); pairs = []
    k = 0
    while k < n:
        kind = int(rng.integers(0, 4))
        x = 0.0 if rng.random() < 0.05 else rng.uniform(-80.0, 80.0)
        ln = min(n - k, (1, int(rng.integers(2, 200)), 2, 2)[kind])
        sza[k:k + ln] = x; saa[k:k + ln] = rng.uniform(-400.0, 400.0)
        if kind >= 2 and ln == 2 and x != 0.0:
            sza[k + 1] = -x
            if kind == 3:
                saa[k + 1] = rng.uniform(-400.0, 400.0)
            pairs.append(k)
        k += ln
    return sza, saa, np.array(pairs, dtype=np.int64)


def make_angles(rng, M, G, per_set):
    """[4][M][G] (per set) or [4][G] degrees, and the first lines of the +/- pairs (flat line index m * G + g when per
    set).  Shared geometry: the last line repeats the first line's sun, so that every set boundary falls between two
    lines with the same sun; per set, runs cross set boundaries anyway."""
    n = M * G if per_set else G
    sza, saa, pairs = sun_sequence(rng, n)
    vza = rng.uniform(-85.0, 85.0, n); vaa = rng.uniform(-30.0, 400.0, n)
    if not per_set:
        sza[G - 1], saa[G - 1] = sza[0], saa[0]
        pairs = pairs[pairs + 1 < G - 1]
        return np.stack([vza, vaa, sza, saa]), pairs
    return np.stack([vza, vaa, sza, saa]).reshape(4, M, G), pairs


CASES = {
    # name: M, G, W, row pitch (0: dense), scomp, per-set geometry, per-set spectra, rsurf offset in doubles, kernels
    "lpt2_few_lines":       (4, 3000, 300, 0, False, False, True, 0, "geom_kernel", "rsurf_wide_kernel<2,0,0>"),
    "lpt2_many_lines":      (3, 20000, 301, 0, False, False, True, 0, "geom_lines_kernel", "rsurf_wide_kernel<2,0,0>"),
    "hyperspectral_tma":    (2000, 16, 211, 224, False, True, True, 0, "geom_kernel", "rsurf_wide_kernel<4,0,3>"),
    "hyperspectral_thread": (5000, 16, 211, 0, False, True, True, 0, "geom_lines_kernel", "rsurf_wide_kernel<4,0,0>"),
    "signatures_tma":       (1500, 7, 97, 112, True, True, True, 0, "geom_kernel", "rsurf_wide_kernel<2,1,2>"),
    "signatures_thread":    (1500, 7, 97, 0, True, True, False, 0, "geom_kernel", "rsurf_wide_kernel<2,1,0>"),
    "bands_geom_lines":     (4000, 16, 7, 0, True, True, True, 0, "geom_lines_kernel", "rsurf_flat_kernel"),
    "unaligned_rsurf":      (2, 1200, 2101, 2112, False, False, False, 1, "geom_kernel", "rsurf_wide_kernel<4,0,0>"),
    # rows that cannot take TMA with 65..96 (or 96 written) columns: LPT = 3 wastes the fewest columns
    "lpt3_dense":           (300, 16, 95, 0, False, True, True, 0, "geom_kernel", "rsurf_wide_kernel<3,0,0>"),
    "lpt3_padded_unaligned": (2, 1500, 90, 96, False, False, False, 1, "geom_kernel", "rsurf_wide_kernel<3,0,0>"),
}


class Inputs:
    def __init__(self, gort, seed, M, G, W, gps, sps):
        rng = np.random.Generator(np.random.PCG64(seed))
        self.M, self.G, self.W, self.gps, self.sps = M, G, W, gps, sps
        self.st = wk.random_structures(rng, M)
        leaf = wk.random_leaves(rng, M)
        wl = wk.MODIS_BANDS if W == 7 else np.sort(rng.uniform(400.0, 2500.0, W))
        self.ang, self.pairs = make_angles(rng, M, G, gps)
        self.lut = gort.lut(self.st)
        rl, tl, rs = gort.spectra(leaf, np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), M, axis=1), wl)
        self.spectra = (rl, tl, rs) if sps else (rl[0], tl[0], rs[0])
        self.rng = rng

    def ang_of(self, m):
        return self.ang[:, m, :] if self.gps else self.ang

    def spectra_of(self, m):
        return tuple(s[m] for s in self.spectra) if self.sps else self.spectra

    def subset(self, sets):
        """the inputs of the sets `sets` (an index array), as one batch"""
        st = np.ascontiguousarray(self.st[:, sets]); lut = np.ascontiguousarray(self.lut[sets])
        ang = np.ascontiguousarray(self.ang[:, sets, :]) if self.gps else self.ang
        sp = tuple(np.ascontiguousarray(s[sets]) for s in self.spectra) if self.sps else self.spectra
        return st, lut, ang, sp


def run_brdf(gort, traced, st, lut, ang, spectra, pitch, want_scomp, offset, opt):
    """one gort_brdf_batch_dev call into sentinel-filled buffers; rsurf is a view `offset` doubles into its buffer.
    -> dict(buf = rsurf's whole buffer, rsurf [M][G][pitch], scomp, kprop, kernels)"""
    import torch
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    M, G, W = st.shape[1], ang.shape[-1], spectra[0].shape[-1]
    P = pitch or W
    n = M * G * P
    buf = torch.full((n + 2,), SENT, dtype=torch.float64, device=dev)
    out = buf[offset:offset + n].view(M, G, P)
    sc = torch.full((M, G, P, 4), SENT, dtype=torch.float64, device=dev) if want_scomp else None
    kp = torch.full((M, G, 4), SENT, dtype=torch.float64, device=dev)
    args = [t(a) for a in (st, lut, ang) + tuple(spectra)]

    def call():
        gort.brdf_dev(*args, out, scomp=sc, kprop=kp, **opt)
        gort.synchronize()
    _, kernels = traced(call)
    b = buf.cpu().numpy()
    return dict(buf=b, rsurf=b[offset:offset + n].reshape(M, G, P), scomp=None if sc is None else sc.cpu().numpy(),
                kprop=kp.cpu().numpy(), kernels=kernels)


def written_columns(W, P):
    """columns of a row the call writes (include/gort_b200.h, out_pitch): the padding up to the end of the row's last
    128-byte line when the pitch is a multiple of 16"""
    return min(P, (W + 15) // 16 * 16) if P % 16 == 0 else W


def check_padding(res, W, P, what):
    ncol = written_columns(W, P)
    for k in ("rsurf", "scomp"):
        a = res[k]
        if a is None:
            continue
        if ncol > W:
            assert np.array_equal(a[:, :, W:ncol], np.repeat(a[:, :, W - 1:W], ncol - W, axis=2), equal_nan=True), \
                "%s: %s padding columns do not repeat the last band" % (what, k)
        assert np.all(a[:, :, ncol:] == SENT), "%s: %s columns beyond the padded line were written" % (what, k)
    return ncol


def line_sample(x, n_sets=8, n_random=40):
    """{set: sorted lines} for the oracle: first and last line (the set boundaries) and random lines of a sample of
    sets, the stage boundary at line 128, and both lines of every +/- pair"""
    rng, M, G = x.rng, x.M, x.G
    sets = set(range(M)) if M <= n_sets else {0, M - 1} | set(rng.choice(M, n_sets - 2, replace=False).tolist())
    picks = {m: {0, G - 1, *[g for g in (127, 128, 129) if g < G], *rng.integers(0, G, n_random).tolist()} for m in sets}
    both = np.concatenate([x.pairs, x.pairs + 1])
    if x.gps:
        for line in both:
            picks.setdefault(int(line // G), set()).add(int(line % G))
    else:
        for m in picks:
            picks[m] |= set(both.tolist())
    return {m: np.array(sorted(g)) for m, g in sorted(picks.items())}


def check_oracle(oracle, x, res, opt, what):
    W = x.W
    want_scomp = res["scomp"] is not None
    for m, gs in line_sample(x).items():
        A = np.ascontiguousarray(x.ang_of(m)[:, gs].T)
        sp = x.spectra_of(m)
        r_o, s_o, k_o = oracle.brdf(x.st[:, m], x.lut[m], A, *sp, want_scomp=want_scomp, **opt)
        assert_close(res["rsurf"][m, gs, :W], r_o, "%s: rsurf set %d" % (what, m))
        if want_scomp:
            assert_close(res["scomp"][m, gs, :W], s_o, "%s: scomp set %d" % (what, m))
        # Kt = max(0, 1 - Kc - Kz - Kg) is a difference of O(1) areal proportions: conditioning-aware where the strict
        # bound is missed
        k = res["kprop"][m, gs]
        try:
            assert_close(k, k_o, "")
        except AssertionError:
            ks = sensitivity(lambda c: c.brdf(x.st[:, m], x.lut[m], A, *sp, want_scomp=False, **opt)[2], k_o)
            assert_close_cond(k, k_o, ks, "%s: kprop set %d" % (what, m))


def assert_same_rows(part, full, sets, ncol, what):
    for k in ("rsurf", "scomp", "kprop"):
        if full[k] is None:
            continue
        a = part[k][:, :, :ncol] if k != "kprop" else part[k]
        b = full[k][sets][:, :, :ncol] if k != "kprop" else full[k][sets]
        assert np.array_equal(a, b, equal_nan=True), "%s: %s differs from the batched call" % (what, k)


@pytest.mark.parametrize("opt", OPTIONS, ids=["plain", "beta_fd"])
@pytest.mark.parametrize("case", list(CASES))
def test_brdf_dispatch_matrix(gort, oracle, traced, case, opt):
    M, G, W, pitch, want_scomp, gps, sps, offset, geom, per_wl = CASES[case]
    x = Inputs(gort, 700 + list(CASES).index(case), M, G, W, gps, sps)
    P = pitch or W
    full = run_brdf(gort, traced, x.st, x.lut, x.ang, x.spectra, pitch, want_scomp, offset, opt)
    assert full["kernels"] == {geom, per_wl}, "%s ran %r" % (case, sorted(full["kernels"]))
    ncol = check_padding(full, W, P, case)
    assert full["buf"][-1] == SENT and (offset == 0 or full["buf"][0] == SENT), "stores outside the rows of rsurf"
    check_oracle(oracle, x, full, opt, case)

    # partition invariance: a few sets alone (other CTA line ranges, geom_kernel) ...
    for m in sorted({0, M // 2, M - 1}):
        st, lut, ang, sp = x.subset(np.array([m]))
        part = run_brdf(gort, traced, st, lut, ang, sp, pitch, want_scomp, offset, opt)
        assert part["kernels"] == {"geom_kernel", per_wl}, "set %d alone ran %r" % (m, sorted(part["kernels"]))
        assert_same_rows(part, full, [m], ncol, "%s: set %d alone" % (case, m))
    # ... and a contiguous slice of sets in another batch: without the first set when the batch is large enough for
    # geom_lines_kernel, else repeated until it takes that kernel; either way the kprop of both geometry kernels meets
    if geom == "geom_lines_kernel":
        sets = np.arange(1, M)
    else:
        lo, n = M // 4, max(1, M // 3)
        reps = by_line_threshold() // (n * G) + 1
        sets = np.tile(np.arange(lo, lo + n), reps)
    st, lut, ang, sp = x.subset(sets)
    part = run_brdf(gort, traced, st, lut, ang, sp, pitch, want_scomp, offset, opt)
    assert part["kernels"] == {"geom_lines_kernel", per_wl}, "slice ran %r" % sorted(part["kernels"])
    assert_same_rows(part, full, sets, ncol, "%s: sets %d.. in a batch of %d" % (case, sets[0], sets.size))

    if case == "unaligned_rsurf":
        # the same rows into an aligned buffer take the bulk-store path: same bits, padding included
        al = run_brdf(gort, traced, x.st, x.lut, x.ang, x.spectra, pitch, want_scomp, 0, opt)
        assert al["kernels"] == {geom, "rsurf_wide_kernel<4,0,3>"}, "aligned rows ran %r" % sorted(al["kernels"])
        assert np.array_equal(al["rsurf"], full["rsurf"], equal_nan=True)
        assert np.array_equal(al["kprop"], full["kprop"], equal_nan=True)


# ---- component signatures: alignment -----------------------------------------------------------------------------
@pytest.mark.parametrize("nw", [7, 97], ids=["flat", "wide"])
def test_misaligned_scomp_is_refused(gort, oracle, nw):
    """scomp must be 32-byte aligned (include/gort_b200.h): the flat kernel stores each { C, G, T, Z } as one double4,
    the wide kernel as two double2.  An address 8 or 16 bytes off is refused before anything is enqueued, and the
    context keeps working."""
    import torch
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    x = Inputs(gort, 800 + nw, 2, 9, nw, False, False)
    args = [t(a) for a in (x.st, x.lut, x.ang) + x.spectra]
    n = 2 * 9 * nw
    out = torch.full((2, 9, nw), SENT, dtype=torch.float64, device=dev)
    sbuf = torch.full((4 * n + 4,), SENT, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    for off in (1, 2):
        with pytest.raises(gort_b200.GortError) as ei:
            gort.brdf_dev(*args, out, scomp=sbuf[off:off + 4 * n].view(2, 9, nw, 4))
        assert ei.value.code == 1 and "aligned" in str(ei.value)
    gort.synchronize()
    assert torch.all(out == SENT).item() and torch.all(sbuf == SENT).item()
    sc = sbuf[4:4 + 4 * n].view(2, 9, nw, 4)
    gort.brdf_dev(*args, out, scomp=sc)
    gort.synchronize()
    for m in range(2):
        r_o, s_o, _ = oracle.brdf(x.st[:, m], x.lut[m], x.ang.T, *x.spectra)
        assert_close(out[m].cpu().numpy(), r_o, "rsurf set %d" % m)
        assert_close(sc[m].cpu().numpy(), s_o, "scomp set %d" % m)


# ---- energy balance -------------------------------------------------------------------------------------------------
ENERGY_OPTIONS = [{}, {"beta": 0.3}, {"fd": 0.8}, {"beta": 0.3, "fd": 0.8}]


@pytest.mark.parametrize("nw", [511, 512, 513, 2101])
def test_energy_matrix(gort, oracle, nw):
    """energy_kernel strides the wavelengths by its 512 threads: W around and well beyond one stride; per-set suns with
    sza = 0, sza < 0 and saa > 360; every combination of -beta / -diffuse; shared and per-set spectra."""
    rng = np.random.Generator(np.random.PCG64(900 + nw))
    M, G = 3, 4
    st = wk.random_structures(rng, M)
    leaf = wk.random_leaves(rng, M)
    wl = np.sort(rng.uniform(400.0, 2500.0, nw))
    sza = np.array([[0.0, -35.0, 50.0, 70.0], [-60.0, 0.0, 20.0, -10.0], [45.0, -45.0, 0.0, 30.0]])
    saa = np.array([[0.0, 400.0, -30.0, 725.0], [10.0, 361.0, -200.0, 90.0], [370.0, 0.0, 180.0, -90.0]])
    ang = np.stack([rng.uniform(-60.0, 60.0, (M, G)), rng.uniform(0.0, 400.0, (M, G)), sza, saa])
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(leaf, np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), M, axis=1), wl)
    for per_set in (True, False):
        sp = (rl, tl, rs) if per_set else (rl[0], tl[0], rs[0])
        for opt in ENERGY_OPTIONS:
            what = "W %d %s spectra %r" % (nw, "per-set" if per_set else "shared", opt)
            alb, fv, fs = gort.energy(st, lut, ang, *sp, **opt)
            total = alb + fv + fs
            assert np.isfinite(total).mean() > 0.9, what
            assert np.nanmax(np.abs(total - 1.0)) <= 1e-12, what
            for m in range(M):
                spm = tuple(s[m] for s in sp) if per_set else sp
                a_o, v_o, s_o = oracle.energy(st[:, m], lut[m], np.ascontiguousarray(ang[:, m, :].T), *spm, **opt)
                assert_close(alb[m], a_o, "%s: albedo set %d" % (what, m))
                assert_close(fv[m], v_o, "%s: favegt set %d" % (what, m), rtol=1e-8)   # 1 - albedo - Fd2 + Fu2: cancellation
                assert_close(fs[m], s_o, "%s: fasoil set %d" % (what, m))


# ---- ensemble forward operator and Jacobian with many bands ----------------------------------------------------------
def test_hyperspectral_forward_and_jacobian(gort, oracle):
    """3000 members (three chunks of gort_forward_batch, the last one ragged) x 16 per-member geometries x 211 bands"""
    rng = np.random.Generator(np.random.PCG64(950))
    M, G = 3000, 16
    st = wk.random_structures(rng, M)
    leaf = wk.random_leaves(rng, M)
    soil = np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), M, axis=1)
    wl = np.arange(400.0, 2500.0 + 0.5, 10.0)
    ang, _ = make_angles(rng, M, G, True)
    got = gort.forward(st, leaf, soil, wl, ang)
    lut = gort.lut(st)
    want = gort.brdf(st, lut, ang, *gort.spectra(leaf, soil, wl))
    assert np.array_equal(got, want, equal_nan=True)
    jac, rsurf = gort.jacobian(st, leaf, soil, wl, ang, param=gort_b200.JAC_LAI, rel_step=H, want_rsurf=True)
    assert np.array_equal(rsurf, got, equal_nan=True)
    finite = np.isfinite(rsurf).all(axis=(1, 2))
    members = []
    for m in (0, 1023, 1024, 2047, 2048, M - 1):         # first and last members of the forward chunks
        while not finite[m]:
            m -= 1
        members.append(m)
    for m in members:
        want = oracle_jacobian(oracle, st[:, m].copy(), leaf[:, m], soil[:, m], wl, np.ascontiguousarray(ang[:, m, :].T), 5, True)
        err = np.max(np.abs(jac[m] - want)) / np.max(np.abs(want))
        assert err <= 1e-7, "member %d: Jacobian differs by %.3e of its largest entry" % (m, err)
