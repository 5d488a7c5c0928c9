"""Overlap mode (gort_set_overlap, include/gort_b200.h) on every per-wavelength kernel, and on the call sequences that
must and must not overlap.

In overlap mode the geometry kernel of call i+1 runs as a programmatic dependent under the store phase of call i.  The
results then rest on synchronisation inside the kernels: line records, (set, lambda) tables and ready flags alternate
between two buffers by call parity, and before its first store every per-wavelength CTA waits until the CTA with the
same index in the previous launch has finished.  They must still be exactly those of the calls made one at a time.

Every test works on contexts of its own, never on the session context, whose pipeline state other tests share.  The
expected bits of a call are those of the same call made alone, with overlap off, into sentinel-filled buffers of the
same layout (test_dispatch_matrix_gpu ties those calls to the oracle).  The comparison covers rsurf with its padding
columns and the guard elements around it, and scomp; beyond the padded line every column must keep the sentinel.
Consecutive calls cycle through K = 3 input sets, each with device tensors of its own and its own structure, LUT,
spectra and sun sequence.  The period 3 is coprime with the parity of the record buffers, so a call that read the
records, tables or flags of the call two back would produce different bits.

Engagement witness: with GORT_TIMELINE=<n> in the environment of gort_create, the n-th per-wavelength launch of the
context prints its timeline to stderr (timeline_report, gort_brdf.cu).  Its line "previous call: end ... max X" is the
time, in microseconds after the first CTA entry of launch n, at which the last CTA of launch n-1 finished.  X > 0:
launch n-1 was still storing when launch n started, the calls overlapped.  X < 0: strict order; that is deterministic
when the calls are not overlapped, because the next geometry kernel then waits for every CTA of launch n-1 to exit.
Launches n-1 and n must have the same grid for the stamps to be comparable.
"""
import os
import re
from pathlib import Path

import numpy as np
import pytest

import gort_b200
from gort_b200 import workloads as wk
from test_dispatch_matrix_gpu import CASES, OPTIONS, SENT, Inputs, by_line_threshold, check_padding
from test_jacobian_gpu import H

ROOT = Path(__file__).resolve().parent.parent
K = 3                                                          # input sets per test, cycled with period 3
CHAIN_CASES = [c for c in CASES if CASES[c][2] >= 64]          # every row that takes a per-wavelength kernel
# Rows whose calls are too short for a conclusive witness (2-4 MB of rsurf: call n-1 may finish before call n's CTAs
# start, overlap on or off).  On a B200 at 1000 W, over three runs, their witness read -1.4 .. +0.3 us; every other
# row read +5.6 .. +55 us with overlap on and -14 .. -3.4 us with it off.
SHORT = ("lpt3_dense", "lpt3_padded_unaligned")
SEQ_CASE = "hyperspectral_thread"                              # dense rows: the host-pointer calls can take them too


# ---- engagement witness ---------------------------------------------------------------------------------------------
_WITNESS = re.compile(r"previous call: end\s+min\s+(-?[\d.]+)\s+avg\s+(-?[\d.]+)\s+max\s+(-?[\d.]+)")


def witness(text):
    """X of the one timeline report in `text`: when the last CTA of the previous launch ended, in us after the first
    CTA entry of the reported launch"""
    found = _WITNESS.findall(text)
    assert len(found) == 1, "expected one timeline report, found %d in:\n%s" % (len(found), text[-3000:])
    return float(found[0][2])


def test_witness_parser():
    text = (ROOT / "profiles" / "r2_timeline_rsurf_wide.txt").read_text()
    assert witness(text) == 10.05                  # recorded on the C2 bench with overlap on
    assert witness(text.replace("max    10.05", "max   -12.40")) == -12.4
    for bad in ("", text + text):
        with pytest.raises(AssertionError):
            witness(bad)


@pytest.fixture
def contexts():
    """contexts(**env) -> a new gort_b200.Gort(0) created with `env` (GORT_TIMELINE=<n>, ...) in the environment, which
    is restored right after gort_create has read it.  Every context is closed when the test ends."""
    made = []

    def make(**env):
        saved = {k: os.environ.get(k) for k in env}
        os.environ.update({k: str(v) for k, v in env.items()})
        try:
            g = gort_b200.Gort(0)
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        made.append(g)
        return g
    yield make
    for g in made:
        g.close()


# ---- buffers, references, comparison --------------------------------------------------------------------------------
def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda:0"))


class Layout:
    """Output buffers of one shape: rsurf [M][G][pitch] as a view `offset` doubles into a buffer with one guard element
    at each end, optional scomp [M][G][pitch][4] and kprop [M][G][4]."""

    def __init__(self, M, G, W, pitch=0, scomp=False, offset=0, kprop=False):
        import torch
        full = lambda *shape: torch.full(shape, SENT, dtype=torch.float64, device=torch.device("cuda:0"))
        self.M, self.G, self.W, self.P, self.offset = M, G, W, pitch or W, offset
        n = M * G * self.P
        self.buf = full(n + 2)
        self.rsurf = self.buf[offset:offset + n].view(M, G, self.P)
        self.scomp = full(M, G, self.P, 4) if scomp else None
        self.kprop = full(M, G, 4) if kprop else None

    def outputs(self):
        return dict(rsurf=self.rsurf, scomp=self.scomp, kprop=self.kprop)

    def _whole(self):
        return {k: v for k, v in (("buf", self.buf), ("scomp", self.scomp), ("kprop", self.kprop)) if v is not None}

    def reset(self):
        """sentinel everywhere, complete before anything else is enqueued"""
        import torch
        for v in self._whole().values():
            v.fill_(SENT)
        torch.cuda.synchronize()

    def host(self):
        return {k: v.cpu().numpy() for k, v in self._whole().items()}

    def snapshot(self):
        """clones of the buffers, enqueued on the current stream"""
        return {k: v.clone() for k, v in self._whole().items()}


def reference(g, args, lay, opt):
    """the call alone on a context with overlap off, into sentinel-filled buffers -> host copies of the buffers, and
    rsurf [M][G][pitch] (what a host-pointer call returns for a dense layout)"""
    lay.reset()
    g.synchronize()
    g.brdf_dev(*args, **lay.outputs(), **opt)
    g.synchronize()
    res = lay.host()
    n = lay.M * lay.G * lay.P
    res["rsurf"] = res["buf"][lay.offset:lay.offset + n].reshape(lay.M, lay.G, lay.P)
    check_padding(dict(rsurf=res["rsurf"], scomp=res.get("scomp")), lay.W, lay.P, "reference")
    assert res["buf"][-1] == SENT and (lay.offset == 0 or res["buf"][0] == SENT), "reference: stores outside the rows"
    return res


def assert_bits(got, want, what):
    for k, v in got.items():
        w = want[k]
        same = (v == w) | (np.isnan(v) & np.isnan(w))
        assert same.all(), "%s: %s differs from the call made alone in %d of %d doubles (first at %r)" % (
            what, k, (~same).sum(), same.size, np.unravel_index(np.argmin(same), same.shape))


class Rig:
    """K input sets of one shape (a CASES row without its kernel columns), each with device tensors of its own, one
    output layout, and the expected bits of each set's call"""

    def __init__(self, ref_g, row, opt, seed, kprop=False):
        M, G, W, pitch, want_scomp, gps, sps, offset = row[:8]
        self.M, self.G, self.W, self.opt = M, G, W, opt
        self.xs = [Inputs(ref_g, seed + k, M, G, W, gps, sps) for k in range(K)]
        self.args = [[to_dev(a) for a in (x.st, x.lut, x.ang) + tuple(x.spectra)] for x in self.xs]
        self.lay = Layout(M, G, W, pitch, want_scomp, offset, kprop)
        self._bound = {}
        self.want = [reference(ref_g, a, self.lay, opt) for a in self.args]
        # the sets differ in their suns (so run boundaries move from call to call) and in their results
        sza = [x.ang[2] for x in self.xs]
        for i in range(K):
            j = (i + 1) % K
            assert not np.array_equal(sza[i], sza[j]), "input sets %d and %d share their sun sequence" % (i, j)
            assert not np.array_equal(self.want[i]["buf"], self.want[j]["buf"]), "sets %d and %d give the same bits" % (i, j)

    def with_(self, k, idx, tensor):
        """set k's arguments with argument idx (0 structure, 1 lut, 2 angles, 3 rleaf, 4 tleaf, 5 rsoil) replaced"""
        a = list(self.args[k])
        a[idx] = tensor
        return a

    def call(self, g, k, args=None, lay=None, stream=None):
        """enqueue set k's call (or `args`) into `lay` (default: the rig's layout) -> its host getter.  The plain form
        is bound once per context (brdf_dev_bind), so that the host stays ahead of the GPU."""
        if args is None and lay is None and stream is None:
            key = (id(g), k)
            if key not in self._bound:
                self._bound[key] = g.brdf_dev_bind(*self.args[k], **self.lay.outputs(), **self.opt)
            self._bound[key]()
            return self.lay.host
        lay = lay or self.lay
        g.brdf_dev(*(args or self.args[k]), **lay.outputs(), **self.opt, stream=stream)
        return lay.host


def run_chain(g, calls, n, lay):
    """from a synchronised start, calls[i % len(calls)]() for i < n into one output layout -> its buffers"""
    lay.reset()
    g.synchronize()
    for i in range(n):
        calls[i % len(calls)]()
    g.synchronize()
    return lay.host()


def host_of(snap):
    return {k: v.cpu().numpy() for k, v in snap.items()}


# ---- A. chains that must overlap ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("opt", OPTIONS, ids=["plain", "beta_fd"])
@pytest.mark.parametrize("case", CHAIN_CASES)
def test_chain_overlaps(contexts, capfd, record_property, case, opt):
    """Chains of n = 1..5 calls into one output buffer, each from a synchronised start: the buffer must hold exactly
    call n alone, so every call is checked as the last of an overlapped chain.  Launch 15 of the context is the last
    call of the 5-call chain; its witness shows whether it overlapped call 4.  The control, the same chain with overlap
    off, must run in strict order."""
    rig = Rig(contexts(), CASES[case], opt, 1000 + 10 * list(CASES).index(case))
    g = contexts(GORT_TIMELINE=15)
    g.set_overlap(True)
    calls = [g.brdf_dev_bind(*rig.args[k], **rig.lay.outputs(), **opt) for k in range(K)]
    capfd.readouterr()
    for n in range(1, 6):
        assert_bits(run_chain(g, calls, n, rig.lay), rig.want[(n - 1) % K], "%s: chain of %d calls" % (case, n))
    x_on = witness(capfd.readouterr().err)

    g_off = contexts(GORT_TIMELINE=5)
    calls = [g_off.brdf_dev_bind(*rig.args[k], **rig.lay.outputs(), **opt) for k in range(K)]
    assert_bits(run_chain(g_off, calls, 5, rig.lay), rig.want[4 % K], "%s: chain of 5 calls, overlap off" % case)
    x_off = witness(capfd.readouterr().err)
    record_property("witness_on_us", x_on)
    record_property("witness_off_us", x_off)
    assert x_off < 0, "%s, overlap off: launch 4 ended %.2f us after launch 5 started" % (case, x_off)
    if case not in SHORT:
        assert x_on > 0, "%s, overlap on: launch 4 ended %.2f us before launch 5 started: no overlap" % (case, -x_on)


def skewed_angles(rng, M, G, busy):
    """[4][M][G] degrees: sets below `busy` have a new sun on every line (the per-wavelength kernel re-derives its
    (sun, lambda) terms for each), the other sets one sun for all their lines"""
    vza = rng.uniform(-60.0, 60.0, (M, G)); vaa = rng.uniform(0.0, 360.0, (M, G))
    sza = np.repeat(rng.uniform(5.0, 70.0, (M, 1)), G, axis=1); saa = np.repeat(rng.uniform(0.0, 360.0, (M, 1)), G, axis=1)
    sza[:busy] = rng.uniform(5.0, 70.0, (busy, G)); saa[:busy] = rng.uniform(0.0, 360.0, (busy, G))
    return np.stack([vza, vaa, sza, saa])


@pytest.mark.gpu
def test_gate_holds_back_fast_ctas(contexts, capfd, record_property):
    """Call A spends ~10x longer in its low-index CTAs (a new sun on every line) than in the others; call B, the same
    shape, is cheap everywhere.  CTAs are dispatched in index order, so B's low-index CTAs start as A's cheap
    high-index CTAs retire, finish their start-up while A's CTAs of the same index are still storing, and store
    nothing before those are done only because of the per-CTA gate: without it part of A's rows would land on top
    of B's.  The chains A, B and A, B, A, B must leave exactly B alone."""
    M, G, W, P = 64, 4000, 211, 224
    ref_g = contexts()
    rng = np.random.Generator(np.random.PCG64(1700))
    st = wk.random_structures(rng, M)
    lut = ref_g.lut(st)
    wl = np.sort(rng.uniform(400.0, 2500.0, W))
    sp = ref_g.spectra(wk.random_leaves(rng, M), np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), M, axis=1), wl)
    lay = Layout(M, G, W, P)
    args = [[to_dev(a) for a in (st, lut, skewed_angles(rng, M, G, busy)) + tuple(sp)] for busy in (M // 4, 0)]
    want = [reference(ref_g, a, lay, {}) for a in args]
    assert not np.array_equal(want[0]["buf"], want[1]["buf"])
    # witness on launch 6, the last B: the first two calls of a context allocate the two record buffers, and that
    # allocation waits for the whole device, so launch 2 can never overlap launch 1
    g = contexts(GORT_TIMELINE=6)
    g.set_overlap(True)
    calls = [g.brdf_dev_bind(*a, **lay.outputs()) for a in args]
    capfd.readouterr()
    for n in (2, 4):
        assert_bits(run_chain(g, calls * 2, n, lay), want[1], "chain of %d calls" % n)
    x = witness(capfd.readouterr().err)
    record_property("witness_on_us", x)
    assert x > 0, "B's CTAs started %.2f us after A's last CTA ended: nothing was held back" % -x


@pytest.mark.gpu
def test_chain_with_kprop(contexts):
    """A call that requests kprop never overlaps the previous one: kprop is in launch_brdf's alias list and the
    signature requires the same kprop, so kprop always aliases the previous call's.  Bits only, no witness."""
    rig = Rig(contexts(), CASES["signatures_tma"], {}, 1500, kprop=True)
    g = contexts()
    g.set_overlap(True)
    calls = [g.brdf_dev_bind(*rig.args[k], **rig.lay.outputs()) for k in range(K)]
    for n in range(1, 6):
        assert_bits(run_chain(g, calls, n, rig.lay), rig.want[(n - 1) % K], "kprop chain of %d calls" % n)


# ---- B. a consumer between calls ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["hyperspectral_tma", "signatures_tma", "unaligned_rsurf", "lpt3_padded_unaligned"])
def test_consumer_between_calls(contexts, case):
    """call, consume, call: on one caller stream every call is followed by torch clones of its outputs.  The library
    still sees a wide call before each call; the clone kernel in between never triggers its dependents."""
    import torch
    rig = Rig(contexts(), CASES[case], {}, 1200 + 10 * list(CASES).index(case))
    g = contexts()
    g.set_overlap(True)
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()
    snaps = []
    with torch.cuda.stream(ts):
        for i in range(7):
            rig.call(g, i % K, stream=ts.cuda_stream)
            snaps.append(rig.lay.snapshot())
    g.synchronize()
    torch.cuda.synchronize()
    for i, snap in enumerate(snaps):
        assert_bits(host_of(snap), rig.want[i % K], "%s: snapshot after call %d" % (case, i + 1))


# ---- C. sequences that must serialise -------------------------------------------------------------------------------
def soil_from_table_dev(g, table, wl, rsoil, stream=None):
    M, W = rsoil.shape
    g._check(g._lib.gort_soil_from_table_dev(g._h, stream, table.data_ptr(), M, W, wl.data_ptr(), rsoil.data_ptr()))


class Aux:
    """what the sequences need beyond the rig: a second output buffer, work copies of inputs that other operations
    rewrite, and the expected bits of the calls that read them"""

    def __init__(self, ref_g, rig, seed):
        import torch
        M, G, W = rig.M, rig.G, rig.W
        a2 = rig.args[2]
        lay = rig.lay
        self.lay2 = Layout(M, G, W, lay.P if lay.P != W else 0, lay.scomp is not None, lay.offset)
        self.ts = torch.cuda.Stream()
        # a caller copy rewrites the angles
        self.ang_host = [torch.from_numpy(np.ascontiguousarray(x.ang)).pin_memory() for x in rig.xs]
        self.ang_w = torch.empty_like(rig.args[0][2])
        # gort_energy_batch_dev writes the albedo [M][1][W] of one sun line into the next call's rleaf
        self.sun = to_dev(np.array([[0.0], [0.0], [35.0], [120.0]]))
        self.rl_w = torch.empty_like(a2[3])
        self.fv, self.fs = (torch.empty((M, 1, W), dtype=torch.float64, device=a2[3].device) for _ in range(2))
        alb = torch.empty_like(self.fv)
        ref_g.energy_dev(a2[0], a2[1], self.sun, a2[3], a2[4], a2[5], alb, self.fv, self.fs)
        ref_g.synchronize()
        self.want_energy = reference(ref_g, rig.with_(2, 3, alb.view(M, W)), lay, rig.opt)
        # gort_soil_from_table_dev writes the next call's rsoil
        self.table = to_dev(0.12 + 0.1 * np.sin(np.arange(gort_b200.SOIL_TABLE_NW) / 150.0))
        self.wl = to_dev(np.linspace(400.0, 2500.0, W))
        self.rs_w = torch.empty_like(a2[5])
        rs = torch.empty_like(a2[5])
        soil_from_table_dev(ref_g, self.table, self.wl, rs)
        ref_g.synchronize()
        self.want_soil = reference(ref_g, rig.with_(2, 5, rs), lay, rig.opt)
        for w in (self.want_energy, self.want_soil):
            assert not np.array_equal(w["buf"], rig.want[2]["buf"])
        # a W < 64 call (rsurf_flat_kernel)
        fx = Inputs(ref_g, seed, 50, 16, 7, True, True)
        self.flat_args = [to_dev(a) for a in (fx.st, fx.lut, fx.ang) + tuple(fx.spectra)]
        self.flat_lay = Layout(50, 16, 7, 0, True)
        self.flat_want = reference(ref_g, self.flat_args, self.flat_lay, {})

    def reset(self, rig):
        """sentinel-filled outputs; the work inputs hold values the rewritten call must not see"""
        import torch
        for lay in (rig.lay, self.lay2, self.flat_lay):
            lay.reset()
        self.ang_w.copy_(rig.args[1][2])
        self.rl_w.copy_(rig.args[0][3])
        self.rs_w.copy_(rig.args[0][5])
        torch.cuda.synchronize()


# Each sequence enqueues BRDF calls and other operations on a context with overlap on; after each BRDF call it yields
# (getter of that call's output, expected bits).
def seq_plain(g, rig, aux):
    for i in range(4):
        yield rig.call(g, i % K), rig.want[i % K]


def seq_two_buffers(g, rig, aux):
    for i in range(4):
        yield rig.call(g, i % K, lay=(rig.lay, aux.lay2)[i % 2]), rig.want[i % K]


def seq_caller_copy(g, rig, aux):
    """a non-blocking host-to-device copy_ on the context's stream rewrites the angles before every call"""
    import torch
    ext = torch.cuda.ExternalStream(g.stream)
    for i in range(4):
        k = i % K
        with torch.cuda.stream(ext):
            aux.ang_w.copy_(aux.ang_host[k], non_blocking=True)
        yield rig.call(g, k, args=rig.with_(k, 2, aux.ang_w)), rig.want[k]


def seq_energy(g, rig, aux):
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    a2 = rig.args[2]
    g.energy_dev(a2[0], a2[1], aux.sun, a2[3], a2[4], a2[5], aux.rl_w.view(rig.M, 1, rig.W), aux.fv, aux.fs)
    yield rig.call(g, 2, args=rig.with_(2, 3, aux.rl_w)), aux.want_energy
    yield rig.call(g, 0), rig.want[0]


def seq_soil_table(g, rig, aux):
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    soil_from_table_dev(g, aux.table, aux.wl, aux.rs_w)
    yield rig.call(g, 2, args=rig.with_(2, 5, aux.rs_w)), aux.want_soil
    yield rig.call(g, 0), rig.want[0]


def seq_stream_switch(g, rig, aux):
    """the third call on another caller stream, its inputs written on that stream; the fourth back on the context's"""
    import torch
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    with torch.cuda.stream(aux.ts):
        args = [a.clone() for a in rig.args[2]]
    yield rig.call(g, 2, args=args, stream=aux.ts.cuda_stream), rig.want[2]
    yield rig.call(g, 0), rig.want[0]


def seq_toggle(g, rig, aux):
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    g.set_overlap(False)
    g.set_overlap(True)
    yield rig.call(g, 2), rig.want[2]
    yield rig.call(g, 0), rig.want[0]


def seq_profile(g, rig, aux):
    """gort_profile_begin armed for the third and fourth call"""
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    g.profile_begin(2)
    try:
        yield rig.call(g, 2), rig.want[2]
        yield rig.call(g, 0), rig.want[0]
        yield rig.call(g, 1), rig.want[1]
    finally:
        g.profile_end()


def seq_stamps(g, rig, aux):
    """kernel stamps on for the third call.  A stamped launch still releases its dependents and publishes its epochs,
    so the fourth call may overlap it: its bits show that it gates correctly on a stamped launch."""
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    g.kernel_stamps_enable(True)
    try:
        yield rig.call(g, 2), rig.want[2]
    finally:
        g.kernel_stamps_enable(False)
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]


def seq_narrow_between(g, rig, aux):
    """a W < 64 call between two wide calls; it is not a per-wavelength launch of the timeline"""
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    g.brdf_dev(*aux.flat_args, **aux.flat_lay.outputs())
    yield aux.flat_lay.host, aux.flat_want
    yield rig.call(g, 2), rig.want[2]
    yield rig.call(g, 0), rig.want[0]


def _host_call(g, rig, k):
    x = rig.xs[k]
    r = g.brdf(x.st, x.lut, x.ang, *x.spectra, **rig.opt)
    return (lambda: {"rsurf": r}), rig.want[k]


def seq_host_calls(g, rig, aux):
    for i in range(3):
        yield _host_call(g, rig, i % K)


def seq_host_between(g, rig, aux):
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    yield _host_call(g, rig, 2)
    yield rig.call(g, 0), rig.want[0]


def seq_synchronize(g, rig, aux):
    yield rig.call(g, 0), rig.want[0]
    yield rig.call(g, 1), rig.want[1]
    g.synchronize()
    yield rig.call(g, 2), rig.want[2]
    yield rig.call(g, 0), rig.want[0]


# name: sequence, per-wavelength launches whose witness must read X < 0 (X > 0 for the uninterrupted control)
SEQUENCES = {
    "plain": (seq_plain, [3]),
    "two_buffers": (seq_two_buffers, [3]),
    "caller_copy": (seq_caller_copy, [3]),
    "energy_into_rleaf": (seq_energy, [3]),
    "soil_table_into_rsoil": (seq_soil_table, [3]),
    "stream_switch": (seq_stream_switch, [3, 4]),
    "overlap_toggled": (seq_toggle, [3]),
    "profile_armed": (seq_profile, [3, 5]),
    "stamps_on": (seq_stamps, [3]),
    "narrow_between": (seq_narrow_between, [3]),
    "host_calls": (seq_host_calls, [2, 3]),
    "host_between": (seq_host_between, [3, 4]),
    "synchronize": (seq_synchronize, [3]),
}


def run_sequence(g, seq, rig, aux, stop=None):
    """seq from a synchronised start, cut after its `stop`-th BRDF call (None: run it all)
    -> (BRDF calls made, host copies of the last call's output, its expected bits)"""
    import torch
    aux.reset(rig)
    g.synchronize()
    gen = seq(g, rig, aux)
    n = 0
    for get, want in gen:
        n += 1
        if n == stop:
            break
    g.synchronize()
    torch.cuda.synchronize()
    got = get()
    gen.close()
    return n, got, want


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SEQUENCES))
def test_sequence(contexts, capfd, record_property, name):
    """Each witness launch is checked on a context of its own that runs the whole sequence.  Then every BRDF call's
    bits are checked as the last call of the sequence cut after it."""
    seq, launches = SEQUENCES[name]
    ref_g = contexts()
    rig = Rig(ref_g, CASES[SEQ_CASE], {}, 1400)
    aux = Aux(ref_g, rig, 1450)
    for w in launches:
        g = contexts(GORT_TIMELINE=w)
        g.set_overlap(True)
        capfd.readouterr()
        n, got, want = run_sequence(g, seq, rig, aux)
        assert_bits(got, want, "%s: call %d" % (name, n))
        x = witness(capfd.readouterr().err)
        record_property("witness_us_launch_%d" % w, x)
        if name == "plain":
            assert x > 0, "uninterrupted: launch %d ended %.2f us before launch %d started" % (w - 1, -x, w)
        else:
            assert x < 0, "%s: launch %d ended %.2f us after launch %d started" % (name, w - 1, x, w)
    for j in range(1, n):
        _, got, want = run_sequence(g, seq, rig, aux, stop=j)
        assert_bits(got, want, "%s: call %d" % (name, j))


# ---- D. buffers regrowing mid-chain ---------------------------------------------------------------------------------
@pytest.mark.gpu
def test_regrowth_mid_chain(contexts):
    """S1, S1, S2, S2, S1, S1, S3, S3 on one context with overlap on, a snapshot after each call.  S2 has twice the
    lines of S1; S3 takes geom_lines_kernel.  Record buffers and flag arrays regrow under cudaDeviceSynchronize and the
    new flags are zeroed on the stream: parity, call numbers and the per-CTA epochs must survive that."""
    import torch
    ref_g = contexts()
    sets = {"S1": 600, "S2": 1200, "S3": 3000}             # x 16 lines x 211 bands, rows of 224
    assert 16 * sets["S2"] < by_line_threshold() <= 16 * sets["S3"]
    rigs = {s: Rig(ref_g, (M, 16, 211, 224, False, True, True, 0), {}, 1600 + 10 * i) for i, (s, M) in enumerate(sets.items())}
    order = ["S1", "S1", "S2", "S2", "S1", "S1", "S3", "S3"]
    g = contexts()
    g.set_overlap(True)
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()
    snaps = []
    with torch.cuda.stream(ts):
        for i, s in enumerate(order):
            rigs[s].call(g, i % K, stream=ts.cuda_stream)
            snaps.append(rigs[s].lay.snapshot())
    g.synchronize()
    torch.cuda.synchronize()
    for i, (s, snap) in enumerate(zip(order, snaps)):
        assert_bits(host_of(snap), rigs[s].want[i % K], "call %d (%s)" % (i + 1, s))


# ---- E. composite entry points --------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_composites_with_overlap(contexts):
    """gort_forward_batch and gort_jacobian_batch (with rsurf) give the same bits with overlap on as with it off:
    3000 members, 16 per-member geometries, 211 bands"""
    from test_dispatch_matrix_gpu import make_angles
    rng = np.random.Generator(np.random.PCG64(950))
    M, G = 3000, 16
    st = wk.random_structures(rng, M)
    leaf = wk.random_leaves(rng, M)
    soil = np.repeat(wk.DEFAULT_SOIL.reshape(4, 1), M, axis=1)
    wl = np.arange(400.0, 2500.0 + 0.5, 10.0)
    ang, _ = make_angles(rng, M, G, True)
    res = {}
    for on in (False, True):
        g = contexts()
        g.set_overlap(on)
        fwd = g.forward(st, leaf, soil, wl, ang)
        jac, rsurf = g.jacobian(st, leaf, soil, wl, ang, param=gort_b200.JAC_LAI, rel_step=H, want_rsurf=True)
        res[on] = dict(forward=fwd, again=g.forward(st, leaf, soil, wl, ang), jac=jac, rsurf=rsurf)
    assert np.isfinite(res[False]["forward"]).mean() > 0.9
    assert_bits(res[True], res[False], "overlap on")
    assert_bits(dict(again=res[True]["again"]), dict(again=res[False]["forward"]), "overlap on, repeated forward")
