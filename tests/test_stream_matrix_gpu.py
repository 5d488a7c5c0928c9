"""Consecutive calls on one context run one after the other, whatever streams they use (include/gort_b200.h).

The calls share the context's device scratch: the LUT plan, work lists, counters and per-zenith arrays, the energy
path's zenith records and the DFMA microbenchmark all live in one workspace, and the BRDF pipeline's record buffers
and flags are shared as well.  A call on another stream than the previous call's must therefore wait for the previous
call (order_after_previous, gort_abi.cu), and gort_synchronize() must wait for every call.

Every test enqueues a bounded spin (torch.cuda._sleep) on the first call's stream, then the first call A, then right
after it the second call B.  As soon as B is complete, A must be complete too.  The spin goes BEFORE A, so that an
unordered B runs and finishes during the spin and A then runs alone: no two workspace users ever run at the same time,
ordered or not.  Then the outputs of both calls must hold the bits of the same calls made alone.

Before a pair runs, A and B run alone twice at exactly its shapes: the first run gives the expected bits, and the two
runs grow every buffer the pair needs (the BRDF record buffers alternate by call parity).  A buffer that grew inside
the pair would wait for the whole device and order the calls for the wrong reason.

All tests use a context of this file's own, not the session context, so that what it last enqueued and how large its
buffers have grown is known here.  The inputs are 48 distinct crown shapes with 4 lines each, 7 and 211 bands.
"""
import math
import time

import numpy as np
import pytest
import torch

import gort_b200
from gort_b200 import workloads as wk
from test_chain_matrix_gpu import same_bits
from test_overlap_matrix_gpu import soil_from_table_dev

SENT = -7.0                          # what output buffers hold before a call
M, G, W_WIDE = 48, 4, 211            # crown shapes, lines per set, bands of the wide calls (7 MODIS bands otherwise)
SPIN_FACTOR, SPIN_MIN_MS = 20, 20.0  # the spin lasts at least 20 times the slowest solo B and at least 20 ms


def inputs():
    """host inputs: structure [6][M], leaf [7][M], soil [4][M], per-set angles [4][M][G], both band sets, soil table"""
    w = wk.c4_enkf(n_members=M, seed=2200, n_geom=G)
    rng = np.random.Generator(np.random.PCG64(2201))
    w["wl_wide"] = np.sort(rng.uniform(400.0, 2500.0, W_WIDE))
    w["table"] = 0.12 + 0.1 * np.sin(np.arange(gort_b200.SOIL_TABLE_NW) / 150.0)
    return w


def test_oracle_is_finite_on_these_inputs(oracle):
    """The GPU tests below require every solo result to be finite, so that two NaN arrays cannot pass as the same
    bits: the oracle gives finite values for every output of every set here."""
    x = inputs()
    st, leaf, soil, ang = x["structure"], x["leaf"], x["soil"], x["angles"]
    for m in range(M):
        arrays = {"lut q08": oracle.lut(st[:, m], 1)}
        rc, dead = oracle.lut_dead_rc(st[:, m])
        assert rc == 0, "set %d: the reference exits on this structure" % m
        arrays.update(("intermediates " + k, v) for k, v in dead.items())
        lut = arrays["lut full"] = oracle.lut(st[:, m], 0)
        a = ang[:, m, :].T
        for wl, tag in ((x["wavelength"], "narrow"), (x["wl_wide"], "wide")):
            sp = oracle.spectra(leaf[:, m], soil[:, m], wl)
            arrays.update(("spectra %s %d" % (tag, i), v) for i, v in enumerate(sp))
            arrays.update(("brdf %s %d" % (tag, i), v) for i, v in enumerate(oracle.brdf(st[:, m], lut, a, *sp)))
            arrays.update(("energy %s %d" % (tag, i), v) for i, v in enumerate(oracle.energy(st[:, m], lut, a, *sp)))
        for k, v in arrays.items():
            assert np.isfinite(v).all(), "set %d: %s" % (m, k)


# ---- the calls -------------------------------------------------------------------------------------------------------
class Rig:
    """the inputs on the host and on the GPU; LUTs and spectra made once by the context's own host calls"""

    def __init__(self, g):
        x = inputs()
        self.st, self.leaf, self.soil, self.ang = x["structure"], x["leaf"], x["soil"], x["angles"]
        self.wl7, self.wlw = x["wavelength"], x["wl_wide"]
        self.lut = g.lut(self.st)
        self.sp7 = g.spectra(self.leaf, self.soil, self.wl7)
        self.spw = g.spectra(self.leaf, self.soil, self.wlw)
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda:0"))
        self.d_st, self.d_lut, self.d_ang = d(self.st), d(self.lut), d(self.ang)
        self.d_leaf, self.d_soil, self.d_wlw, self.d_table = d(self.leaf), d(self.soil), d(self.wlw), d(x["table"])
        self.d_sp7 = [d(a) for a in self.sp7]
        self.d_spw = [d(a) for a in self.spw]


# name: (output shapes, enqueue(g, rig, outputs, stream))
DEV_CALLS = {
    "lut_full": (dict(lut=(M, gort_b200.LUT_STRIDE)),
                 lambda g, r, o, s: g.lut_dev(r.d_st, o["lut"], gort_b200.LUT_FULL, stream=s)),
    "lut_q08": (dict(lut=(M, gort_b200.LUT_STRIDE)),
                lambda g, r, o, s: g.lut_dev(r.d_st, o["lut"], gort_b200.LUT_Q08, stream=s)),
    "lut_scatter": (dict(lut=(M, gort_b200.LUT_STRIDE), further=(M, gort_b200.LUT_STRIDE)),
                    lambda g, r, o, s: g.lut_scatter_dev(r.d_st, o["lut"], [o["further"].data_ptr()], stream=s)),
    "lut_intermediates": (dict(vb=(M, 15), fb=(M, 15, gort_b200.NTH), t_open=(M, 15, 15), dt_open=(M, 15, 15),
                               dk_open=(M, 15), k_open=(M, 15)),
                          lambda g, r, o, s: g.lut_intermediates_dev(r.d_st, **o, stream=s)),
    "energy": (dict(albedo=(M, G, 7), favegt=(M, G, 7), fasoil=(M, G, 7)),
               lambda g, r, o, s: g.energy_dev(r.d_st, r.d_lut, r.d_ang, *r.d_sp7, o["albedo"], o["favegt"], o["fasoil"],
                                               stream=s)),
    "spectra": (dict(rleaf=(M, W_WIDE), tleaf=(M, W_WIDE), rsoil=(M, W_WIDE)),
                lambda g, r, o, s: g.spectra_dev(r.d_leaf, r.d_soil, r.d_wlw, o["rleaf"], o["tleaf"], o["rsoil"], stream=s)),
    "soil_from_table": (dict(rsoil=(M, W_WIDE)),
                        lambda g, r, o, s: soil_from_table_dev(g, r.d_table, r.d_wlw, o["rsoil"], stream=s)),
    # W < 64 (rsurf_flat_kernel), with the signatures and kprop; W >= 64 (a per-wavelength kernel)
    "brdf_narrow": (dict(rsurf=(M, G, 7), scomp=(M, G, 7, 4), kprop=(M, G, 4)),
                    lambda g, r, o, s: g.brdf_dev(r.d_st, r.d_lut, r.d_ang, *r.d_sp7, o["rsurf"], o["scomp"], o["kprop"],
                                                  stream=s)),
    "brdf_wide": (dict(rsurf=(M, G, W_WIDE)),
                  lambda g, r, o, s: g.brdf_dev(r.d_st, r.d_lut, r.d_ang, *r.d_spw, o["rsurf"], stream=s)),
}

# name: g, rig -> outputs
HOST_CALLS = {
    "lut": lambda g, r: dict(lut=g.lut(r.st)),
    "lut_intermediates": lambda g, r: g.lut_intermediates(r.st),
    "energy": lambda g, r: dict(zip(("albedo", "favegt", "fasoil"), g.energy(r.st, r.lut, r.ang, *r.sp7))),
    "brdf": lambda g, r: dict(rsurf=g.brdf(r.st, r.lut, r.ang, *r.spw)),
    "spectra": lambda g, r: dict(zip(("rleaf", "tleaf", "rsoil"), g.spectra(r.leaf, r.soil, r.wlw))),
    "forward": lambda g, r: dict(rsurf=g.forward(r.st, r.leaf, r.soil, r.wl7, r.ang)),
    "jacobian": lambda g, r: dict(jac=g.jacobian(r.st, r.leaf, r.soil, r.wl7, r.ang)),
    "dfma_peak": lambda g, r: dfma_peak(g),
}


def dfma_peak(g):
    """a workspace user whose result is a timing: nothing to compare"""
    g.dfma_peak_tflops()
    return {}

# a call is (where, name): where is "s1" / "s2" (caller streams), "ctx" (stream=None, the context's own stream),
# "host" (a host-pointer call) or "sync" (gort_synchronize alone)
FIRST = [("s1", n) for n in DEV_CALLS]
SECOND = ([("s2", n) for n in DEV_CALLS] + [("ctx", "lut_full"), ("ctx", "energy")] + [("host", n) for n in HOST_CALLS]
          + [("sync", None)])


def call_id(c):
    return c[0] if c[1] is None else "%s_%s" % c


class Env:
    def __init__(self, g):
        self.g = g
        self.rig = Rig(g)
        self.s = {"s1": torch.cuda.Stream(), "s2": torch.cuda.Stream(), "ctx": torch.cuda.ExternalStream(g.stream)}

    def prepare(self, c):
        """the call's outputs: sentinel-filled device tensors for a _dev call, an empty dict for the others"""
        where, name = c
        if where in self.s:
            return {k: torch.full(shape, SENT, dtype=torch.float64, device=torch.device("cuda:0"))
                    for k, shape in DEV_CALLS[name][0].items()}
        return {}

    def enqueue(self, c, out):
        where, name = c
        if where in self.s:
            DEV_CALLS[name][1](self.g, self.rig, out, None if where == "ctx" else self.s[where].cuda_stream)
        elif where == "host":
            out.update(HOST_CALLS[name](self.g, self.rig))
        else:
            self.g.synchronize()

    def complete(self, c):
        """wait for the call with nothing of the library: torch's synchronize of its stream (host-pointer calls and
        gort_synchronize are complete when they return)"""
        if c[0] in self.s:
            self.s[c[0]].synchronize()

    def host(self, c, out):
        return {k: v.cpu().numpy() for k, v in out.items()} if c[0] in self.s else out

    def solo(self, c):
        """the call alone, from a synchronised device -> its outputs on the host"""
        out = self.prepare(c)
        torch.cuda.synchronize()
        self.enqueue(c, out)
        self.complete(c)
        torch.cuda.synchronize()
        return self.host(c, out)

    def warm_up(self, calls):
        """each call alone, twice over -> the first outputs of each, which the second must repeat bit for bit.  Ends
        with gort_synchronize: the context has nothing pending and no previous stream."""
        first = [self.solo(c) for c in calls]
        again = [self.solo(c) for c in calls]
        for c, a, b in zip(calls, first, again):
            assert_same(b, a, "%s run alone twice" % call_id(c))
            for k, v in a.items():
                assert np.isfinite(v).all(), "%s alone: %s has %d non-finite values" % (call_id(c), k, (~np.isfinite(v)).sum())
        self.g.synchronize()
        torch.cuda.synchronize()
        return first

    def spin(self, where, cycles):
        with torch.cuda.stream(self.s[where]):
            torch.cuda._sleep(cycles)


def assert_same(got, want, what):
    assert sorted(got) == sorted(want), what
    for k in want:
        assert same_bits(got[k], want[k]), "%s: %s differs from the call made alone" % (what, k)


@pytest.fixture(scope="module")
def env():
    g = gort_b200.Gort(0)
    e = Env(g)
    yield e
    torch.cuda.synchronize()
    g.close()


@pytest.fixture(scope="module")
def cycles(env):
    """torch.cuda._sleep cycles for a spin of at least SPIN_FACTOR times the slowest solo B and SPIN_MIN_MS"""
    torch.cuda._sleep(1000)
    torch.cuda.synchronize()
    probe = 20_000_000
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(env.s["s1"]):
        e0.record()
        torch.cuda._sleep(probe)
        e1.record()
    e1.synchronize()
    ms_per_cycle = e0.elapsed_time(e1) / probe
    solo_ms = {}
    for c in SECOND:
        env.warm_up([c])
        out = env.prepare(c)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        env.enqueue(c, out)
        env.complete(c)
        solo_ms[call_id(c)] = (time.perf_counter() - t0) * 1e3
    slowest = max(solo_ms, key=solo_ms.get)
    spin_ms = max(SPIN_FACTOR * solo_ms[slowest], SPIN_MIN_MS)
    n = int(math.ceil(spin_ms / ms_per_cycle))
    print("\nspin: %.4f ms per million cycles (%s)" % (ms_per_cycle * 1e6, torch.cuda.get_device_name(0)))
    print("solo B, issue to completion on the host [ms]: " + ", ".join("%s %.3f" % kv for kv in solo_ms.items()))
    print("slowest solo B: %s, %.3f ms -> spin of %d cycles, %.1f ms" % (slowest, solo_ms[slowest], n, n * ms_per_cycle))
    return n


def run_ordered(env, cycles, calls, watch):
    """the spin on calls[0]'s stream, then every call; as soon as the last one is complete -> (the watched stream has
    nothing left, the outputs of every call)"""
    outs = [env.prepare(c) for c in calls]
    torch.cuda.synchronize()
    try:
        env.spin(calls[0][0], cycles)
        for c, o in zip(calls, outs):
            env.enqueue(c, o)
        env.complete(calls[-1])
        done = env.s[watch].query()
    finally:
        torch.cuda.synchronize()
    return done, [env.host(c, o) for c, o in zip(calls, outs)]


# ---- pairs: A on a caller stream, then B ----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("b", SECOND, ids=call_id)
@pytest.mark.parametrize("a", FIRST, ids=call_id)
def test_pair(env, cycles, a, b):
    want = env.warm_up([a, b])
    done, got = run_ordered(env, cycles, [a, b], "s1")
    assert_same(got[0], want[0], "A = %s, followed by %s" % (call_id(a), call_id(b)))
    assert_same(got[1], want[1], "B = %s, after %s" % (call_id(b), call_id(a)))
    assert done, "%s was complete while %s on s1 was still pending: it was not ordered after it" % (call_id(b), call_id(a))


# ---- sequences ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_return_to_stream(env, cycles):
    """A on s1, B on s2, C back on s1: C waits for B, so C's completion implies B's"""
    calls = [("s1", "lut_full"), ("s2", "energy"), ("s1", "lut_intermediates")]
    want = env.warm_up(calls)
    done, got = run_ordered(env, cycles, calls, "s2")
    for c, o, w in zip(calls, got, want):
        assert_same(o, w, "%s in A, B, C" % call_id(c))
    assert done, "C on s1 was complete while B on s2 was still pending"
    assert env.s["s1"].query()


@pytest.mark.gpu
@pytest.mark.parametrize("b", [("s2", "lut_q08"), ("s2", "energy"), ("s2", "brdf_narrow")], ids=call_id)
@pytest.mark.parametrize("a", [("ctx", "lut_full"), ("ctx", "brdf_wide")], ids=call_id)
def test_context_stream_then_caller_stream(env, cycles, a, b):
    """the spin and A on the context's own stream, B on a caller stream"""
    want = env.warm_up([a, b])
    done, got = run_ordered(env, cycles, [a, b], "ctx")
    assert_same(got[0], want[0], "A = %s" % call_id(a))
    assert_same(got[1], want[1], "B = %s" % call_id(b))
    assert done, "%s was complete while %s on the context's stream was still pending" % (call_id(b), call_id(a))
