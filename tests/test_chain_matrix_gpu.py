"""gort_jacobian_batch and gort_forward_batch (gort_abi.cu) by path: every parameter under both LUT methods, shared and
per-member geometry, the user_leaf / user_soil overrides, the canopy options, the default step, more than one member
chunk, and the forward operator's chunk cap.

The Jacobian is checked bit for bit against (F(st+) - F(st-)) / (2 h p) formed in numpy from gort.forward: the
perturbed structures, the difference and the quotient are products, one subtraction and one IEEE division with no
contraction (csrc/Makefile: -fmad=false), and LUT and BRDF results do not depend on batch composition
(test_lut_matrix_gpu.py, test_dispatch_matrix_gpu.py).  The forward side is tied to the oracle separately, for the
parameters the older Jacobian test does not reach (jacobian_oracle_link)."""
import numpy as np
import pytest

import gort_b200
from gort_b200 import workloads as wk
import spectra_catalogue as sc
from checkers import assert_close, assert_close_cond, sensitivity

pytestmark = pytest.mark.gpu

H = 1e-4
PARAMS = [("lambda", gort_b200.JAC_LAMBDA), ("r", gort_b200.JAC_R), ("b", gort_b200.JAC_B), ("h1", gort_b200.JAC_H1),
          ("h2", gort_b200.JAC_H2), ("favd", gort_b200.JAC_FAVD), ("lai", gort_b200.JAC_LAI)]
METHODS = [("full", gort_b200.LUT_FULL), ("q08", gort_b200.LUT_Q08)]


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True) and np.array_equal(np.signbit(a), np.signbit(b))


def identity(gort, st, param, h, leaf, soil, wl, ang, method, **kw):
    """(F(st+) - F(st-)) / (2 h p) with st+-[row] = st[row] * (1 +- h); p as jac_diff_kernel forms it"""
    row = 5 if param == gort_b200.JAC_LAI else param
    sp, sm = st.copy(), st.copy()
    sp[row] = st[row] * (1.0 + h)
    sm[row] = st[row] * (1.0 - h)
    fp = gort.forward(sp, leaf, soil, wl, ang, method=method, **kw)
    fm = gort.forward(sm, leaf, soil, wl, ang, method=method, **kw)
    p = st[row]
    if param == gort_b200.JAC_LAI:
        p = st[5] * (st[0] * st[1] * st[1] * np.pi * st[2] * 4.0) / 3.0
    return (fp - fm) / (2.0 * h * p)[:, None, None]


def _members(n, seed, n_geom):
    w = wk.c4_enkf(n_members=n, seed=seed, n_geom=n_geom)
    return w["structure"], w["leaf"], w["soil"], w["wavelength"], w["angles"]


@pytest.mark.parametrize("mname,method", METHODS)
@pytest.mark.parametrize("pname,param", PARAMS)
def test_jacobian_identity(gort, pname, param, mname, method):
    st, leaf, soil, wl, ang = _members(6, 900 + param, 5)
    variants = [
        ("member geometry", dict(leaf=leaf, soil=soil, ang=ang, kw={})),
        ("shared geometry, user_leaf, beta + fd", dict(leaf=None, soil=soil, ang=np.ascontiguousarray(ang[:, 0, :]),
                                                       kw=dict(user_leaf=0.41, beta=0.3, fd=0.7))),
        ("member geometry, user_soil", dict(leaf=leaf, soil=None, ang=ang, kw=dict(user_soil=0.13))),
        ("shared geometry, both overrides", dict(leaf=None, soil=None, ang=np.ascontiguousarray(ang[:, 0, :]),
                                                 kw=dict(user_leaf=0.41, user_soil=0.13))),
    ]
    for what, v in variants:
        args = (st, v["leaf"], v["soil"], wl, v["ang"])
        jac0, rsurf = gort.jacobian(*args, param=param, rel_step=0.0, method=method, want_rsurf=True, **v["kw"])
        jac1 = gort.jacobian(*args, param=param, rel_step=H, method=method, **v["kw"])
        assert same_bits(jac0, jac1), "%s: rel_step 0 is not the 1e-4 default" % what
        assert same_bits(rsurf, gort.forward(*args, method=method, **v["kw"])), "%s: rsurf != F(st)" % what
        want = identity(gort, st, param, H, v["leaf"], v["soil"], wl, v["ang"], method, **v["kw"])
        assert np.isfinite(want).mean() > 0.5, what
        bad = ~((jac0 == want) | (np.isnan(jac0) & np.isnan(want)))
        assert same_bits(jac0, want), "%s: %d entries differ from the difference quotient of gort.forward" % (what, bad.sum())


def test_jacobian_chunks(gort):
    """two member chunks, the last one ragged: the second pass's inputs and per-member angles start at member 998"""
    M, G = 998 + 41, 16
    wl = np.arange(400.0, 2501.0)
    st, leaf, soil, _, ang = _members(M, 77, G)
    C = sc.jac_chunk(M, G, wl.shape[0])
    assert C == 998 and sc.n_chunks(M, C) == 2
    assert not np.array_equal(ang[:, C - 41:C], ang[:, C:])          # a wrong angle offset is visible
    jac = gort.jacobian(st, leaf, soil, wl, ang, param=gort_b200.JAC_LAI)
    want = identity(gort, st, gort_b200.JAC_LAI, H, leaf, soil, wl, ang, gort_b200.LUT_FULL)
    assert np.isfinite(want[C:]).mean() > 0.5
    assert same_bits(jac[:C], want[:C]), "first chunk"
    assert same_bits(jac[C:], want[C:]), "second chunk"


def _oracle_chain(c, st6, leaf7, soil4, wl, ang4g):
    lut = c.lut(st6)
    rl, tl, rs = c.spectra(leaf7, soil4, wl)
    return c.brdf(st6, lut, ang4g, rl, tl, rs, want_scomp=False)[0]


@pytest.mark.parametrize("pname,param", PARAMS[1:5])
def test_jacobian_oracle_link(gort, oracle, pname, param):
    """F(st+-) of gort.forward against the oracle chain at st+-.  The quotient is not compared: in r, b, h1 and h2 the
    chain is only piecewise smooth (crown-count histogram bins), and a bin that flips in one chain and not the other,
    divided by 2h, is not a kernel error."""
    st, leaf, soil, wl, ang = _members(8, 300 + param, 4)
    excused = 0
    for side in (1.0 + H, 1.0 - H):
        s = st.copy()
        s[param] = st[param] * side
        f = gort.forward(s, leaf, soil, wl, ang)
        for m in range(8):
            a = np.ascontiguousarray(ang[:, m, :].T)
            want = _oracle_chain(oracle, s[:, m].copy(), leaf[:, m], soil[:, m], wl, a)
            try:
                assert_close(f[m], want, "%s member %d" % (pname, m))
            except AssertionError:
                sens = sensitivity(lambda c: _oracle_chain(c, s[:, m].copy(), leaf[:, m], soil[:, m], wl, a), want)
                excused += assert_close_cond(f[m], want, sens, "%s member %d" % (pname, m))[1]
    print("%s: %d entries excused by conditioning" % (pname, excused))


def test_forward_cap(gort):
    """131 073 members: the chunk is capped at 16 384, 9 chunks, the last of one member"""
    M = 131073
    st, leaf, soil, wl, ang = _members(M, 55, 16)
    ang = np.ascontiguousarray(ang[:, 0, :])
    C = sc.forward_chunk(M)
    assert C == 16384 and sc.n_chunks(M, C) == 9 and M - 8 * C == 1
    lut = gort.lut(st)
    rl, tl, rs = gort.spectra(leaf, soil, wl)
    want = gort.brdf(st, lut, ang, rl, tl, rs)
    assert same_bits(gort.forward(st, leaf, soil, wl, ang), want)
    rl, tl, rs = gort.spectra(leaf, None, wl, user_soil=0.13)
    want = gort.brdf(st, lut, ang, rl, tl, rs)
    assert same_bits(gort.forward(st, leaf, None, wl, ang, user_soil=0.13), want)
