"""The gap-probability LUT kernels (gort_b200/csrc/gort_lut.cu) on the paths the workload tests leave unchecked,
organised by kernel path.  Every case (1) asserts on the CPU that its inputs reach the path (lut_catalogue.py; the
same assertions run without a GPU in test_lut_matrix_cpu.py), (2) compares with the oracle, strictly to 1e-9 and
conditioning-aware only where that misses, and (3) checks that every set's row has the bits of the set computed
alone.  Bit equality catches a merge of two crown shapes or stem densities that differ by 1 ULP, which the oracle
cannot see.

  beyond_table   oblate crowns whose crown-count loop reaches bins beyond the 512-bin exp table: the redo loop's
                 direct formula, with each member's own favd, in lut_crown_kernel<1> and <8>
  thin_layer     K = 0 (lut_vg_kernel's literal proj_volume fallback) and K = 1 midpoints, full and Q08 methods
  plan           one batch through every branch of lut_plan_kernel's group and sub-group assignment, and the same
                 batch behind 1 .. 63 leading sets (another partition)
  passes         shape and lambda runs across the pass boundary of gort_lut (16 384 sets) and of
                 gort_lut_intermediates (8 192 sets), with a ragged last pass
  intermediates  gort_lut_intermediates (launch_lut_dead) on the oblate, thin and plan catalogues, and on sets where
                 the reference exits on a negative sphere volume (vb must be NaN exactly there)
"""
import numpy as np
import pytest

import lut_catalogue as lc
from checkers import DEAD_KEYS, assert_close_cond, check_set, rel_err, sensitivity

pytestmark = pytest.mark.gpu
FULL, Q08 = 0, 1

_alone = {}


def alone(gort, st6, method=FULL):
    key = (np.asarray(st6, dtype=np.float64).tobytes(), method)
    if key not in _alone:
        _alone[key] = gort.lut(np.ascontiguousarray(np.asarray(st6, dtype=np.float64).reshape(6, 1)), method)[0]
    return _alone[key]


def assert_rows_alone(gort, st, lut, idx, what, method=FULL):
    for m in idx:
        a = alone(gort, st[:, m], method)
        assert np.array_equal(lut[m], a, equal_nan=True), "%s: set %d %r differs from the set computed alone (%d entries)" % (
            what, m, st[:, m], int(np.sum(~((lut[m] == a) | (np.isnan(lut[m]) & np.isnan(a))))))


def assert_oracle(oracle, st, lut, idx, what, method=FULL):
    """strict 1e-9 first; sensitivity() only for a set that misses it"""
    excused = 0
    for m in idx:
        want = oracle.lut(st[:, m], method)
        try:
            if rel_err(lut[m], want) <= 1e-9:
                continue
        except AssertionError:
            pass                                          # NaN positions differ: let assert_close_cond report it
        sens = sensitivity(lambda c: c.lut(st[:, m], method), want)
        excused += assert_close_cond(lut[m], want, sens, "%s: set %d %r" % (what, m, st[:, m]))[1]
    return excused


# ---- beyond_table ---------------------------------------------------------------------------------------------------
def _assert_beyond_table(oracle, st):
    for m in range(st.shape[1]):
        nt = lc.n_tab(st[:, m])
        assert int(oracle.lut_bins(st[:, m]).max()) >= nt, "set %d stays inside the %d-bin table" % (m, nt)


def test_beyond_table_single(gort, oracle):
    st = lc.beyond_table_singles()
    _assert_beyond_table(oracle, st)
    assert np.all(lc.plan(st)[1] == 1)
    lut = gort.lut(st)
    assert np.isfinite(lut).all()
    assert_oracle(oracle, st, lut, range(st.shape[1]), "beyond_table single")
    assert_rows_alone(gort, st, lut, range(st.shape[1]), "beyond_table single")


def test_beyond_table_subgroups(gort, oracle):
    st = lc.beyond_table_subgroups()
    _assert_beyond_table(oracle, st)
    groups = lc.sub_groups(lc.plan(st)[1])
    assert sorted(s for _, s in groups) == list(range(2, lc.LUT_SUB + 1))
    lut = gort.lut(st)
    assert np.isfinite(lut).all()
    assert_oracle(oracle, st, lut, range(st.shape[1]), "beyond_table sub-group member")
    assert_rows_alone(gort, st, lut, range(st.shape[1]), "beyond_table sub-group member")
    # the members differ only in favd: their epgap rows must differ from the head's
    for e, s in groups:
        for j in range(1, s):
            assert not np.array_equal(lut[e + j, 91:182], lut[e, 91:182])


# ---- thin_layer -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", [FULL, Q08], ids=["full", "q08"])
def test_thin_layer(gort, oracle, method):
    st, K = lc.thin_layers()
    assert np.array_equal(K, [lc.midpoints_k(st[:, m]) for m in range(st.shape[1])])
    assert (K == 0).any() and (K == 1).any()
    lut = gort.lut(st, method)
    assert_oracle(oracle, st, lut, range(st.shape[1]), "thin_layer K=%s" % K.tolist(), method)
    assert_rows_alone(gort, st, lut, range(st.shape[1]), "thin_layer", method)
    if method == FULL:
        assert np.all(lut[K == 0, :91] == 1.0)           # K = 0: v_g = 0, so p_n0 = 1 exactly


# ---- plan -----------------------------------------------------------------------------------------------------------
def test_plan(gort, oracle):
    st, notes = lc.plan_batch()
    n = st.shape[1]
    head, sub = lc.plan(st)
    groups = lc.sub_groups(sub)
    assert {s for _, s in groups} == set(range(1, lc.LUT_SUB + 1))
    cap_cuts = [e for e in range(lc.GROUP_CAP, n, lc.GROUP_CAP) if lc._same_shape(st, e, e - 1) and st[0, e] == st[0, e - 1]]
    assert cap_cuts
    lut = gort.lut(st)
    assert_rows_alone(gort, st, lut, range(n), "plan batch")
    for k in (1, 17, 40, 63):
        sh = lc.shifted(st, k)
        assert lc.sub_groups(lc.plan(sh)[1][k:]) != groups
        lut_k = gort.lut(sh)
        bad = np.flatnonzero(~np.all((lut_k[k:] == lut) | (np.isnan(lut_k[k:]) & np.isnan(lut)), axis=1))
        assert bad.size == 0, "plan batch behind %d leading sets: sets %s change bits" % (k, bad[:10].tolist())
    heads = [e for e in range(n) if head[e] == e]
    lasts = [e + s - 1 for e, s in groups]
    ulps = [e for e, _, how in notes["pairs"] if how == "ulp"] + [e - 1 for e, _, how in notes["pairs"] if how == "ulp"]
    idx = sorted(set(heads) | set(lasts) | set(ulps))
    assert_oracle(oracle, st, lut, idx, "plan batch")


# ---- passes ---------------------------------------------------------------------------------------------------------
def test_passes_lut(gort, oracle):
    P, extra = lc.LUT_CHUNK, 100
    st = lc.passes_batch(P, extra)
    assert np.all(st[:5, P - 41:P + 59] == st[:5, P - 41:P - 40])
    lut = gort.lut(st)
    near = list(range(P - 70, P + 70)) + list(range(P + extra - 8, P + extra))
    assert_rows_alone(gort, st, lut, near, "gort_lut pass boundary")
    assert_oracle(oracle, st, lut, [0, 4097, P - 41, P - 1, P, P + 58, P + extra - 1], "gort_lut passes")


def test_passes_intermediates(gort, oracle):
    P, extra = lc.DEAD_CHUNK, 37
    st = lc.passes_batch(P, extra)
    assert np.all(st[:5, P - 41:P + 59] == st[:5, P - 41:P - 40])
    got = gort.lut_intermediates(st)
    for m in list(range(P - 66, P + 3)) + [P + extra - 1]:
        one = gort.lut_intermediates(np.ascontiguousarray(st[:, m:m + 1]))
        for q in DEAD_KEYS:
            assert np.array_equal(got[q][m], one[q][0], equal_nan=True), "%s of set %d differs when computed alone" % (q, m)
    for m in (P - 1, P, P + extra - 1):
        check_set({q: got[q][m] for q in DEAD_KEYS}, st[:, m], oracle, "intermediates passes, set %d" % m)


# ---- intermediates --------------------------------------------------------------------------------------------------
def test_intermediates_catalogues(gort, oracle):
    thin, K = lc.thin_layers()
    plan_st, _ = lc.plan_batch()
    head, sub = lc.plan(plan_st)
    plan_idx = [e for e in range(plan_st.shape[1]) if head[e] == e][::6]
    exits = lc.vb_exit_sets()
    st = np.ascontiguousarray(np.concatenate([lc.beyond_table_singles()[:, ::4], exits[:, :1], lc.beyond_table_subgroups()[:, ::9],
                                              thin[:, ::3], plan_st[:, plan_idx], exits[:, 1:]], axis=1))
    got = gort.lut_intermediates(st)
    n_exit = 0
    for m in range(st.shape[1]):
        rc, _ = oracle.lut_dead_rc(st[:, m])
        gpu_exit = bool(np.isnan(got["vb"][m]).any())
        assert gpu_exit == (rc != 0), "set %d %r: oracle exit %d, GPU vb %r" % (m, st[:, m], rc, got["vb"][m])
        if rc:                                            # the reference exits: nothing else to compare
            n_exit += 1
            continue
        check_set({q: got[q][m] for q in DEAD_KEYS}, st[:, m], oracle, "intermediates set %d %r" % (m, st[:, m]))
    assert n_exit == exits.shape[1]
