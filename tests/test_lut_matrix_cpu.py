"""The inputs of test_lut_matrix_gpu.py reach the LUT kernel paths each case is named for.  Checked here, without a GPU,
with the oracle's crown-count bins (gort_oracle_lut_bins) and the restatements in lut_catalogue.py."""
import numpy as np

import lut_catalogue as lc


def _bins(oracle, st):
    return np.array([int(oracle.lut_bins(st[:, m]).max()) for m in range(st.shape[1])])


def test_lut_bins_helper(oracle):
    st = np.array([0.1, 1.0, 2.0, 3.0, 8.0, 0.8])
    u = oracle.lut_bins(st)
    assert u[-1] == 0.0 and np.all(u[:-1] >= 0.5)
    # the path s is below s' <= (z2' - height_p[0]) / cos(theta'): the bins stay inside the reference's histogram
    inter = oracle.lut_intermediates(st)
    s_max = (inter["derived"][13] - inter["height_p"][0]) / np.cos(inter["theta_p"][:-1]) / inter["derived"][8] + 0.5
    assert np.all(u[:-1] <= s_max)
    # C3-range crowns stay inside the table
    assert int(u.max()) < lc.n_tab(st) - 1


def test_beyond_table_reached(oracle):
    for st in (lc.beyond_table_singles(), lc.beyond_table_subgroups()):
        nt = np.array([lc.n_tab(st[:, m]) for m in range(st.shape[1])])
        assert np.all(nt == lc.LUT_TAB)
        bins = _bins(oracle, st)
        assert np.all(bins >= nt), "sets %s stay inside the table" % np.flatnonzero(bins < nt)
    _, sub = lc.plan(lc.beyond_table_singles())
    assert np.all(sub == 1)                                   # crown<1> only
    _, sub = lc.plan(lc.beyond_table_subgroups())
    sizes = [s for _, s in lc.sub_groups(sub)]
    assert sorted(sizes) == [2, 3, 4, 5, 6, 7, 8]             # crown<8> with every member count but one
    st = lc.beyond_table_subgroups()
    for e, s in lc.sub_groups(sub):
        assert len(set(st[5, e:e + s])) == s                  # every member its own favd


def test_thin_layers_reached(oracle):
    st, K = lc.thin_layers()
    assert set(K.tolist()) >= {0, 1}
    assert (K == 0).sum() >= 8 and (K == 1).sum() >= 8
    for m in range(st.shape[1]):
        vg = oracle.lut_intermediates(st[:, m])["v_g"]
        assert (K[m] == 0) == (not vg.any()), m               # K = 0: the midpoint rule has no point, v_g = 0
        dh, edge = st[4, m] - st[3, m], 2 * st[2, m] / 27
        if abs(dh - edge) > 1e-9 * edge:                        # away from the boundary, K = 0 <=> h2 - h1 < 2b/27
            assert (dh < edge) == (K[m] == 0), m
    # K changes between the two floats at each boundary
    steps = [(K[m], K[m + 1]) for m in range(st.shape[1] - 1)]
    assert (0, 1) in steps and (1, 2) in steps


def _runs(v):
    """[(start, length)] of runs of equal values"""
    cut = np.flatnonzero(np.diff(v) != 0) + 1
    edges = np.concatenate([[0], cut, [len(v)]])
    return [(int(a), int(b - a)) for a, b in zip(edges[:-1], edges[1:])]


def _shape_ids(st):
    _, inv = np.unique(st[1:5].T, axis=0, return_inverse=True)
    return inv.ravel()


def test_plan_batch_reaches_every_branch():
    st, notes = lc.plan_batch()
    n = st.shape[1]
    for k in (0, 1, 17, 63):
        s = lc.shifted(st, k) if k else st
        head, sub = lc.plan(s)
        sizes = {sz for e, sz in lc.sub_groups(sub) if e >= k}
        assert sizes == set(range(1, lc.LUT_SUB + 1)), (k, sizes)
        # every set in exactly one sub-group, inside its group
        owner = np.full(s.shape[1], -1)
        for e, sz in lc.sub_groups(sub):
            assert np.all(owner[e:e + sz] == -1)
            owner[e:e + sz] = e
            assert np.all(head[e:e + sz] == head[e])
        assert np.all(owner >= 0)
        # the 64-cap cuts a shape run and a lambda run (of one shape) of this batch
        ids, lam = _shape_ids(s), s[0]
        cuts = [e for e in range(lc.GROUP_CAP, s.shape[1], lc.GROUP_CAP) if ids[e] == ids[e - 1]]
        assert cuts and any(lam[e] == lam[e - 1] for e in cuts), k
        # lambda runs cut at 8 inside a group
        assert any(sub[e] == lc.LUT_SUB and e + 8 < s.shape[1] and sub[e + 8] > 0 and lam[e + 8] == lam[e] and
                   head[e + 8] == head[e] for e in range(s.shape[1]))
    # the shifts give different partitions
    parts = {tuple(lc.sub_groups(lc.plan(lc.shifted(st, k) if k else st)[1][k:] if k else lc.plan(st)[1]))
             for k in (0, 1, 17, 63)}
    assert len(parts) == 4
    # shape runs longer than 64 starting at odd offsets
    long_runs = [(a, L) for a, L in _runs(_shape_ids(st)) if L > lc.GROUP_CAP]
    assert len(long_runs) >= 2 and all(a % 2 == 1 for a, _ in long_runs)
    # lambda runs of every length 1 .. 17 inside one shape run
    a, L = long_runs[0]
    assert sorted(L2 for _, L2 in _runs(st[0, a:a + L])) == list(range(1, 18))
    # neighbours differing in exactly one field, by a step and by one ULP
    for e, field, how in notes["pairs"]:
        diff = np.flatnonzero(st[:, e] != st[:, e - 1])
        assert diff.tolist() == [lc.FIELDS.index(field)]
        if how == "ulp":
            assert np.nextafter(st[diff[0], e - 1], np.inf) == st[diff[0], e]
    assert {(f, h) for _, f, h in notes["pairs"]} == {(f, h) for f in lc.FIELDS for h in ("step", "ulp")}
    # A-B-A: a shape (and a lambda inside one shape) that returns after one other
    ids = _shape_ids(st)
    assert any(ids[e] == ids[e + 2] != ids[e + 1] for e in range(n - 2))
    assert any(ids[e] == ids[e + 1] == ids[e + 2] and st[0, e] == st[0, e + 2] != st[0, e + 1] for e in range(n - 2))


def test_passes_batches_straddle():
    for n_pass, extra in ((lc.LUT_CHUNK, 100), (lc.DEAD_CHUNK, 37)):
        st = lc.passes_batch(n_pass, extra)
        assert st.shape[1] == n_pass + extra
        # one shape and one lambda across the pass boundary, from 41 sets before it to 58 after (or the last set)
        w = st[:5, n_pass - 41:n_pass + 59]
        assert np.all(w == w[:, :1])
        assert not np.array_equal(st[:5, n_pass - 42], st[:5, n_pass - 41])
        head, sub = lc.plan(np.ascontiguousarray(st[:, n_pass - 128:]), chunk=128)   # the same cuts: 128 = 2 caps
        assert sub[128] > 0 and head[128] == 0                                          # the pass boundary cuts the run


def test_vb_exit_sets(oracle):
    st = lc.vb_exit_sets()
    assert all(oracle.lut_dead_rc(st[:, m])[0] == 1 for m in range(st.shape[1]))
    thin, _ = lc.thin_layers()
    assert all(oracle.lut_dead_rc(thin[:, m])[0] == 0 for m in range(0, thin.shape[1], 4))
