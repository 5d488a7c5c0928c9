"""The inputs of test_spectra_matrix_gpu.py reach the PROSPECT-D and Price soil paths each case is named for, checked
here without a GPU with the restatements in spectra_catalogue.py.  The oracle is also held to the independent numpy
restatement of test_prospect_independent_cpu.py on the whole edge catalogue, uninterpolated."""
import numpy as np

import spectra_catalogue as sc
from test_prospect_independent_cpu import prospect_db

SOIL = np.array([0.2, 0.1, 0.03726, -0.002426])


def test_k_matches_the_oracle_branch(oracle):
    # k > 85 gives tau = 0 and t = 0: those rows are NaN for N > 1 (b = inf, Rsub = inf / inf) and have tran = 0 for
    # N = 1 (pow(inf, 0) = 1); every other row has 0 < tran < 1
    for leaf in sc.k_branches().T:
        k = sc.k_rows(leaf)
        _, t = oracle.prospect_full(leaf)
        if leaf[0] == 1.0:
            assert np.all(t[k > 85.0] == 0.0)
        else:
            assert np.all(np.isnan(t[k > 85.0]))
        assert np.all((t[k <= 85.0] > 0.0) & (t[k <= 85.0] < 1.0))


def test_k_branches_reached():
    L = sc.k_branches()
    seen = {}
    for leaf in L.T:
        counts = np.bincount(sc.tau_branch(sc.k_rows(leaf)), minlength=4)
        seen.setdefault(leaf[0], np.zeros(4, int))
        seen[leaf[0]] += counts
        if not leaf[1:].any():
            assert counts[0] == sc.NW                                   # transparent: k = 0 on every row
        elif not leaf[5:].any():
            assert counts[0] >= 1000 and counts[1] >= 500               # pigments only: k = 0 beyond the pigment bands
    assert set(seen) == {1.0, 1.5, 2.5}
    for N, c in seen.items():
        assert np.all(c[:3] >= 50), (N, c)                             # k <= 0, (0, 4], (4, 85] on many rows
        if N != 2.5:
            assert c[3] >= 20, (N, c)                                  # k > 85 for N = 1 and for N = 1.5


def test_k_boundaries_exact():
    L, rows = sc.k_boundaries()
    assert L.shape == (7, 6)
    k = np.array([sc.k_rows(L[:, j])[rows[j]] for j in range(6)])
    for j, edge in ((0, 4.0), (3, 85.0)):
        assert k[j] == np.nextafter(edge, 0.0) and k[j + 1] == edge and k[j + 2] == np.nextafter(edge, np.inf)
    assert sc.tau_branch(k).tolist() == [1, 1, 2, 2, 2, 3]
    assert np.all(L[1:] == L[1:, :1])                                  # only N differs
    assert np.all((L[0] >= 1.0) & (L[0] <= 2.0))


def test_nan_edge_reached(oracle):
    L, wls = sc.nan_edge()
    expect = {0: (1518, 1917.0), 1: None}
    for m in range(L.shape[1]):
        k = sc.k_rows(L[:, m])
        runs = sc.k_runs(k > 85.0)
        assert runs, m
        refl, tran = oracle.prospect_full(L[:, m])
        assert L[0, m] > 1.0
        # every k > 85 row is NaN for N > 1, every other row finite
        assert np.array_equal(np.isnan(refl), k > 85.0) and np.array_equal(np.isnan(tran), k > 85.0)
        lower, upper, f = sc.leaf_index(wls[m])
        assert np.all(f[0::2] == 0.0) and np.all(f[1::2] == 0.5)
        assert np.all(~np.isnan(refl[lower])) and np.all(np.isnan(refl[upper]))
        rl, tl, _ = oracle.spectra(L[:, m], SOIL, wls[m])
        assert np.isnan(rl).all() and np.isnan(tl).all()
        if expect[m]:
            assert runs[0][0] == expect[m][0] and wls[m][0] == expect[m][1]
    # N = 1: pow(inf, 0) = 1, the k > 85 rows stay finite
    wet1 = sc.k_branches()[:, 3]
    assert wet1[0] == 1.0 and (sc.k_rows(wet1) > 85.0).any()
    assert np.isfinite(oracle.prospect_full(wet1)[0]).all()


def test_wavelength_catalogue():
    lo, hi, f = sc.leaf_index(sc.wl_ends())
    assert lo.tolist() == [0, 0, 2099, 2100] and hi.tolist() == [1, 1, 2100, 2101]
    assert f[0] == 0.0 and f[3] == 0.0 and 0.0 < f[1] < 1e-6 and f[2] == 1.0      # (float)(2100 - 1 ULP) == 2100
    lo, hi, f = sc.leaf_index(sc.wl_integers())
    assert np.all(f == 0.0) and np.all(hi == lo + 1)
    w1 = sc.wl_fraction_one()
    lo, hi, f = sc.leaf_index(w1)
    assert len(w1) > 200 and np.all(f == np.float32(1.0)) and np.all(np.float32(1) - f == 0.0)
    assert np.all(lo == np.round(w1 - 400.0) - 1)
    wf = sc.wl_float_fraction(np.random.Generator(np.random.PCG64(7)))
    lo, _, f = sc.leaf_index(wf)
    assert len(wf) == 64 and np.all(np.abs(f - ((wf - 400.0) - lo)) > 1e-6)
    all_wl = sc.wavelengths()
    assert np.all((all_wl >= sc.WL_MIN) & (all_wl <= sc.WL_MAX))


def test_soil_indices():
    nodes = sc.wl_soil_nodes()
    n = (len(nodes) + 1) // 2
    lo, hi, f = sc.soil_index(nodes[:n])
    assert np.all(f == 0.0) and np.all(lo == (nodes[:n] - 400.0) / 5.0)
    assert hi[-1] == sc.SOIL_NW                                        # 2500 nm: the upper node is one past the table
    lo, hi, f = sc.soil_index(nodes[n:])
    assert np.all(lo == np.round((nodes[n:] - 400.0) / 5.0) - 1) and np.all((f > 0.999) & (f < 1.0))


def test_chunk_formulas():
    assert sc.jac_chunk(998 + 41, 16, 2101) == 998
    assert sc.n_chunks(998 + 41, sc.jac_chunk(998 + 41, 16, 2101)) == 2
    assert sc.jac_chunk(10 ** 6, 16, 211) == 9939 and sc.jac_chunk(3000, 16, 211) == 3000    # one pass at 3000 x 16 x 211
    assert sc.forward_chunk(131073) == 16384 and sc.n_chunks(131073, 16384) == 9
    assert 131073 - 8 * 16384 == 1


def test_oracle_against_independent_restatement(oracle):
    """oracle/prospect_d_oracle.c against prospect_db on every row of every edge leaf: 1e-11, NaN positions equal.
    k = 0 rows of N != 1 leaves have r + t within an ULP of 1, where the two restatements may take different branches
    (the Stokes formula and the zero-absorption limit differ by up to 2e-8 there): 1e-7, counted.  For N = 1 the two
    branches agree exactly and those rows stay strict."""
    T = sc.tables()
    leaves = np.concatenate([sc.k_branches(), sc.k_boundaries()[0], sc.nan_edge()[0]], axis=1)
    loose = worst = 0
    for leaf in leaves.T:
        k = sc.k_rows(leaf)
        want = oracle.prospect_full(leaf)
        with np.errstate(all="ignore"):
            got = prospect_db(T, *leaf)
        for x, y in zip(got, want):
            assert np.array_equal(np.isnan(x), np.isnan(y)), leaf
            ok = ~np.isnan(y)
            rel = np.zeros(sc.NW)
            rel[ok] = np.abs(x[ok] - y[ok]) / np.maximum(np.abs(y[ok]), 1e-12)
            ill = (k == 0.0) & (leaf[0] != 1.0)
            assert np.all(rel[~ill] <= 1e-11), (leaf, rel[~ill].max())
            assert np.all(rel[ill] <= 1e-7), (leaf, rel[ill].max())
            loose += int((rel[ill] > 1e-11).sum())
            worst = max(worst, rel[~ill].max(initial=0.0))
    print("oracle vs numpy restatement: worst strict rel %.3e, %d k = 0 entries (N != 1) between 1e-11 and 1e-7"
          % (worst, loose))
