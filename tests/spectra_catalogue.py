"""Inputs for test_spectra_matrix_*.py and test_chain_matrix_gpu.py, and Python restatements of the index arithmetic
the kernels use, so that every case can assert on the CPU that its inputs reach the path it is named for.

  k_rows        PROSPECT-D absorption k of every table row, in prospect_row's order (gort_spectra.cu): with
                -fmad=false (csrc/Makefile) and -ffp-contract=off (oracle/Makefile) it has the bits of both
  tau_branch    which branch of plate_tau each row takes: 0 k <= 0, 1 (0, 4], 2 (4, 85], 3 k > 85
  leaf_index    lower / upper / float fraction of a wavelength on the 1-nm PROSPECT grid (gortt.c:1338,1364)
  soil_index    the same on the 5-nm Price soil grid (gortt.c:1311-1321)
  jac_chunk     members per pass of gort_jacobian_batch;  forward_chunk  the same for gort_forward_batch
"""
import numpy as np

from test_prospect_independent_cpu import tables_from_header

NW = 2101
SOIL_NW = 421
WL_MIN, WL_MAX = 400.0, 2500.0

_T = {}


def tables():
    if not _T:
        _T.update(tables_from_header())
    return _T


def k_rows(leaf7):
    N, cab, car, anth, cbrown, cw, cm = (float(x) for x in leaf7)
    T = tables()
    return (((((cab * T["k_Cab"] + car * T["k_Car"]) + anth * T["k_Anth"]) + cbrown * T["k_Brown"])
             + cw * T["k_Cw"]) + cm * T["k_Cm"]) / N


def tau_branch(k):
    k = np.asarray(k)
    return np.where(k <= 0.0, 0, np.where(k <= 4.0, 1, np.where(k <= 85.0, 2, 3)))


def leaf_index(wl):
    """(lower, upper, fraction as float32) per wavelength, as gortt_prospect_interface: the fraction is
    (float)(wl - 400) widened to double, minus lower, rounded to float."""
    wl = np.asarray(wl, dtype=np.float64)
    upper = np.trunc(1 + (wl - 400.0) / 1.0).astype(np.int64)
    lower = np.trunc((wl - 400.0) / 1.0).astype(np.int64)
    fraction = (np.float32(wl - 400.0).astype(np.float64) / 1.0 - lower).astype(np.float32)
    return lower, upper, fraction


def soil_index(wl):
    wl = np.asarray(wl, dtype=np.float64)
    upper = np.trunc(1. + (wl - 400) / 5.0).astype(np.int64)
    lower = np.trunc((wl - 400) / 5.0).astype(np.int64)
    fraction = (wl - 400.) / 5.0 - lower
    return lower, upper, fraction


def jac_chunk(M, G, W):
    c = (256 << 20) // (G * W * 8)
    return min(max(c, 1), M)


def forward_chunk(M):
    c = min((M + 7) // 8, 16384)
    return min(max(c, 1024), M)


def n_chunks(M, c):
    return -(-M // c)


# ---- leaves ---------------------------------------------------------------------------------------
def _leaf(N, cab, car, anth, cbrown, cw, cm):
    return np.array([N, cab, car, anth, cbrown, cw, cm], dtype=np.float64)


def k_branches():
    """[7][L]: every N in {1, 1.5, 2.5} with a transparent leaf (k = 0, tau = 1 on every row), a pigment-only leaf
    (k = 0 beyond the pigment bands), an ordinary leaf and two wet/dry-matter-heavy leaves (k > 85 in the water bands)."""
    kinds = [(0, 0, 0, 0, 0, 0),                 # transparent
             (40, 10, 2, 0.3, 0, 0),             # pigments only
             (45, 10, 1, 0.1, 0.012, 0.008),     # ordinary
             (30, 7, 1, 0, 1.0, 0.01),           # wet
             (30, 7, 1, 0, 1.5, 0.6)]            # wet and dry matter heavy
    return np.stack([_leaf(N, *kd) for N in (1.0, 1.5, 2.5) for kd in kinds], axis=1)


_BOUNDARY_LEAF = (30, 7, 1, 0.2, 1.2, 0.02)


def _n_for_k(S, k_want, N0):
    """the float N nearest N0 with S / N == k_want exactly (None if no float within 64 ULP does)"""
    lo = hi = N0
    for _ in range(64):
        for N in (lo, hi):
            if S / N == k_want:
                return N
        lo, hi = np.nextafter(lo, 0.0), np.nextafter(hi, np.inf)
    return None


def k_boundaries():
    """leaves [7][6] and the row of each: three N that put k at one row on 4.0 and one ULP either side of it, then
    three around 85.0 at another row.  k = S / N with S the row's absorber sum, so N = S / 4 (exact) gives k == 4.0;
    for 85 the floats around S / 85 are searched.  The rows are the first whose N lies in [1.2, 1.9]."""
    base = _leaf(1.0, *_BOUNDARY_LEAF)
    S_rows = k_rows(base)
    leaves, rows = [], []
    for edge in (4.0, 85.0):
        for row in np.flatnonzero((S_rows / edge >= 1.2) & (S_rows / edge <= 1.9)):
            S = float(S_rows[row])
            Ns = [_n_for_k(S, k_want, S / edge) for k_want in (np.nextafter(edge, 0.0), edge, np.nextafter(edge, np.inf))]
            if None not in Ns:
                break
        else:
            raise AssertionError("no row reaches k == %g" % edge)
        leaves += [_leaf(N, *_BOUNDARY_LEAF) for N in Ns]
        rows += [int(row)] * 3
    return np.stack(leaves, axis=1), np.array(rows)


NAN_EDGE_LEAVES = np.stack([_leaf(1.5, 30, 7, 1, 0, 1.0, 0.01), _leaf(2.0, 30, 7, 1, 0, 1.5, 0.01)], axis=1)


def k_runs(mask):
    """[(first, last)] row runs where mask holds"""
    m = np.concatenate([[False], mask, [False]]).astype(np.int8)
    d = np.diff(m)
    return list(zip(np.flatnonzero(d == 1), np.flatnonzero(d == -1) - 1))


def nan_edge():
    """leaves [7][2] and, per leaf, the integer wavelength just before each k > 85 run (fraction 0: its upper row is
    NaN for N > 1) and the half-integer beside it"""
    wls = []
    for m in range(NAN_EDGE_LEAVES.shape[1]):
        w = []
        for first, _ in k_runs(k_rows(NAN_EDGE_LEAVES[:, m]) > 85.0):
            w += [400.0 + first - 1, 400.0 + first - 0.5]
        wls.append(np.array(w))
    return NAN_EDGE_LEAVES, wls


# ---- wavelengths ----------------------------------------------------------------------------------
def wl_ends():
    return np.array([WL_MIN, np.nextafter(WL_MIN, np.inf), np.nextafter(WL_MAX, 0.0), WL_MAX])


def wl_integers():
    return np.concatenate([np.arange(400.0, 420.0), np.arange(1900.0, 1950.0), np.arange(2480.0, 2501.0)])


def wl_fraction_one():
    """400 + i - 2**-20 where (float)(wl - 400) rounds up to i: lower = i - 1 with weight 1 - 1.0f = 0"""
    i = np.arange(8, NW - 1, 7, dtype=np.float64)
    wl = 400.0 + i - 2.0 ** -20
    return wl[np.float32(wl - 400.0) == i]


def wl_float_fraction(rng, n=64):
    """wavelengths whose float fraction differs from the double fraction (wl - 400) - lower by more than 1e-6"""
    wl = rng.uniform(1500.0, 2500.0, 8 * n)
    lower, _, f = leaf_index(wl)
    keep = np.abs(f.astype(np.float64) - ((wl - 400.0) - lower)) > 1e-6
    return wl[keep][:n]


def wl_soil_nodes():
    nodes = 400.0 + 5.0 * np.arange(0, SOIL_NW, 3)
    below = np.nextafter(nodes[1:], 0.0)
    return np.concatenate([nodes, below])


def wavelengths(seed=7):
    rng = np.random.Generator(np.random.PCG64(seed))
    return np.concatenate([wl_ends(), wl_integers(), wl_fraction_one(), wl_float_fraction(rng), wl_soil_nodes(),
                           rng.uniform(WL_MIN, WL_MAX, 200)])
