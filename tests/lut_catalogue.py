"""Inputs that drive the gap-probability LUT kernels (gort_b200/csrc/gort_lut.cu) down paths the workload tests never
take, and Python restatements of the quantities that decide which path a set takes.  Shared by
test_lut_matrix_cpu.py, which asserts on the CPU that every case reaches its path, and test_lut_matrix_gpu.py.

Structures are [6][M] float64 columns (lambda, r, b, h1, h2, favd) as in include/gort_b200.h.

Restated from gort_lut.cu (the same IEEE operations in the same order, so the results are exact):
  n_tab(st6)        bins of the exp(-s_bin tau') table of lut_crown_kernel
  midpoints_k(st6)  K, the number of crown-centre heights of the v_g midpoint rule (lut_vg_kernel)
  plan(st)          group heads and sub-group sizes of lut_plan_kernel
"""
import numpy as np

from gort_b200.api import structure_from_options

NLAYERS = 15
LUT_TAB = 512
LUT_SUB = 8
GROUP_CAP = 64
LUT_CHUNK = 16384              # sets per pass of gort_lut
DEAD_CHUNK = LUT_CHUNK // 2    # sets per pass of gort_lut_intermediates
FIELDS = ("lambda", "r", "b", "h1", "h2", "favd")


# ---- restatements --------------------------------------------------------------------------------------------------
def _shape(st6):
    lam, r, b, h1, h2, favd = (float(v) for v in st6)
    ellip = b / r
    z1 = h1 - r * ellip
    z2 = h2 + r * ellip
    dz = (z2 - z1) / (NLAYERS - 1.0)
    return r, ellip, h1 / ellip, h2 / ellip, dz, dz / ellip


def n_tab(st6):
    """lut_crown_kernel: (int) fmin(LUT_TAB, 42 r / ds + 2); bins at or beyond n_tab - 1 raise `redo`, and bins
    from n_tab on are evaluated with the formula instead of the table."""
    r, _, _, _, ds, _ = _shape(st6)
    return int(min(float(LUT_TAB), 42.0 * r / ds + 2.0))


def midpoints_k(st6):
    """lut_vg_kernel: K counted with the running sum z += dz' from h1' + dz'/2 while z <= h2' (K = 17 stands for
    more than 16).  K = 0 or K >= 16 takes the literal proj_volume fallback."""
    _, _, h1p, h2p, _, dzp = _shape(st6)
    z, k = h1p + dzp / 2.0, 0
    while z <= h2p and k < 16:
        k += 1
        z += dzp
    if k == 16 and z <= h2p:
        k = 17
    return k


def _same_shape(st, a, b):
    return all(st[q, a] == st[q, b] for q in (1, 2, 3, 4))


def plan(st, chunk=LUT_CHUNK, cap=GROUP_CAP):
    """lut_plan_kernel over a whole call (m0 = 0): head[e] = pass-local index of set e's group head, sub[e] = size of
    the sub-group set e heads (0 if it heads none).  Pass boundaries every `chunk` sets, group cuts at multiples of
    `cap` of the global index."""
    n = st.shape[1]
    chunk = min(n, chunk)
    head = np.zeros(n, dtype=np.int64)
    sub = np.zeros(n, dtype=np.int64)
    for e in range(n):
        base = e // chunk * chunk
        i, n_pass = e - base, min(chunk, n - base)
        h = i
        while h > 0 and (base + h) % cap != 0 and _same_shape(st, base + h, base + h - 1):
            h -= 1
        head[e] = h
        rs = i
        while rs > h and st[0, base + rs - 1] == st[0, e]:
            rs -= 1
        if (i - rs) % LUT_SUB == 0:
            nj = 1
            while (nj < LUT_SUB and i + nj < n_pass and (base + i + nj) % cap != 0 and
                   _same_shape(st, base + i + nj, base + i + nj - 1) and st[0, base + i + nj] == st[0, e]):
                nj += 1
            sub[e] = nj
    return head, sub


def sub_groups(sub):
    """[(first set, size)] of the sub-groups of a plan."""
    return [(int(e), int(sub[e])) for e in np.flatnonzero(sub)]


# ---- catalogues ----------------------------------------------------------------------------------------------------
def _set(br, r, dh, cover, favd, h0=1.0):
    b = br * r
    h1 = b + h0
    return [cover / (np.pi * r * r), r, b, h1, h1 + dh, favd]


def _cols(rows):
    return np.ascontiguousarray(np.array(rows, dtype=np.float64).T)


# Oblate crowns whose crown-count loop reaches bins beyond the 512-bin table: r / ds = 14 r / (h2 - h1 + 2 b) is large
# for b / r <= 0.3 and thin layers.  Dense covers weight the far bins (temp1 grows as the layer thins), so a wrong
# beyond-table value moves epgap by 1e-8 .. 1e-4.  (b / r >= 0.4 stays inside the table: 42 r / ds + 2 > 512 still,
# but the path length s < s' does not reach 512 ds.)
# (b/r, r, h2 - h1, cover, favd)
OBLATE = [
    (0.1, 0.5, 0.05, 0.8, 0.3), (0.1, 0.5, 0.05, 0.3, 2.0), (0.1, 0.5, 0.05, 0.8, 2.0),
    (0.1, 1.5, 0.05, 0.8, 0.3), (0.1, 1.5, 0.05, 0.3, 0.3), (0.1, 1.5, 0.5, 0.8, 2.0),
    (0.1, 3.0, 0.05, 0.8, 2.0), (0.1, 3.0, 0.5, 0.8, 0.3),
    (0.2, 0.5, 0.05, 0.8, 2.0), (0.2, 1.5, 0.05, 0.8, 0.3), (0.2, 3.0, 0.05, 0.8, 0.3), (0.2, 3.0, 0.5, 0.8, 0.3),
    (0.3, 1.5, 0.05, 0.8, 0.3), (0.2, 0.5, 0.05, 0.3, 0.3), (0.3, 1.5, 0.05, 0.8, 2.0),
]
# the reference CLI's -HB / -BR / -PCC / -LAI (r = 10)
OBLATE_CLI = [dict(hb=0.1, br=0.3, pcc=0.7), dict(hb=0.3, br=0.2, pcc=0.8, lai=1.0), dict(hb=0.1, br=0.3, pcc=0.7, lai=1.0),
              dict(hb=0.02, br=0.1, pcc=0.9, lai=0.5)]


def beyond_table_singles():
    """Every set its own sub-group of one (no two neighbours share shape and lambda): lut_crown_kernel<1>."""
    return _cols([_set(*p) for p in OBLATE] + [list(structure_from_options(**kw)) for kw in OBLATE_CLI])


# Sub-groups of 2 .. 8 members: one shape and one lambda each, every member its own favd (the head's differs from the
# others', so a member given the head's favd beyond the table is visible).  Consecutive sub-groups differ in shape or
# lambda, and the batch is shorter than the group cap, so the plan cuts exactly these runs.
SUB_SHAPES = [(0.1, 1.5, 0.05), (0.2, 3.0, 0.05), (0.1, 3.0, 0.5), (0.3, 1.5, 0.05)]
SUB_LAYOUT = [(0, 8, 0.8), (1, 2, 0.8), (0, 3, 0.75), (2, 7, 0.8), (1, 5, 0.8), (3, 6, 0.8), (0, 4, 0.8)]   # (shape, size, cover)


def beyond_table_subgroups():
    rows = []
    for s, size, cover in SUB_LAYOUT:
        for j, favd in enumerate(np.linspace(0.3, 2.4, size)[::-1]):
            rows.append(_set(*SUB_SHAPES[s], cover, float(favd)))
    return _cols(rows)


def _k_boundary(br, r, k):
    """The smallest h2 - h1 (h1 = b + 1) at which midpoints_k reaches k, to the last bit (bisection on the float)."""
    def kk(dh):
        return midpoints_k(_set(br, r, dh, 0.5, 1.0))
    lo, hi = 0.0, 4.0 * br * r
    assert kk(lo) < k <= kk(hi)
    while np.nextafter(lo, np.inf) < hi:
        mid = 0.5 * (lo + hi)
        if mid <= lo or mid >= hi:
            break
        lo, hi = (lo, mid) if kk(mid) >= k else (mid, hi)
    return hi


def thin_layers():
    """Sets with K = 0 (h2 - h1 < 2b/27: no midpoint, the literal fallback, v_g = 0) and K = 1 (a single midpoint),
    including the two floats on either side of the K = 0 / 1 and K = 1 / 2 boundaries.  -> (structure, K per set)."""
    rows = []
    for br, r, cover, favd in ((2.0, 1.0, 0.6, 0.8), (0.45, 10.0, 0.3, 0.5), (0.1, 1.5, 0.8, 0.3), (1.0, 0.4, 0.9, 2.0)):
        b = br * r
        for dh in (0.3 * 2 * b / 27, 0.9 * 2 * b / 27, 1.5 * 2 * b / 27, 0.2 * b):
            rows.append(_set(br, r, dh, cover, favd))
        for k in (1, 2):
            edge = _k_boundary(br, r, k)
            rows.append(_set(br, r, np.nextafter(edge, 0.0), cover, favd))
            rows.append(_set(br, r, edge, cover, favd))
    rows.append(list(structure_from_options(hb=0.05, br=0.45, pcc=0.3)))
    rows.append(list(structure_from_options(hb=0.05, br=0.45, pcc=0.3, lai=2.0)))
    st = _cols(rows)
    return st, np.array([midpoints_k(st[:, m]) for m in range(st.shape[1])])


def vb_exit_sets():
    """Sets on which gortt_calc_vb finds a sphere volume below -1e-7 and the reference exits.  The volume of a sphere
    centred on a layer and cut by the h1' and h2' planes is never negative in exact arithmetic (the two caps are
    smaller than complementary ones); in a thin layer it is the difference of nearly equal cap volumes, with a rounding
    error of order eps r^3, so the exit needs crowns of r ~ 3000.  Thin layers of ordinary crowns do not exit."""
    return _cols([_set(0.1, 3000.0, 1e-3, 0.5, 1e-3), _set(0.45, 3000.0, 0.1, 0.5, 1e-3)])


def _bump(v, how):
    return float(np.nextafter(v, np.inf)) if how == "ulp" else v * 1.05


def plan_batch():
    """One batch for every branch of lut_plan_kernel.  -> (structure, notes) where notes['pairs'] lists
    (index, field, 'ulp' | 'step') for neighbours (index - 1, index) that differ in exactly that field."""
    A = _set(2.0, 1.0, 5.0, 0.5, 0.8)
    B = _set(1.0, 0.8, 2.0, 0.4, 1.2)
    C = _set(0.3, 1.5, 0.05, 0.8, 0.3)          # oblate, beyond the table
    rows, pairs = [], []
    # a lead-in of distinct shapes so that the long runs below start at odd offsets
    for q in range(5):
        rows.append(_set(1.5, 0.5 + 0.1 * q, 3.0, 0.3, 1.0))
    # one shape run of 153 sets: lambda runs of length 1 .. 17 (every sub-group size, runs cut at 8), the 64-cap
    # inside both; favd differs within each lambda run
    for L in range(1, 18):
        lam = A[0] * (1.0 + 0.01 * L)
        for j in range(L):
            rows.append([lam] + A[1:5] + [0.4 + 0.1 * j])
    # neighbours that differ in exactly one field, by a step and by one ULP; the first of each pair repeats the
    # preceding set's shape so that a wrong merge has a group to join
    for how in ("step", "ulp"):
        for f in range(6):
            base = list(B)
            rows.append(list(base))
            rows.append(list(base))
            other = list(base)
            other[f] = _bump(base[f], how)
            rows.append(other)
            pairs.append((len(rows) - 1, FIELDS[f], how))
    # A-B-A of shapes, and of lambda inside one shape
    for s in (A, B, A, C, A, C):
        rows.append(list(s))
    lam2 = C[0] * 1.1
    for lam in (C[0], C[0], lam2, C[0], C[0], lam2, lam2, C[0]):
        rows.append([lam] + C[1:])
    # a second long run at an odd offset: one lambda, 101 sets (sub-groups of 8 cut by the cap), favd cycling
    if len(rows) % 2 == 0:
        rows.append(list(B))
    for j in range(101):
        rows.append(C[:5] + [0.2 + 0.05 * (j % 13)])
    return _cols(rows), dict(pairs=pairs)


def shifted(st, k, filler=None):
    """st behind k leading sets (the filler shares no shape with st unless given): moves every group cut."""
    if filler is None:
        filler = _set(0.7, 2.2, 7.0, 0.2, 0.6)
    return np.ascontiguousarray(np.concatenate([np.repeat(np.array(filler, dtype=np.float64).reshape(6, 1), k, axis=1), st], axis=1))


def passes_batch(n_pass, extra, seed=1005):
    """n_pass + extra sets in shape runs of 1 .. 100 (lambda runs of 1 .. 11 inside), one run straddling set n_pass."""
    rng = np.random.Generator(np.random.PCG64(seed))
    rows = []

    def run(L, lam_runs=True):
        shape = _set(float(rng.uniform(0.5, 4.0)), float(rng.uniform(0.3, 3.0)), float(rng.uniform(0.5, 15.0)), 0.5, 1.0,
                     h0=float(rng.uniform(0.0, 5.0)))
        j = 0
        while j < L:
            lam = shape[0] * float(rng.uniform(0.2, 1.8))
            for _ in range(min(int(rng.integers(1, 12)) if lam_runs else L, L - j)):
                rows.append([lam] + shape[1:5] + [float(rng.uniform(0.1, 3.0))])
                j += 1

    while len(rows) < n_pass - 140:
        run(int(rng.integers(1, 101)))
    run(n_pass - 41 - len(rows))
    run(100, lam_runs=False)                  # sets n_pass - 41 .. n_pass + 58: one shape, one lambda
    while len(rows) < n_pass + extra:
        run(int(rng.integers(1, 101)))
    return _cols(rows[:n_pass + extra])
