"""PROSPECT-D (SURVEY.md row a16) is "parity unpinned": the reference's implementation is Fortran 90 and no Fortran
compiler exists in the build image.  This test does not change that; it narrows the gap with a SECOND restatement,
written in numpy directly from the Fortran text (PROSPECT-D/prospect_DB.f90:72-191, tav_abs.f90:16-60), with the
tables parsed from PROSPECT-D/dataSpec_PDB.f90 itself when the reference tree is present.  The two restatements
(this one and oracle/prospect_d_oracle.c, which the CUDA kernel is tested against) were written independently of
each other's code; they must agree to rounding, and the table generator's output must equal the Fortran literals
rounded to REAL(4).
"""
import os
import re
from pathlib import Path

import numpy as np
import pytest

from gort_b200 import workloads as wk

ROOT = Path(__file__).resolve().parent.parent
REF = Path("/root/reference/PROSPECT-D/dataSpec_PDB.f90")
# os.path.isfile, not Path.exists: a tree this user may not enter counts as absent instead of raising PermissionError
HAVE_REF = os.path.isfile(REF)
NW = 2101
NAMES = ["refractive", "k_Cab", "k_Car", "k_Anth", "k_Brown", "k_Cw", "k_Cm"]


def tables_from_fortran():
    """DATA statements of dataSpec_PDB.f90: unsuffixed literals are REAL(4) constants widened on assignment."""
    txt = REF.read_text(errors="replace")
    out = {}
    for name in NAMES:
        vals = np.zeros(NW)
        for m in re.finditer(r"data\s*\(\s*%s\s*\(i\)\s*,\s*i\s*=\s*(\d+)\s*,\s*(\d+)\s*\)\s*/(.*?)/" % re.escape(name), txt, re.S | re.I):
            lo, hi = int(m.group(1)), int(m.group(2))
            body = re.sub(r"&|\n|!.*", " ", m.group(3))
            nums = []
            for x in body.replace(",", " ").split():
                if "*" in x:                          # Fortran repeat count: 1701*0.
                    n, v = x.split("*")
                    nums += [v] * int(n)
                else:
                    nums.append(x)
            assert len(nums) == hi - lo + 1, (name, lo, hi, len(nums))
            vals[lo - 1:hi] = [float(np.float32(float(x.lower().replace("d", "e")))) for x in nums]
        out[name] = vals
    return out


def tables_from_header():
    """gort_b200/data/gort_tables.h: binary32 bit patterns written by tools/gen_tables.py."""
    txt = (ROOT / "gort_b200" / "data" / "gort_tables.h").read_text()
    out = {}
    for name in NAMES:
        m = re.search(r"gort_tab_%s_f32\[[^\]]*\]\s*=\s*\{(.*?)\};" % name.lower(), txt, re.S)
        assert m, name
        bits = np.array([int(x, 16) for x in re.findall(r"0x[0-9a-fA-F]+", m.group(1))], dtype=np.uint32)
        assert bits.size == NW, (name, bits.size)
        out[name] = bits.view(np.float32).astype(np.float64)
    return out


def tav_abs(theta, nr):
    pi = float(np.float32(np.arctan(np.float32(1.0))) * np.float32(4.0))      # pi = atan(1.)*4.   in REAL(4)
    rd = pi / 180.0
    n2 = np.power(nr, 2.0)
    npp = n2 + 1.0
    nm = n2 - 1.0
    a = (nr + 1.0) * (nr + 1.0) / 2.0
    k = -((n2 - 1.0) * (n2 - 1.0) / 4.0)
    sa = np.sin(theta * rd)
    if theta == 90.0:
        b1 = np.zeros_like(nr)
    else:
        b1 = np.sqrt((sa * sa - npp / 2.0) * (sa * sa - npp / 2.0) + k)
    b2 = sa * sa - npp / 2.0
    b = b1 - b2
    b3 = b * b * b
    a3 = a * a * a
    ts = (np.power(k, 2.0) / (6.0 * b3) + k / b - b / 2.0) - (np.power(k, 2.0) / (6.0 * a3) + k / a - a / 2.0)
    tp1 = -(2.0 * n2 * (b - a) / (npp * npp))
    tp2 = -(2.0 * n2 * npp * np.log(b / a) / (nm * nm))
    tp3 = n2 * (1.0 / b - 1.0 / a) / 2.0
    tp4 = 16.0 * np.power(n2, 2.0) * (n2 * n2 + 1.0) * np.log((2.0 * npp * b - nm * nm) / (2.0 * npp * a - nm * nm)) \
        / (np.power(npp, 3.0) * (nm * nm))
    tp5 = 16.0 * np.power(n2, 3.0) * (1.0 / (2.0 * npp * b - nm * nm) - 1.0 / (2.0 * npp * a - nm * nm)) / (npp * npp * npp)
    tp = tp1 + tp2 + tp3 + tp4 + tp5
    return (ts + tp) / (2.0 * (sa * sa))


C1 = [-3.60311230482612224e-13, 3.46348526554087424e-12, -2.99627399604128973e-11, 2.57747807106988589e-10,
      -2.09330568435488303e-9, 1.59501329936987818e-8, -1.13717900285428895e-7, 7.55292885309152956e-7,
      -4.64980751480619431e-6, 2.63830365675408129e-5, -1.37089870978830576e-4, 6.47686503728103400e-4,
      -2.76060141343627983e-3, 1.05306034687449505e-2, -3.57191348753631956e-2, 1.07774527938978692e-1,
      -2.96997075145080963e-1, 8.64664716763387311e-1, 7.42047691268006429e-1]
C2 = [-1.62806570868460749e-12, -8.95400579318284288e-13, -4.08352702838151578e-12, -1.45132988248537498e-11,
      -8.35086918940757852e-11, -2.13638678953766289e-10, -1.10302431467069770e-9, -3.67128915633455484e-9,
      -1.66980544304104726e-8, -6.11774386401295125e-8, -2.70306163610271497e-7, -1.05565006992891261e-6,
      -4.72090467203711484e-6, -1.95076375089955937e-5, -9.16450482931221453e-5, -4.05892130452128677e-4,
      -2.14213055000334718e-3, -1.06374875116569657e-2, -8.50699154984571871e-2, 9.23755307807784058e-1]


def horner(c, x):
    y = np.full_like(x, c[0])
    for ck in c[1:]:
        y = y * x + ck
    return y


def prospect_db(T, N, Cab, Car, Anth, Cbrown, Cw, Cm):
    k = (Cab * T["k_Cab"] + Car * T["k_Car"] + Anth * T["k_Anth"] + Cbrown * T["k_Brown"] + Cw * T["k_Cw"] + Cm * T["k_Cm"]) / N
    tau = np.zeros(NW)
    with np.errstate(all="ignore"):
        m0 = k <= 0.0
        tau[m0] = 1.0
        m1 = (k > 0.0) & (k <= 4.0)
        xx = 0.5 * k[m1] - 1.0
        yy = horner(C1, xx) - np.log(k[m1])
        tau[m1] = (1.0 - k[m1]) * np.exp(-k[m1]) + k[m1] * k[m1] * yy
        m2 = (k > 4.0) & (k <= 85.0)
        xx = 14.5 / (k[m2] + 3.25) - 1.0
        yy = np.exp(-k[m2]) * horner(C2, xx) / k[m2]
        tau[m2] = (1.0 - k[m2]) * np.exp(-k[m2]) + k[m2] * k[m2] * yy
    nr = T["refractive"]
    t12 = tav_abs(90.0, nr)
    talf = tav_abs(40.0, nr)
    ralf = 1.0 - talf
    r12 = 1.0 - t12
    t21 = t12 / (nr * nr)
    r21 = 1.0 - t21
    denom = 1.0 - r21 * r21 * (tau * tau)
    Ta = talf * tau * t21 / denom
    Ra = ralf + r21 * tau * Ta
    t = t12 * tau * t21 / denom
    r = r12 + r21 * tau * t
    D = np.sqrt((1.0 + r + t) * (1.0 + r - t) * (1.0 - r + t) * (1.0 - r - t))
    rq = r * r
    tq = t * t
    a = (1.0 + rq - tq + D) / (2.0 * r)
    b = (1.0 - rq + tq + D) / (2.0 * t)
    bNm1 = np.power(b, N - 1.0)
    bN2 = bNm1 * bNm1
    a2 = a * a
    denom = a2 * bN2 - 1.0
    Rsub = a * (bN2 - 1.0) / denom
    Tsub = bNm1 * (a2 - 1.0) / denom
    z = (r + t) >= 1.0
    Tsub = np.where(z, t / (t + (1.0 - t) * (N - 1.0)), Tsub)
    Rsub = np.where(z, 1.0 - Tsub, Rsub)
    denom = 1.0 - Rsub * r
    return Ra + Ta * Rsub * t / denom, Ta * Tsub / denom


def test_table_generator_matches_fortran_literals():
    if not HAVE_REF:
        pytest.skip("reference tree not present")
    tf, th = tables_from_fortran(), tables_from_header()
    for name in NAMES:
        assert np.array_equal(tf[name], th[name]), name


def test_second_restatement_agrees_with_the_oracle(oracle):
    T = tables_from_fortran() if HAVE_REF else tables_from_header()
    rng = np.random.Generator(np.random.PCG64(77))
    leaves = np.concatenate([wk.DEFAULT_LEAF.reshape(7, 1), wk.random_leaves(rng, 12)], axis=1)
    leaves[4, 3] = 0.0          # Cbrown = 0
    leaves[0, 5] = 1.0          # N = 1: b**(N-1) = 1
    wl = np.arange(400.0, 2501.0)
    worst = 0.0
    for m in range(leaves.shape[1]):
        refl, tran = prospect_db(T, *leaves[:, m])
        rl, tl, _ = oracle.spectra(leaves[:, m], wk.DEFAULT_SOIL, wl)
        for x, y in ((refl, rl), (tran, tl)):
            e = np.max(np.abs(x - y) / np.maximum(np.abs(y), 1e-12))
            worst = max(worst, e)
            assert e < 1e-11, "leaf %d: %.3e" % (m, e)
    print("numpy restatement vs oracle: worst rel diff %.3e" % worst)
