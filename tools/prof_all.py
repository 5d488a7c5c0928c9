"""ncu target (round 2): one invocation of every kernel of the library on shapes large enough to fill the GPU for a few
hundred microseconds: the LUT pipeline (ungrouped shapes, shape groups, Q08, the dead intermediates), spectra, the BRDF
path (geometry, per-wavelength kernel with and without component signatures, band kernel) and the energy balance."""
import sys
from pathlib import Path
import numpy as np
import torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import gort_b200
from gort_b200 import workloads as wk
g = gort_b200.Gort(0)
dev = torch.device("cuda:0")
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
rng = np.random.Generator(np.random.PCG64(3))
st = wk.random_structures(rng, 8192)
lut = g.lut(st)                                     # LUT pipeline, every set its own crown shape (C4b-like)
grid = np.ascontiguousarray(wk.c5_lut_grid()["structure"][:, :16384])
lg = g.lut(grid)                                    # LUT pipeline, shape groups of 64, sub-groups of 8
lq = g.lut(st[:, :2000], gort_b200.LUT_Q08)         # lut_q08_kernel
dead = g.lut_intermediates(st[:, :2000])            # lut_es_all_kernel, lut_dead_kernel
w = wk.c3_albedo(n_sets=600)
l2 = g.lut(w["structure"])
rl, tl, rs = g.spectra(w["leaf"], w["soil"], w["wavelength"])       # spectra_kernel
a, v, s = g.energy(w["structure"], l2, w["angles"], rl, tl, rs)     # energy_zenith_kernel, energy_kernel
w4 = wk.c4_enkf(n_members=20000)
l4 = np.repeat(g.lut(w4["structure"][:, :64])[:1], 20000, axis=0)
r4, t4, s4 = g.spectra(w4["leaf"], w4["soil"], w4["wavelength"])
b4 = g.brdf(w4["structure"], l4, w4["angles"], r4, t4, s4)          # geom_lines_kernel, rsurf_flat_kernel
w2 = wk.c2_hemisphere()
l1 = g.lut(w2["structure"])
r2, t2, s2 = g.spectra(w2["leaf"], w2["soil"], w2["wavelength"])
G = w2["angles"].shape[1]
d = [T(w2["structure"]), T(l1), T(w2["angles"]), T(r2[0]), T(t2[0]), T(s2[0])]
out = torch.empty((1, G, 2112), dtype=torch.float64, device=dev)
sc = torch.empty((1, G, 2112, 4), dtype=torch.float64, device=dev)
g.brdf_dev(*d, out); g.synchronize()                 # geom_kernel, rsurf_wide_kernel (TMA rows)
g.brdf_dev(*d, out, scomp=sc); g.synchronize()       # rsurf_wide_kernel with component signatures
print("ok", np.isfinite(lut).mean(), np.isfinite(a).mean(), np.isfinite(b4).mean(), float(torch.isfinite(sc).double().mean()))
