"""Python host binding over the C ABI of libgort_b200.so (include/gort_b200.h).

This is the ctypes stub a maintainer of a Python data-assimilation system would add (see
INTEGRATION.md); it contains no model arithmetic.  It mirrors the reference's function
boundary (include/gortt.h:216-292) in batched form:

    reference                                           here
    gortt_init_params + gortt_gap_probabilities[_Q08]   Gort.lut(structure, method)
    gortt_price_soil + gortt_prospect_interface         Gort.spectra(leaf, soil, wavelength, ...)
    gortt_set_zenith_dependant_probabilities + rsurf    Gort.brdf(structure, lut, angles, spectra)
    gortt_energy / gortt_albedo / gauleg                Gort.energy(...), Gort.gauleg()

Host entry points take / return numpy arrays (H2D and D2H copies happen inside the library).
`*_dev` entry points take torch CUDA tensors (device pointers) and enqueue on a CUDA stream;
torch is used only for device memory and streams.

There is no CPU fallback: if the shared library is missing or no GPU is present, constructing
`Gort` raises.
"""
import ctypes as C
import os
from pathlib import Path

import numpy as np

NTH = 91
LUT_STRIDE = 2 * NTH + 2
LUT_FULL, LUT_Q08 = 0, 1
JAC_LAMBDA, JAC_R, JAC_B, JAC_H1, JAC_H2, JAC_FAVD, JAC_LAI = range(7)
PROSPECT_NW = 2101
SOIL_TABLE_NW = 2101
MAX_BANDS = 64

_LIB_PATH = Path(__file__).resolve().parent / "libgort_b200.so"
_dp = C.POINTER(C.c_double)


class GortError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("gort_b200 error %d: %s" % (code, msg))
        self.code = code


class _Options(C.Structure):
    _fields_ = [("use_beta", C.c_int), ("beta", C.c_double), ("use_fd", C.c_int), ("fd", C.c_double)]


class _Shape(C.Structure):
    _fields_ = [("n_sets", C.c_int), ("n_geom", C.c_int), ("n_wl", C.c_int),
                ("geom_per_set", C.c_int), ("spectra_per_set", C.c_int), ("opt", _Options),
                ("out_pitch", C.c_int)]


_lib = None

# every symbol include/gort_b200.h declares
ABI_SYMBOLS = [
    "gort_create", "gort_destroy", "gort_last_error", "gort_stream", "gort_synchronize",
    "gort_device_count", "gort_host_alloc", "gort_host_free", "gort_launch_count",
    "gort_lut_batch", "gort_lut_batch_dev", "gort_lut_batch_scatter_dev", "gort_spectra_batch", "gort_spectra_batch_dev",
    "gort_prospect_batch", "gort_brdf_batch", "gort_brdf_batch_dev", "gort_energy_batch",
    "gort_energy_batch_dev", "gort_gauleg", "gort_lut_write_text", "gort_lut_read_text",
    "gort_dfma_peak", "gort_profile_begin", "gort_profile_end", "gort_set_overlap", "gort_kernel_stamps_enable", "gort_kernel_stamps",
    "gort_forward_batch", "gort_jacobian_batch", "gort_lut_intermediates_batch", "gort_lut_intermediates_batch_dev", "gort_host_alloc_near", "gort_host_alloc_on_cpus", "gort_host_placement", "gort_soil_table_read", "gort_soil_from_table", "gort_soil_from_table_dev",
    "gort_brdf_band_batch", "gort_brdf_band_batch_dev", "gort_energy_band_batch", "gort_energy_band_batch_dev",
    "gort_forward_band_batch",
    "gort_lut_tangent_batch_dev", "gort_brdf_tangent_batch_dev", "gort_lai_tangent_batch",
]


def load_library():
    """Load libgort_b200.so and declare the prototypes. Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise GortError(2, "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % _LIB_PATH)
    lib = C.CDLL(str(_LIB_PATH))
    vp = C.c_void_p
    lib.gort_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.gort_destroy.argtypes = [vp]
    lib.gort_destroy.restype = None
    lib.gort_last_error.argtypes = [vp]
    lib.gort_last_error.restype = C.c_char_p
    lib.gort_stream.argtypes = [vp]
    lib.gort_stream.restype = vp
    lib.gort_synchronize.argtypes = [vp]
    lib.gort_set_overlap.argtypes = [vp, C.c_int]
    lib.gort_kernel_stamps_enable.argtypes = [vp, C.c_int]
    lib.gort_kernel_stamps.argtypes = [vp, _dp, _dp, _dp, C.POINTER(C.c_int)]
    lib.gort_soil_table_read.argtypes = [C.c_char_p, vp, C.c_char_p, C.c_size_t]
    lib.gort_soil_from_table.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp]
    lib.gort_soil_from_table_dev.argtypes = [vp, vp, vp, C.c_int, C.c_int, vp, vp]
    lib.gort_device_count.restype = C.c_int
    lib.gort_host_alloc.argtypes = [C.c_size_t]
    lib.gort_host_alloc.restype = vp
    lib.gort_host_alloc_on_cpus.argtypes = [C.c_size_t, C.POINTER(C.c_int), C.c_int]
    lib.gort_host_alloc_on_cpus.restype = vp
    lib.gort_host_alloc_near.argtypes = [vp, C.c_size_t]
    lib.gort_host_alloc_near.restype = vp
    lib.gort_host_placement.argtypes = [vp, C.c_char_p, C.c_size_t]
    lib.gort_host_free.argtypes = [vp]
    lib.gort_host_free.restype = None
    lib.gort_launch_count.argtypes = [vp]
    lib.gort_launch_count.restype = C.c_long
    lib.gort_lut_batch.argtypes = [vp, C.c_int, vp, C.c_int, vp]
    lib.gort_lut_batch_dev.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp]
    lib.gort_lut_batch_scatter_dev.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp, C.c_int, C.POINTER(vp), C.c_int]
    lib.gort_lut_intermediates_batch.argtypes = [vp, C.c_int] + [vp] * 7
    lib.gort_lut_intermediates_batch_dev.argtypes = [vp, vp, C.c_int] + [vp] * 7
    lib.gort_spectra_batch.argtypes = [vp, C.c_int, vp, vp, C.c_double, C.c_double, C.c_int, vp, vp, vp, vp]
    lib.gort_spectra_batch_dev.argtypes = [vp, vp, C.c_int, vp, vp, C.c_double, C.c_double, C.c_int, vp, vp, vp, vp]
    lib.gort_prospect_batch.argtypes = [vp, C.c_int, vp, vp, vp]
    sp = C.POINTER(_Shape)
    lib.gort_brdf_batch.argtypes = [vp, sp] + [vp] * 9
    lib.gort_brdf_batch_dev.argtypes = [vp, vp, sp] + [vp] * 9
    lib.gort_energy_batch.argtypes = [vp, sp] + [vp] * 9
    lib.gort_energy_batch_dev.argtypes = [vp, vp, sp] + [vp] * 9
    lib.gort_forward_batch.argtypes = [vp, sp, C.c_int, vp, vp, vp, C.c_double, C.c_double, vp, vp, vp, vp]
    lib.gort_brdf_band_batch.argtypes = [vp, sp, C.c_int] + [vp] * 8
    lib.gort_brdf_band_batch_dev.argtypes = [vp, vp, sp, C.c_int] + [vp] * 8
    lib.gort_energy_band_batch.argtypes = [vp, sp, C.c_int] + [vp] * 10
    lib.gort_energy_band_batch_dev.argtypes = [vp, vp, sp, C.c_int] + [vp] * 10
    lib.gort_forward_band_batch.argtypes = [vp, sp, C.c_int, vp, vp, vp, C.c_double, C.c_double, vp, C.c_int, vp, vp, vp, vp]
    lib.gort_jacobian_batch.argtypes = [vp, sp, C.c_int, C.c_int, C.c_double, vp, vp, vp, C.c_double, C.c_double, vp, vp, vp, vp]
    lib.gort_lut_tangent_batch_dev.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp, vp]
    lib.gort_brdf_tangent_batch_dev.argtypes = [vp, vp, sp] + [vp] * 8
    lib.gort_lai_tangent_batch.argtypes = [vp, sp, C.c_int, C.c_int, vp, vp, vp, C.c_double, C.c_double, vp, vp, vp, vp]
    lib.gort_gauleg.argtypes = [vp, vp, vp]
    lib.gort_lut_write_text.argtypes = [vp, vp]
    lib.gort_lut_write_text.restype = C.c_long
    lib.gort_lut_read_text.argtypes = [C.c_char_p, vp]
    lib.gort_dfma_peak.argtypes = [vp, _dp]
    lib.gort_profile_begin.argtypes = [vp, C.c_int]
    lib.gort_profile_end.argtypes = [vp, _dp, _dp, C.POINTER(C.c_int)]
    _lib = lib
    return lib


def _np(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(a):
    """numpy array or torch tensor -> raw address (None -> NULL)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
        return a.ctypes.data
    # torch tensor
    assert a.is_contiguous() and a.dtype.is_floating_point and a.element_size() == 8
    return a.data_ptr()


class PinnedArray:
    """A numpy float64 view over pinned host memory from gort_host_alloc; with cpus=[...] pinned while running on those
    CPUs (gort_host_alloc_on_cpus); with near=<Gort> placed by that context's own probe (gort_host_alloc_near)."""

    def __init__(self, shape, near=None, cpus=None):
        self._lib = load_library()
        n = int(np.prod(shape))
        if cpus:
            arr = (C.c_int * len(cpus))(*[int(c) for c in cpus])
            self._p = self._lib.gort_host_alloc_on_cpus(max(n, 1) * 8, arr, len(cpus))
        elif near is not None:
            self._p = self._lib.gort_host_alloc_near(near._h, max(n, 1) * 8)
        else:
            self._p = self._lib.gort_host_alloc(max(n, 1) * 8)
        if not self._p:
            raise GortError(4, "gort_host_alloc failed")
        buf = (C.c_double * n).from_address(self._p)
        self.array = np.frombuffer(buf, dtype=np.float64).reshape(shape)

    def free(self):
        if self._p:
            self.array = None
            self._lib.gort_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Gort:
    """One context = one GPU + one CUDA stream + grow-only device scratch."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = C.c_void_p()
        rc = self._lib.gort_create(device, C.byref(h))
        if rc != 0:
            raise GortError(rc, self._lib.gort_last_error(None).decode())
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gort_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise GortError(rc, self._lib.gort_last_error(self._h).decode())

    # ---- misc ----
    @property
    def stream(self):
        return self._lib.gort_stream(self._h)

    def synchronize(self):
        self._check(self._lib.gort_synchronize(self._h))

    def set_overlap(self, enable=True):
        """Let consecutive same-shape brdf_dev calls overlap on the GPU (contract: include/gort_b200.h)."""
        self._check(self._lib.gort_set_overlap(self._h, int(bool(enable))))

    def host_placement(self):
        """what gort_host_alloc_near found out about pinned-buffer placement (a sentence)"""
        buf = C.create_string_buffer(600)
        self._check(self._lib.gort_host_placement(self._h, buf, 600))
        return buf.value.decode()

    def launch_count(self):
        return self._lib.gort_launch_count(self._h)

    def dfma_peak_tflops(self):
        v = C.c_double()
        self._check(self._lib.gort_dfma_peak(self._h, C.byref(v)))
        return v.value

    def profile_begin(self, max_steps):
        self._check(self._lib.gort_profile_begin(self._h, int(max_steps)))

    def profile_end(self):
        """-> (mean geometry-kernel ms, mean per-wavelength-kernel ms, calls recorded)"""
        g = C.c_double(); r = C.c_double(); n = C.c_int()
        self._check(self._lib.gort_profile_end(self._h, C.byref(g), C.byref(r), C.byref(n)))
        return g.value, r.value, n.value

    def kernel_stamps_enable(self, enable=True):
        self._check(self._lib.gort_kernel_stamps_enable(self._h, int(bool(enable))))

    def kernel_stamps(self):
        """-> dict: in-kernel span (first CTA entry to last CTA exit), mean per-CTA start-up and store phase [us], CTAs"""
        a = C.c_double(); b = C.c_double(); c = C.c_double(); n = C.c_int()
        self._check(self._lib.gort_kernel_stamps(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(n)))
        return {"span_us": a.value, "startup_us_per_cta": b.value, "store_phase_us_per_cta": c.value, "ctas": n.value}

    def gauleg(self):
        x = np.empty(32); w = np.empty(32)
        self._check(self._lib.gort_gauleg(self._h, _ptr(x), _ptr(w)))
        return x, w

    # ---- shapes ----
    @staticmethod
    def _shape(n_sets, n_geom, n_wl, geom_per_set, spectra_per_set, beta=None, fd=None, out_pitch=0):
        sh = _Shape()
        sh.out_pitch = int(out_pitch)
        sh.n_sets, sh.n_geom, sh.n_wl = n_sets, n_geom, n_wl
        sh.geom_per_set, sh.spectra_per_set = int(geom_per_set), int(spectra_per_set)
        sh.opt.use_beta = beta is not None
        sh.opt.beta = 0.0 if beta is None else float(beta)
        sh.opt.use_fd = fd is not None
        sh.opt.fd = 0.0 if fd is None else float(fd)
        return sh

    # ---- host API ----
    def lut(self, structure, method=LUT_FULL):
        """structure [6][M] -> LUT records [M][184]."""
        st = _np(structure)
        assert st.ndim == 2 and st.shape[0] == 6
        M = st.shape[1]
        out = np.empty((M, LUT_STRIDE))
        self._check(self._lib.gort_lut_batch(self._h, M, _ptr(st), method, _ptr(out)))
        return out

    def lut_intermediates(self, structure):
        """The intermediates the BRDF never reads (gortt_calc_vb / _fb / _t_open, dk_open, k_open[h]): dict of arrays
        vb [M][15], fb [M][15][91], t_open / dt_open [M][15][15], dk_open / k_open [M][15]."""
        st = _np(structure)
        M = st.shape[1]
        out = dict(vb=np.empty((M, 15)), fb=np.empty((M, 15, NTH)), t_open=np.empty((M, 15, 15)),
                   dt_open=np.empty((M, 15, 15)), dk_open=np.empty((M, 15)), k_open=np.empty((M, 15)))
        self._check(self._lib.gort_lut_intermediates_batch(self._h, M, _ptr(st), *[_ptr(out[k]) for k in
                                                           ("vb", "fb", "t_open", "dt_open", "dk_open", "k_open")]))
        return out

    def lut_intermediates_dev(self, structure, vb=None, fb=None, t_open=None, dt_open=None, dk_open=None, k_open=None, stream=None):
        M = structure.shape[1]
        self._check(self._lib.gort_lut_intermediates_batch_dev(self._h, stream, M, _ptr(structure), _ptr(vb), _ptr(fb),
                                                               _ptr(t_open), _ptr(dt_open), _ptr(dk_open), _ptr(k_open)))

    def spectra(self, leaf, soil, wavelength, user_leaf=-1.0, user_soil=-1.0, n_sets=None):
        """leaf [7][M], soil [4][M], wavelength [W] -> rleaf, tleaf, rsoil each [M][W]."""
        wl = _np(wavelength).ravel()
        leaf = None if leaf is None else _np(leaf)
        soil = None if soil is None else _np(soil)
        if n_sets is None:
            n_sets = leaf.shape[1] if leaf is not None else (soil.shape[1] if soil is not None else 1)
        M, W = n_sets, wl.shape[0]
        rl = np.empty((M, W)); tl = np.empty((M, W)); rs = np.empty((M, W))
        self._check(self._lib.gort_spectra_batch(self._h, M, _ptr(leaf), _ptr(soil), float(user_leaf),
                                                 float(user_soil), W, _ptr(wl), _ptr(rl), _ptr(tl), _ptr(rs)))
        return rl, tl, rs

    def soil_from_table(self, table, wavelength, n_sets=1):
        """rsoil [M][W] from a 1-nm soil table (soil_table_read): finishes the reference's -soil_spectra."""
        tab = _np(table, (SOIL_TABLE_NW,))
        wl = _np(wavelength).ravel()
        out = np.empty((n_sets, wl.shape[0]))
        self._check(self._lib.gort_soil_from_table(self._h, _ptr(tab), n_sets, wl.shape[0], _ptr(wl), _ptr(out)))
        return out

    def prospect(self, leaf):
        leaf = _np(leaf)
        M = leaf.shape[1]
        r = np.empty((M, PROSPECT_NW)); t = np.empty((M, PROSPECT_NW))
        self._check(self._lib.gort_prospect_batch(self._h, M, _ptr(leaf), _ptr(r), _ptr(t)))
        return r, t

    def _prep(self, structure, lut, angles, rleaf, tleaf, rsoil):
        st = _np(structure)
        M = st.shape[1]
        lut = _np(lut, (M, LUT_STRIDE))
        ang = _np(angles)
        assert ang.ndim in (2, 3) and ang.shape[0] == 4
        geom_per_set = ang.ndim == 3
        if geom_per_set:
            assert ang.shape[1] == M
        G = ang.shape[-1]
        rl, tl, rs = _np(rleaf), _np(tleaf), _np(rsoil)
        spectra_per_set = rl.ndim == 2
        if spectra_per_set:
            assert rl.shape[0] == M
        W = rl.shape[-1]
        return st, lut, ang, rl, tl, rs, M, G, W, geom_per_set, spectra_per_set

    def brdf(self, structure, lut, angles, rleaf, tleaf, rsoil, beta=None, fd=None,
             want_scomp=False, want_kprop=False, out=None):
        """angles [4][G] (shared) or [4][M][G]; spectra [W] (shared) or [M][W].
        Returns rsurf [M][G][W] (+ scomp [M][G][W][4], kprop [M][G][4] when requested)."""
        st, lut, ang, rl, tl, rs, M, G, W, gps, sps = self._prep(structure, lut, angles, rleaf, tleaf, rsoil)
        sh = self._shape(M, G, W, gps, sps, beta, fd)
        rsurf = out if out is not None else np.empty((M, G, W))
        scomp = np.empty((M, G, W, 4)) if want_scomp else None
        kprop = np.empty((M, G, 4)) if want_kprop else None
        self._check(self._lib.gort_brdf_batch(self._h, C.byref(sh), _ptr(st), _ptr(lut), _ptr(ang), _ptr(rl),
                                              _ptr(tl), _ptr(rs), _ptr(rsurf), _ptr(scomp), _ptr(kprop)))
        res = (rsurf,)
        if want_scomp:
            res += (scomp,)
        if want_kprop:
            res += (kprop,)
        return res if len(res) > 1 else rsurf

    def forward(self, structure, leaf, soil, wavelength, angles, method=LUT_FULL, user_leaf=-1.0, user_soil=-1.0,
                beta=None, fd=None, out=None, want_lut=False):
        """Ensemble forward operator (gort_forward_batch): structure [6][M], leaf [7][M], soil [4][M], wavelength [W],
        angles [4][G] or [4][M][G] -> rsurf [M][G][W] (+ LUT records [M][184] with want_lut); LUTs and spectra stay
        on the GPU."""
        st = _np(structure)
        M = st.shape[1]
        leaf = None if leaf is None else _np(leaf)
        soil = None if soil is None else _np(soil)
        wl = _np(wavelength).ravel()
        ang = _np(angles)
        gps = ang.ndim == 3
        G, W = ang.shape[-1], wl.shape[0]
        sh = self._shape(M, G, W, gps, 1, beta, fd)
        rsurf = out if out is not None else np.empty((M, G, W))
        lut = np.empty((M, LUT_STRIDE)) if want_lut else None
        self._check(self._lib.gort_forward_batch(self._h, C.byref(sh), method, _ptr(st), _ptr(leaf), _ptr(soil),
                                                 float(user_leaf), float(user_soil), _ptr(wl), _ptr(ang), _ptr(rsurf), _ptr(lut)))
        return (rsurf, lut) if want_lut else rsurf

    def jacobian(self, structure, leaf, soil, wavelength, angles, param=JAC_LAI, rel_step=0.0, method=LUT_FULL,
                 user_leaf=-1.0, user_soil=-1.0, beta=None, fd=None, want_rsurf=False):
        """d rsurf / d parameter [M][G][W] by central differences through the whole chain on the GPU
        (gort_jacobian_batch); param = JAC_LAI (default), JAC_FAVD, JAC_LAMBDA, ... ; optionally rsurf as well."""
        st = _np(structure)
        M = st.shape[1]
        leaf = None if leaf is None else _np(leaf)
        soil = None if soil is None else _np(soil)
        wl = _np(wavelength).ravel()
        ang = _np(angles)
        G, W = ang.shape[-1], wl.shape[0]
        sh = self._shape(M, G, W, ang.ndim == 3, 1, beta, fd)
        jac = np.empty((M, G, W))
        rsurf = np.empty((M, G, W)) if want_rsurf else None
        self._check(self._lib.gort_jacobian_batch(self._h, C.byref(sh), method, int(param), float(rel_step), _ptr(st), _ptr(leaf),
                                                  _ptr(soil), float(user_leaf), float(user_soil), _ptr(wl), _ptr(ang),
                                                  _ptr(jac), _ptr(rsurf)))
        return (jac, rsurf) if want_rsurf else jac

    def lai_tangent(self, structure, leaf, soil, wavelength, angles, param=JAC_LAI, method=LUT_FULL,
                    user_leaf=-1.0, user_soil=-1.0, beta=None, fd=None, want_rsurf=False):
        """d rsurf / d LAI (JAC_LAI, default) or d / d favd (JAC_FAVD) [M][G][W], exact, by forward-mode tangents
        through the whole chain on the GPU (gort_lai_tangent_batch); optionally rsurf as well (the bits of forward())."""
        st = _np(structure)
        M = st.shape[1]
        leaf = None if leaf is None else _np(leaf)
        soil = None if soil is None else _np(soil)
        wl = _np(wavelength).ravel()
        ang = _np(angles)
        G, W = ang.shape[-1], wl.shape[0]
        sh = self._shape(M, G, W, ang.ndim == 3, 1, beta, fd)
        jac = np.empty((M, G, W))
        rsurf = np.empty((M, G, W)) if want_rsurf else None
        self._check(self._lib.gort_lai_tangent_batch(self._h, C.byref(sh), method, int(param), _ptr(st), _ptr(leaf),
                                                     _ptr(soil), float(user_leaf), float(user_soil), _ptr(wl), _ptr(ang),
                                                     _ptr(jac), _ptr(rsurf)))
        return (jac, rsurf) if want_rsurf else jac

    def energy(self, structure, lut, angles, rleaf, tleaf, rsoil, beta=None, fd=None):
        st, lut, ang, rl, tl, rs, M, G, W, gps, sps = self._prep(structure, lut, angles, rleaf, tleaf, rsoil)
        sh = self._shape(M, G, W, gps, sps, beta, fd)
        alb = np.empty((M, G, W)); fv = np.empty((M, G, W)); fs = np.empty((M, G, W))
        self._check(self._lib.gort_energy_batch(self._h, C.byref(sh), _ptr(st), _ptr(lut), _ptr(ang), _ptr(rl),
                                                _ptr(tl), _ptr(rs), _ptr(alb), _ptr(fv), _ptr(fs)))
        return alb, fv, fs

    # ---- sensor bands: weighted means over spectral response functions (definition: include/gort_b200.h) ----
    def brdf_band(self, structure, lut, angles, rleaf, tleaf, rsoil, weights, beta=None, fd=None):
        """brdf() averaged over bands: weights [B][W] (raw SRF values on the spectra's W columns, see band_weights)
        -> rband [M][G][B]."""
        st, lut, ang, rl, tl, rs, M, G, W, gps, sps = self._prep(structure, lut, angles, rleaf, tleaf, rsoil)
        w, B = _band_weights_arg(weights, W)
        sh = self._shape(M, G, W, gps, sps, beta, fd)
        rband = np.empty((M, G, B))
        self._check(self._lib.gort_brdf_band_batch(self._h, C.byref(sh), B, _ptr(w), _ptr(st), _ptr(lut), _ptr(ang),
                                                   _ptr(rl), _ptr(tl), _ptr(rs), _ptr(rband)))
        return rband

    def energy_band(self, structure, lut, angles, rleaf, tleaf, rsoil, weights, beta=None, fd=None):
        """energy() averaged over bands: -> albedo, favegt, fasoil each [M][G][B]."""
        st, lut, ang, rl, tl, rs, M, G, W, gps, sps = self._prep(structure, lut, angles, rleaf, tleaf, rsoil)
        w, B = _band_weights_arg(weights, W)
        sh = self._shape(M, G, W, gps, sps, beta, fd)
        out = [np.empty((M, G, B)) for _ in range(3)]
        self._check(self._lib.gort_energy_band_batch(self._h, C.byref(sh), B, _ptr(w), _ptr(st), _ptr(lut), _ptr(ang),
                                                     _ptr(rl), _ptr(tl), _ptr(rs), *[_ptr(o) for o in out]))
        return tuple(out)

    def forward_band(self, structure, leaf, soil, wavelength, weights, angles, method=LUT_FULL, user_leaf=-1.0,
                     user_soil=-1.0, beta=None, fd=None, want_lut=False):
        """forward() averaged over bands (gort_forward_band_batch): weights [B][W] on wavelength [W] -> rband [M][G][B]
        (+ LUT records [M][184] with want_lut).  Spectra are computed on the union of the bands' supports only."""
        st = _np(structure)
        M = st.shape[1]
        leaf = None if leaf is None else _np(leaf)
        soil = None if soil is None else _np(soil)
        wl = _np(wavelength).ravel()
        ang = _np(angles)
        G, W = ang.shape[-1], wl.shape[0]
        w, B = _band_weights_arg(weights, W)
        sh = self._shape(M, G, W, ang.ndim == 3, 1, beta, fd)
        rband = np.empty((M, G, B))
        lut = np.empty((M, LUT_STRIDE)) if want_lut else None
        self._check(self._lib.gort_forward_band_batch(self._h, C.byref(sh), method, _ptr(st), _ptr(leaf), _ptr(soil),
                                                      float(user_leaf), float(user_soil), _ptr(wl), B, _ptr(w),
                                                      _ptr(ang), _ptr(rband), _ptr(lut)))
        return (rband, lut) if want_lut else rband

    # ---- device API (torch CUDA tensors, float64, contiguous; enqueue only) ----
    def lut_dev(self, structure, out, method=LUT_FULL, stream=None):
        M = structure.shape[1]
        self._check(self._lib.gort_lut_batch_dev(self._h, stream, M, _ptr(structure), method, _ptr(out)))

    def lut_scatter_dev(self, structure, out, dst_ptrs, method=LUT_FULL, multicast=False, stream=None):
        """lut_dev, and the producing kernels also store every row at dst_ptrs[i] (raw device addresses of the same
        block inside other tables: peer GPUs' memory mapped here, or NVSwitch multicast addresses)."""
        M = structure.shape[1]
        arr = (C.c_void_p * max(1, len(dst_ptrs)))(*[int(a) for a in dst_ptrs])
        self._check(self._lib.gort_lut_batch_scatter_dev(self._h, stream, M, _ptr(structure), method, _ptr(out),
                                                         len(dst_ptrs), arr, 1 if multicast else 0))

    def lut_tangent_dev(self, structure, lut, dlut, method=LUT_FULL, stream=None):
        """LUT records into lut (the bits of lut_dev) and their favd tangent into dlut, both [M][184]."""
        M = structure.shape[1]
        self._check(self._lib.gort_lut_tangent_batch_dev(self._h, stream, M, _ptr(structure), method, _ptr(lut), _ptr(dlut)))

    def brdf_tangent_dev(self, structure, lut, dlut, angles, rleaf, tleaf, rsoil, drsurf, beta=None, fd=None, stream=None):
        """d rsurf / d favd [M][G][W] (dense) of brdf_dev's rsurf, from lut and its tangent dlut (lut_tangent_dev)."""
        M = structure.shape[1]
        G, W = angles.shape[-1], rleaf.shape[-1]
        assert tuple(drsurf.shape) == (M, G, W), "drsurf must be [M][G][W]"
        sh = self._shape(M, G, W, angles.dim() == 3, rleaf.dim() == 2, beta, fd)
        self._check(self._lib.gort_brdf_tangent_batch_dev(self._h, stream, C.byref(sh), _ptr(structure), _ptr(lut),
                                                          _ptr(dlut), _ptr(angles), _ptr(rleaf), _ptr(tleaf),
                                                          _ptr(rsoil), _ptr(drsurf)))

    def spectra_dev(self, leaf, soil, wavelength, rleaf, tleaf, rsoil, user_leaf=-1.0, user_soil=-1.0,
                    stream=None):
        M, W = rleaf.shape
        self._check(self._lib.gort_spectra_batch_dev(self._h, stream, M, _ptr(leaf), _ptr(soil), float(user_leaf),
                                                     float(user_soil), W, _ptr(wavelength), _ptr(rleaf),
                                                     _ptr(tleaf), _ptr(rsoil)))

    def brdf_dev(self, structure, lut, angles, rleaf, tleaf, rsoil, rsurf, scomp=None, kprop=None,
                 beta=None, fd=None, stream=None):
        M = structure.shape[1]
        gps = angles.dim() == 3
        sps = rleaf.dim() == 2
        G, W = angles.shape[-1], rleaf.shape[-1]
        # rsurf may be [M][G][pitch] with pitch >= W (a pitch that is a multiple of 4 keeps warp stores aligned)
        pitch = rsurf.shape[-1]
        sh = self._shape(M, G, W, gps, sps, beta, fd, out_pitch=pitch)
        self._check(self._lib.gort_brdf_batch_dev(self._h, stream, C.byref(sh), _ptr(structure), _ptr(lut),
                                                  _ptr(angles), _ptr(rleaf), _ptr(tleaf), _ptr(rsoil),
                                                  _ptr(rsurf), _ptr(scomp), _ptr(kprop)))

    def brdf_dev_bind(self, structure, lut, angles, rleaf, tleaf, rsoil, rsurf, scomp=None, kprop=None,
                      beta=None, fd=None, stream=None):
        """Same call as brdf_dev with every argument converted once: returns a zero-argument callable that
        enqueues one gort_brdf_batch_dev (a few microseconds of host time per call instead of the ctypes
        argument marshalling of brdf_dev).  The tensors are kept alive by the closure."""
        M = structure.shape[1]
        G, W = angles.shape[-1], rleaf.shape[-1]
        sh = self._shape(M, G, W, angles.dim() == 3, rleaf.dim() == 2, beta, fd, out_pitch=rsurf.shape[-1])
        keep = (structure, lut, angles, rleaf, tleaf, rsoil, rsurf, scomp, kprop, sh)
        args = (self._h, C.c_void_p(stream), C.byref(sh)) + tuple(C.c_void_p(_ptr(t)) for t in keep[:9])
        fn, check = self._lib.gort_brdf_batch_dev, self._check

        def call(_keep=keep):
            rc = fn(*args)
            if rc:
                check(rc)
        return call

    def energy_dev(self, structure, lut, angles, rleaf, tleaf, rsoil, albedo, favegt, fasoil,
                   beta=None, fd=None, stream=None):
        M = structure.shape[1]
        gps = angles.dim() == 3
        sps = rleaf.dim() == 2
        G, W = angles.shape[-1], rleaf.shape[-1]
        sh = self._shape(M, G, W, gps, sps, beta, fd)
        self._check(self._lib.gort_energy_batch_dev(self._h, stream, C.byref(sh), _ptr(structure), _ptr(lut),
                                                    _ptr(angles), _ptr(rleaf), _ptr(tleaf), _ptr(rsoil),
                                                    _ptr(albedo), _ptr(favegt), _ptr(fasoil)))

    def brdf_band_dev(self, structure, lut, angles, rleaf, tleaf, rsoil, weights, rband, beta=None, fd=None, stream=None):
        """brdf_band on device tensors: weights [B][W], rband [M][G][B].  A defective weight row gives NaN in its band."""
        M = structure.shape[1]
        G, W = angles.shape[-1], rleaf.shape[-1]
        _check_band_dims(tuple(weights.shape), W)
        assert tuple(rband.shape) == (M, G, weights.shape[0]), "rband must be [M][G][B]"
        sh = self._shape(M, G, W, angles.dim() == 3, rleaf.dim() == 2, beta, fd)
        self._check(self._lib.gort_brdf_band_batch_dev(self._h, stream, C.byref(sh), weights.shape[0], _ptr(weights),
                                                       _ptr(structure), _ptr(lut), _ptr(angles), _ptr(rleaf),
                                                       _ptr(tleaf), _ptr(rsoil), _ptr(rband)))

    def energy_band_dev(self, structure, lut, angles, rleaf, tleaf, rsoil, weights, albedo, favegt, fasoil,
                        beta=None, fd=None, stream=None):
        M = structure.shape[1]
        G, W = angles.shape[-1], rleaf.shape[-1]
        _check_band_dims(tuple(weights.shape), W)
        for o in (albedo, favegt, fasoil):
            assert tuple(o.shape) == (M, G, weights.shape[0]), "outputs must be [M][G][B]"
        sh = self._shape(M, G, W, angles.dim() == 3, rleaf.dim() == 2, beta, fd)
        self._check(self._lib.gort_energy_band_batch_dev(self._h, stream, C.byref(sh), weights.shape[0], _ptr(weights),
                                                         _ptr(structure), _ptr(lut), _ptr(angles), _ptr(rleaf),
                                                         _ptr(tleaf), _ptr(rsoil), _ptr(albedo), _ptr(favegt),
                                                         _ptr(fasoil)))


def _check_band_dims(shape, W):
    """weights must be [B][W] on the call's grid with 1 <= B <= MAX_BANDS: the library reads B * W doubles"""
    if len(shape) != 2 or shape[1] != W or not 1 <= shape[0] <= MAX_BANDS:
        raise ValueError("band weights must be [B][W] with W = %d columns of the call's grid and 1 <= B <= %d, got %s"
                         % (W, MAX_BANDS, shape))


def _band_weights_arg(weights, W):
    w = _np(weights)
    _check_band_dims(w.shape, W)
    return w, w.shape[0]


def band_weights(grid, srf_wavelength, srf_response):
    """Band weights for a call's wavelength grid from tabulated spectral response functions: each SRF is linearly
    interpolated onto `grid` [W], zero outside its table.  srf_wavelength [n] (ascending) and srf_response [n] give one
    band; srf_response [B][n] with a shared srf_wavelength, or lists of per-band tables, give B bands.  Returns [B][W]
    raw weights (the library normalises them).  Host only."""
    grid = np.asarray(grid, dtype=np.float64).ravel()

    def tables(a):
        # one table [n], equal-length tables [B][n], or a list of tables of different lengths
        try:
            a = np.asarray(a, dtype=np.float64)
        except ValueError:
            return [np.asarray(t, dtype=np.float64).ravel() for t in a]
        return [a] if a.ndim == 1 else list(a)

    resp = tables(srf_response)
    wls = tables(srf_wavelength)
    if len(wls) == 1:
        wls = wls * len(resp)
    if len(wls) != len(resp):
        raise ValueError("band_weights: %d wavelength tables for %d responses" % (len(wls), len(resp)))
    rows = []
    for x, y in zip(wls, resp):
        x = np.asarray(x, dtype=np.float64).ravel()
        y = np.asarray(y, dtype=np.float64).ravel()
        if x.shape != y.shape or x.size < 1 or np.any(np.diff(x) <= 0):
            raise ValueError("band_weights: an SRF table needs matching, strictly ascending wavelengths")
        rows.append(np.interp(grid, x, y, left=0.0, right=0.0))
    return np.stack(rows)


# ---- LUT text files ("-W" / "-P", gortt.c:123-146) ------------------------------------------------
def lut_write_text(lut_record, path):
    """Write one LUT record in the reference's "-W" layout using the library's formatter."""
    lib = load_library()
    rec = _np(lut_record, (LUT_STRIDE,))
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
    libc.fclose.argtypes = [C.c_void_p]
    fp = libc.fopen(os.fsencode(path), b"w")
    if not fp:
        raise GortError(5, "cannot open %s" % path)
    n = lib.gort_lut_write_text(_ptr(rec), fp)
    libc.fclose(fp)
    if n < 0:
        raise GortError(-n, "write failed")
    return n


def lut_read_text(path):
    lib = load_library()
    rec = np.zeros(LUT_STRIDE)
    rc = lib.gort_lut_read_text(os.fsencode(path), _ptr(rec))
    if rc != 0:
        raise GortError(rc, "cannot read %s" % path)
    return rec


def soil_table_read(path):
    """"wavelength albedo" text file -> 1-nm table [2101] (the reference's own interpolation, gortt.c:1420-1428).
    Raises GortError(5, <the reference's message>) on a malformed file."""
    lib = load_library()
    tab = np.empty(SOIL_TABLE_NW)
    err = C.create_string_buffer(600)
    rc = lib.gort_soil_table_read(os.fsencode(path), _ptr(tab), err, 600)
    if rc != 0:
        raise GortError(rc, err.value.decode())
    return tab


def structure_from_options(lambda_=0.405, r=0.76, b=None, h1=3.0, h2=8.5, favd=0.858,
                           hb=None, br=None, pcc=None, lai=None):
    """Host-side mirror of the reference CLI's structure derivation (defaults gortt.c:67-72; float-typed
    -HB/-BR/-PCC/-LAI gortt.c:1014,1032-1036; derivation gortt.c:1117-1131). Returns [lambda,r,b,h1,h2,favd]."""
    if b is None:
        b = 3.55263 * r
    if hb is not None or br is not None or pcc is not None:
        hb = np.float32(2.0 if hb is None else hb)
        br = np.float32(1.0 if br is None else br)
        pcc = np.float32(0.5 if pcc is None else pcc)
        r = 10.0
        b = float(br) * r
        h1 = b * 2.0
        h2 = float(hb) * b + h1
        lambda_ = float(pcc) / (r * r * np.pi)
    if lai is not None:
        lai = float(np.float32(lai))
        favd = lai * 3.0 / (lambda_ * r * r * np.pi * b * 4.0)
    return np.array([lambda_, r, b, h1, h2, favd], dtype=np.float64)
