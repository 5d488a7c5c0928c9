"""gort_b200 -- B200-native GORT forest BRDF / albedo forward operator.

The product is the C-ABI shared library `libgort_b200.so` (CUDA kernels for sm_100a, declared in
include/gort_b200.h) plus the C `gortt` command line; this package is the thin ctypes host binding.
"""
from .api import (Gort, GortError, PinnedArray, LUT_FULL, LUT_Q08, LUT_STRIDE, NTH, PROSPECT_NW,  # noqa: F401
                  load_library, lut_read_text, lut_write_text, soil_table_read, structure_from_options, ABI_SYMBOLS,
                  SOIL_TABLE_NW, JAC_LAMBDA, JAC_R, JAC_B, JAC_H1, JAC_H2, JAC_FAVD, JAC_LAI, MAX_BANDS, band_weights)
