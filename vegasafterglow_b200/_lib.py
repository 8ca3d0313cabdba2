"""Loader of the C-ABI library ``libvag_b200.so`` (include/vag.h).  There is deliberately no
fallback: if the CUDA library is missing or no GPU is usable the product raises."""
from __future__ import annotations

import ctypes as C
import os

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VAG_LIB_PATH") or os.path.join(_HERE, "libvag_b200.so")  # override: A/B experiments only
_lib = None


class VagError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). vegasafterglow_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    lib.vag_last_error.restype = C.c_char_p
    lib.vag_version.restype = C.c_char_p
    vp, sz, dp, ip = C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p
    lib.vag_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.vag_destroy.argtypes = [vp]
    lib.vag_params_validate.argtypes = [vp]
    lib.vag_params_default.argtypes = [vp]
    lib.vag_flux_density_grid.argtypes = [vp, vp, sz, dp, sz, dp, sz, dp, ip]
    lib.vag_flux_density_series.argtypes = [vp, vp, sz, dp, dp, sz, dp, ip]
    lib.vag_flux_density_exposures.argtypes = [vp, vp, sz, dp, dp, dp, sz, sz, dp, ip]
    lib.vag_flux_band.argtypes = [vp, vp, sz, dp, sz, C.c_double, C.c_double, sz, dp, ip]
    lib.vag_chi2_series.argtypes = [vp, vp, sz, dp, dp, dp, dp, dp, sz, dp, ip]
    lib.vag_flux_density_grid_dev.argtypes = [vp, vp, sz, dp, sz, dp, sz, dp, ip, vp]
    lib.vag_flux_density_series_dev.argtypes = [vp, vp, sz, dp, dp, sz, dp, ip, vp]
    lib.vag_chi2_series_dev.argtypes = [vp, vp, sz, dp, dp, dp, dp, dp, sz, dp, ip, vp]
    lib.vag_synchronize.argtypes = [vp]
    lib.vag_set_capacity.argtypes = [vp, C.c_int, C.c_int]
    lib.vag_set_profiling.argtypes = [vp, C.c_int]
    lib.vag_set_output_mode.argtypes = [vp, C.c_int]
    lib.vag_last_stage_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.vag_last_launch_count.argtypes = [vp]
    lib.vag_measure_fp64_peak.argtypes = [vp, C.POINTER(C.c_double)]
    lib.vag_selftest_libm.argtypes = [vp, C.c_int, dp, dp, dp, sz]
    lib.vag_chi2.argtypes = [vp, vp, sz, dp, dp, dp, dp, dp, sz, vp, sz, dp, ip]
    lib.vag_chi2_ext.argtypes = [vp, vp, sz, dp, dp, dp, dp, dp, dp, sz, dp, vp, sz, dp, ip]
    lib.vag_params_validate_batch.argtypes = [vp, sz, ip]
    lib.vag_params_validate_batch_dev.argtypes = [vp, vp, sz, ip, C.POINTER(C.c_int), vp]
    lib.vag_flux_band_dev.argtypes = [vp, vp, sz, dp, sz, C.c_double, C.c_double, sz, dp, ip, vp]
    lib.vag_chi2_dev.argtypes = [vp, vp, sz, dp, dp, dp, dp, dp, dp, sz, dp, vp, sz, dp, ip, vp]
    lib.vag_flux_density_series_multi.argtypes = [vp, vp, sz, ip, vp, sz, dp, dp, sz, dp, ip]
    lib.vag_chi2_multi.argtypes = [vp, vp, sz, ip, vp, sz, dp, dp, dp, dp, dp, dp, sz, dp, dp, ip]
    lib.vag_flux_band_multi.argtypes = [vp, vp, sz, ip, vp, sz, dp, ip]
    lib.vag_chi2_multi_bands.argtypes = [vp, vp, sz, ip, vp, sz, dp, dp, dp, dp, dp, dp, sz, dp, vp, sz, dp, ip]
    lib.vag_chi2_multi_bands_exposures.argtypes = [vp, vp, sz, ip, vp, sz, dp, dp, dp, dp, dp, dp, sz, dp, dp, ip, vp, sz,
                                                   dp, ip]
    lib.vag_chi2_multi_bands_dev.argtypes = [vp, vp, sz, ip, vp, sz, dp, dp, dp, dp, dp, dp, sz, dp, vp, sz, dp, ip, vp]
    lib.vag_flux_density_grid_multi.argtypes = [vp, vp, sz, ip, vp, sz, dp, sz, dp, sz, dp, ip]
    lib.vag_flux_quantiles_multi.argtypes = [vp, vp, sz, ip, vp, sz, dp, sz, dp, sz, dp, sz, dp, vp, ip]
    lib.vag_debug_set_ode_limits.argtypes = [vp, C.c_int, C.c_int]
    lib.vag_last_total_alias.argtypes = [vp]
    lib.vag_set_series_mode.argtypes = [vp, C.c_int]
    lib.vag_set_grid_lanes.argtypes = [vp, C.c_int]
    lib.vag_last_work.argtypes = [vp, C.POINTER(C.c_double)]
    lib.vag_details.argtypes = [vp, vp, C.c_double, C.c_double, vp, dp, dp, ip, dp, dp, dp, ip]
    lib.vag_details_photons.argtypes = [vp, vp, C.c_double, C.c_double, dp, dp]
    lib.vag_details_ic.argtypes = [vp, vp, C.c_double, C.c_double, dp, dp]
    _lib = lib
    return lib


EXPORTS = [
    "vag_params_default", "vag_params_validate", "vag_create", "vag_destroy", "vag_last_error", "vag_version",
    "vag_flux_density_grid", "vag_flux_density_series", "vag_flux_band", "vag_chi2_series", "vag_flux_density_grid_dev",
    "vag_flux_density_series_dev", "vag_chi2_series_dev", "vag_synchronize", "vag_set_capacity", "vag_details", "vag_details_photons",
    "vag_set_profiling", "vag_set_output_mode", "vag_last_stage_ms", "vag_last_launch_count", "vag_measure_fp64_peak", "vag_selftest_libm", "vag_chi2", "vag_params_validate_batch", "vag_debug_set_ode_limits", "vag_last_total_alias", "vag_last_work", "vag_set_series_mode", "vag_details_ic",
    "vag_set_grid_lanes", "vag_chi2_ext", "vag_params_validate_batch_dev", "vag_flux_band_dev", "vag_chi2_dev",
    "vag_flux_density_series_multi", "vag_chi2_multi", "vag_flux_band_multi", "vag_chi2_multi_bands",
    "vag_chi2_multi_bands_dev", "vag_flux_density_grid_multi", "vag_flux_quantiles_multi", "vag_flux_density_exposures",
    "vag_chi2_multi_bands_exposures",
]


def check(rc):
    if rc != abi.VAG_OK:
        msg = load().vag_last_error().decode()
        if rc in (abi.VAG_ERR_INVALID,):
            raise ValueError(msg)
        if rc == abi.VAG_ERR_UNSUPPORTED:
            raise NotImplementedError(msg)
        raise VagError(rc, msg)
