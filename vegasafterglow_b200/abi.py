"""ctypes / numpy mirror of ``include/vag.h``.

``PARAMS_DTYPE`` is the numpy structured dtype of ``vag_params`` (one record = one parameter set =
everything the reference's ``Model.__init__`` receives, pybind/pybind.cpp:384-422).  A batch of
models is a 1-D array of this dtype; its bytes are what crosses the C ABI.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

VAG_OK, VAG_ERR_INVALID, VAG_ERR_CUDA, VAG_ERR_UNSUPPORTED, VAG_ERR_CAPACITY = range(5)
JET_TOPHAT, JET_GAUSSIAN, JET_POWERLAW, JET_TWO_COMPONENT, JET_STEP_POWERLAW, JET_POWERLAW_WING = 0, 1, 2, 3, 4, 5
MEDIUM_ISM, MEDIUM_WIND = 0, 1
NCOMP = 5
COMPONENTS = ("total", "fwd_sync", "fwd_ssc", "rvs_sync", "rvs_ssc")
ST_ODE_STEP_CAP, ST_ODE_STALLED, ST_ODE_FAIL500, ST_GRID_NONFINITE, ST_CAPACITY, ST_IC_BAND = 1, 2, 4, 8, 16, 32
ST_INVALID = 64  # rejected by the parameter checks of the device-planned entry points (vag_chi2_dev, vag_flux_band_dev)

RADIATION_DTYPE = np.dtype(
    [("eps_e", "f8"), ("eps_B", "f8"), ("p", "f8"), ("xi_e", "f8"), ("ssc", "i4"), ("kn", "i4")], align=True
)

PARAMS_DTYPE = np.dtype(
    [
        ("jet_type", "i4"),
        ("spreading", "i4"),
        ("theta_c", "f8"),
        ("E_iso", "f8"),
        ("Gamma0", "f8"),
        ("k_e", "f8"),
        ("k_g", "f8"),
        ("duration", "f8"),
        ("theta_w", "f8"),
        ("E_iso_w", "f8"),
        ("Gamma0_w", "f8"),
        ("sigma0", "f8"),
        ("medium_type", "i4"),
        ("pad0_", "i4"),
        ("n_ism", "f8"),
        ("A_star", "f8"),
        ("n0", "f8"),
        ("lumi_dist", "f8"),
        ("z", "f8"),
        ("theta_obs", "f8"),
        ("phi_obs", "f8"),
        ("fwd", RADIATION_DTYPE),
        ("rvs", RADIATION_DTYPE),
        ("has_rvs", "i4"),
        ("axisymmetric", "i4"),
        ("radiative_fireball", "i4"),
        ("pad1_", "i4"),
        ("phi_resol", "f8"),
        ("theta_resol", "f8"),
        ("t_resol", "f8"),
        ("rtol", "f8"),
        ("has_magnetar", "i4"),
        ("pad2_", "i4"),
        ("magnetar_L0", "f8"),
        ("magnetar_t0", "f8"),
        ("magnetar_q", "f8"),
        ("wind_k_m", "f8"),
    ],
    align=True,
)

GRID_INFO_DTYPE = np.dtype(
    [
        ("n_phi", "i4"),
        ("n_theta", "i4"),
        ("n_t", "i4"),
        ("n_reps", "i4"),
        ("symmetry", "i4"),
        ("phi_mirrored", "i4"),
        ("n_phi_eff", "i4"),
        ("status", "i4"),
    ],
    align=True,
)



class BandObs(C.Structure):
    """``vag_band_obs`` (include/vag.h): one band-integrated data set of the likelihood."""

    _fields_ = [("t", C.c_void_p), ("lnF_obs", C.c_void_p), ("sigma_ln", C.c_void_p), ("w", C.c_void_p), ("n", C.c_size_t),
                ("nu_min", C.c_double), ("nu_max", C.c_double), ("num_nu", C.c_size_t)]


class SeriesSet(C.Structure):
    """``vag_series_set`` (include/vag.h): one data set of a ragged series request, a slice of the concatenated points."""

    _fields_ = [("offset", C.c_size_t), ("n", C.c_size_t)]


class MultiSet(C.Structure):
    """``vag_multi_set`` (include/vag.h): one data set of ``vag_chi2_multi_bands`` -- a slice of the concatenated points
    (n = 0: none) and its band-integrated data ``bands[band0 .. band0 + n_bands)``."""

    _fields_ = [("offset", C.c_size_t), ("n", C.c_size_t), ("band0", C.c_size_t), ("n_bands", C.c_size_t)]


class GridSet(C.Structure):
    """``vag_grid_set`` (include/vag.h): one (t x nu) grid of a per-model grid request -- a slice of the concatenated
    times and one of the concatenated frequencies."""

    _fields_ = [("t0", C.c_size_t), ("n_t", C.c_size_t), ("nu0", C.c_size_t), ("n_nu", C.c_size_t)]


c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)


def upgrade_params(old) -> np.ndarray:
    """Records written with an earlier (shorter) ``vag_params`` layout -> the current one: fields are copied by
    name, new fields keep their defaults (committed fixtures stay valid when the struct grows)."""
    old = np.asarray(old)
    if old.dtype == PARAMS_DTYPE:
        return old
    new = default_params(old.size).reshape(old.shape)
    for name in old.dtype.names:
        if name in PARAMS_DTYPE.names:
            new[name] = old[name]
    return new


def default_params(n: int = 1) -> np.ndarray:
    """``n`` records initialised with the reference defaults (pybind/pybind.cpp:419-422)."""
    p = np.zeros(n, dtype=PARAMS_DTYPE)
    p["k_e"] = 2.0
    p["k_g"] = 2.0
    p["theta_w"], p["E_iso_w"], p["Gamma0_w"] = 0.3, 1e50, 50.0
    p["duration"] = 1.0
    p["n0"] = np.inf
    p["fwd"]["xi_e"] = 1.0
    p["rvs"]["xi_e"] = 1.0
    p["fwd"]["eps_e"], p["fwd"]["eps_B"], p["fwd"]["p"] = 0.1, 0.01, 2.3
    p["rvs"]["eps_e"], p["rvs"]["eps_B"], p["rvs"]["p"] = 0.1, 0.01, 2.3
    p["axisymmetric"] = 1
    p["wind_k_m"] = 2.0
    p["radiative_fireball"] = 1
    p["phi_resol"] = p["theta_resol"] = p["t_resol"] = 0.0  # <=0 -> reference defaults
    p["rtol"] = 0.0
    return p


def as_ptr(a: np.ndarray, typ=c_double_p):
    return a.ctypes.data_as(typ)
