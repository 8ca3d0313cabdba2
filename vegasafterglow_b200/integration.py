"""Sampler-side integration with the reference's ``Fitter`` (VegasAfterglow/fitting): the GPU batch evaluator that
replaces the thread pool of ``fit_emcee`` / ``fit_bilby`` (fitting/samplers.py:33-125,128-197).

The reference evaluates one walker per host thread: ``pool.map(eval_one, valid_samples)`` builds a ``Model`` per walker
(``Fitter._build_model``, fitter.py:455-495) and sums its chi-squared (``Fitter._evaluate``, :503-533).  Here the same
``Fitter`` object -- its data, configuration flags and parameter transformer are used as they are -- is evaluated for a
whole ensemble in ONE call of the C ABI (``vag_chi2``, or ``vag_chi2_ext`` with a built-in extinction law and a per-walker
``A_V``): point data + band-integrated data, on one GPU or partitioned by walker over the GPUs of the box
(vegasafterglow_b200/parallel.py).

* ``params_from_fitter(fitter, model_params)``   ModelParams namespaces -> ``vag_params`` records (what ``_build_model`` +
                                                 the default jet / medium factories, fitting/utils.py:31-70, construct)
* ``GpuFitterEvaluator(fitter, engine)``         ``chi2(thetas[n, ndim]) -> chi2[n]`` and ``log_likelihoods(...)``
* ``log_prob_batch_gpu(...)``                    the drop-in for ``log_prob_batch`` of ``fit_emcee`` (samplers.py:72-91)
* ``GpuMapPool(evaluator, log_likelihood_fn)``   a ``pool`` whose ``map`` evaluates dynesty's queue of live-point
                                                 proposals as one batch (dynesty's documented ``pool.map(loglike, queue)``
                                                 protocol; samplers.py:179-183 sets ``use_pool={"loglikelihood": True}``)
* ``integration/samplers_gpu.patch``             the same, as a patch to the reference's samplers.py
                                                 (tests/test_integration_patch.py applies it to a copy and runs it)

Custom (callable) jets / media and custom extinction laws are host callbacks and stay on the reference's CPU path:
``GpuFitterEvaluator`` refuses them loudly.
"""
from __future__ import annotations

import math
from typing import Callable, Sequence

import numpy as np

from . import abi
from .fitting import _ensemble_chi2, band_obs

_JET_CODE = {"tophat": abi.JET_TOPHAT, "uniform": abi.JET_TOPHAT, "gaussian": abi.JET_GAUSSIAN,
             "powerlaw": abi.JET_POWERLAW, "two_component": abi.JET_TWO_COMPONENT,
             "step_powerlaw": abi.JET_STEP_POWERLAW, "powerlaw_wing": abi.JET_POWERLAW_WING}
# jet parameters each registry entry passes to its constructor (fitting/config.py:99-121)
_JET_PARAMS = {"tophat": ("theta_c", "E_iso", "Gamma0"), "gaussian": ("theta_c", "E_iso", "Gamma0"),
               "powerlaw": ("theta_c", "E_iso", "Gamma0", "k_e", "k_g"),
               "two_component": ("theta_c", "E_iso", "Gamma0", "theta_w", "E_iso_w", "Gamma0_w"),
               "step_powerlaw": ("theta_c", "E_iso", "Gamma0", "E_iso_w", "Gamma0_w", "k_e", "k_g"),
               "powerlaw_wing": ("theta_c", "E_iso_w", "Gamma0_w", "k_e", "k_g"), "uniform": ("E_iso", "Gamma0")}
_LN10_OVER_2P5 = math.log(10.0) / 2.5


def params_from_fitter(fitter, model_params: Sequence) -> np.ndarray:
    """``vag_params`` records of ``Fitter._build_model(p)`` for every ModelParams-like namespace ``p``."""
    if getattr(fitter, "_custom_jet", False) or getattr(fitter, "_custom_medium", False):
        raise NotImplementedError("custom (callable) jet / medium factories are host callbacks: use the reference's CPU path")
    jet, medium = fitter.jet, fitter.medium
    if jet not in _JET_CODE:
        raise ValueError(f"Unknown jet type: {jet}")
    if medium not in ("ism", "wind"):
        raise ValueError(f"Unknown medium type: {medium}")
    n = len(model_params)
    P = abi.default_params(n)
    P["jet_type"] = _JET_CODE[jet]
    P["spreading"] = 0  # _default_jet_factory: kwargs["spreading"] = False (fitting/utils.py:44)
    get = lambda name, default=None: np.array([getattr(p, name, default) for p in model_params], dtype=np.float64)  # noqa: E731
    for name in _JET_PARAMS[jet]:
        P[name] = get(name)
    if jet == "uniform":
        P["theta_c"] = math.pi / 2
    P["duration"] = get("tau", 1.0)
    if fitter.magnetar and jet != "powerlaw_wing":
        P["has_magnetar"] = 1
        P["magnetar_L0"], P["magnetar_t0"], P["magnetar_q"] = get("L0"), get("t0"), get("q")
    if medium == "ism":
        P["medium_type"], P["n_ism"] = abi.MEDIUM_ISM, get("n_ism")
    else:
        P["medium_type"] = abi.MEDIUM_WIND
        P["A_star"], P["n_ism"], P["n0"], P["wind_k_m"] = get("A_star"), get("n_ism", 0.0), get("n0", math.inf), get("k_m", 2.0)
    P["lumi_dist"], P["z"], P["theta_obs"] = fitter.lumi_dist, fitter.z, get("theta_v")
    P["fwd"]["eps_e"], P["fwd"]["eps_B"], P["fwd"]["p"], P["fwd"]["xi_e"] = get("eps_e"), get("eps_B"), get("p"), get("xi_e", 1.0)
    P["fwd"]["ssc"], P["fwd"]["kn"] = int(bool(fitter.fwd_ssc)), int(bool(fitter.kn))
    if fitter.rvs_shock:
        P["has_rvs"] = 1
        P["rvs"]["eps_e"], P["rvs"]["eps_B"], P["rvs"]["p"] = get("eps_e_r"), get("eps_B_r"), get("p_r")
        P["rvs"]["xi_e"] = get("xi_e_r", 1.0)
        P["rvs"]["ssc"], P["rvs"]["kn"] = int(bool(fitter.rvs_ssc)), int(bool(fitter.kn))
    if fitter.resolution is not None:
        P["phi_resol"], P["theta_resol"], P["t_resol"] = fitter.resolution
    P["rtol"] = fitter.rtol if fitter.rtol is not None else 0.0
    P["radiative_fireball"] = 1 if fitter.radiative_fireball else 0
    return P


class GpuFitterEvaluator:
    """chi-squared of a whole ensemble for a reference ``Fitter`` (its data, flags and transformer), on the GPU."""

    def __init__(self, fitter, engine, distributed: bool = False):
        if getattr(fitter, "_custom_extinction", False):
            raise NotImplementedError("custom extinction laws are host callbacks: use the reference's CPU path")
        fitter._consolidate_data()
        if fitter._to_params is None:
            raise ValueError("the Fitter has no parameter transformer yet (call validate / fit first)")
        self.fitter, self.engine, self.distributed = fitter, engine, distributed
        self.has_points = len(fitter._all_t) > 0
        self.points = ((fitter._all_t, fitter._all_nu, fitter._all_log_flux, fitter._all_log_err, fitter._all_weights)
                       if self.has_points else None)
        self.bands = [band_obs(bd.t, bd.flux, bd.err, bd.nu_min, bd.nu_max, bd.num_points, bd.weights) for bd in fitter._band_obs]
        # built-in host extinction: F -> F exp(-A_V k(lambda)) is a shift of ln F_obs per point (fitter.py:512-519),
        # ln F_obs - ln(F e^{-A_V k}) = (ln F_obs + A_V k) - ln F, with a walker-dependent A_V.  Without point data
        # there is nothing to shift.
        self.ext_kernel = fitter._ext_kernel if fitter._ext_law is not None and self.has_points else None

    def chi2(self, thetas: np.ndarray) -> np.ndarray:
        thetas = np.atleast_2d(np.asarray(thetas, dtype=np.float64))
        mp = [self.fitter._to_params(th) for th in thetas]
        A_V = None
        if self.ext_kernel is not None:
            A_V = np.array([getattr(p, "A_V", 0.0) for p in mp], dtype=np.float64)
        # the cost proxy of the distributed split spans the point times, or the first band's without points
        window = (self.points[0] if self.has_points else self.bands[0]["t"]) if self.distributed else None
        P = params_from_fitter(self.fitter, mp)
        return _ensemble_chi2(self.engine, P, self.points, self.bands, self.ext_kernel, A_V, window)

    def log_likelihoods(self, thetas, log_likelihood_fn: Callable) -> np.ndarray:
        chi2 = self.chi2(thetas)
        with np.errstate(all="ignore"):
            ll = np.where(np.isfinite(chi2), np.asarray([log_likelihood_fn(c) if np.isfinite(c) else -np.inf for c in chi2]), -np.inf)
        ll[~np.isfinite(ll)] = -np.inf
        return ll


def log_prob_batch_gpu(evaluator: GpuFitterEvaluator, labels, pl, pu, prior_dict, log_likelihood_fn: Callable):
    """Drop-in for the ``log_prob_batch`` closure of ``fit_emcee`` (samplers.py:72-91): same bounds test, same prior
    sum, the likelihoods of all in-bounds walkers from ONE GPU batch instead of ``pool.map(eval_one, ...)``."""

    def log_prob_batch(samples: np.ndarray) -> np.ndarray:
        in_bounds = np.all((samples >= pl) & (samples <= pu), axis=1)
        log_probs = np.full(samples.shape[0], -np.inf)
        valid_indices = np.where(in_bounds)[0]
        if len(valid_indices) > 0:
            valid_array = np.asarray(samples[valid_indices], dtype=np.float64)
            log_likes = evaluator.log_likelihoods(valid_array, log_likelihood_fn)
            log_prior = np.zeros(len(valid_indices))
            for i, name in enumerate(labels):
                log_prior += prior_dict[name].ln_prob(valid_array[:, i])
            log_probs[valid_indices] = log_likes + log_prior
        return log_probs

    return log_prob_batch


class GpuMapPool:
    """``pool`` for dynesty (through bilby, samplers.py:160-183): ``map(fn, queue)`` evaluates the queued parameter
    vectors as ONE GPU batch.  ``fn`` is the sampler's per-point log-likelihood wrapper; it is only used as a fallback
    for items that are not plain parameter vectors of the expected length."""

    def __init__(self, evaluator: GpuFitterEvaluator, log_likelihood_fn: Callable, ndim: int):
        self.evaluator, self.log_likelihood_fn, self.ndim = evaluator, log_likelihood_fn, ndim
        self.size = 1

    def map(self, fn, iterable):
        items = list(iterable)
        try:
            arr = np.asarray(items, dtype=np.float64)
            if arr.ndim == 2 and arr.shape[1] == self.ndim:
                return list(self.evaluator.log_likelihoods(arr, self.log_likelihood_fn))
        except (TypeError, ValueError):
            pass
        return [fn(x) for x in items]

    def close(self):
        pass

    def join(self):
        pass

    def shutdown(self, wait=True):
        pass
