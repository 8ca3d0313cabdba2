"""Batched likelihood: the drop-in for ``log_prob_batch`` of the reference's emcee driver
(VegasAfterglow/fitting/samplers.py:72-91) and for ``Fitter._evaluate`` (fitter.py:503-533).

The reference evaluates each walker on a host thread (``pool.map(eval_one, valid_samples)``);
here the whole ensemble goes to the GPU as ONE batch of ``vag_params`` records, and -- when
``torch.distributed`` is initialised -- the batch is partitioned by walker across the ranks and
only the float64[n_walkers] log-likelihood vector is gathered (vegasafterglow_b200/parallel.py).

Same data conventions as the reference (fitter.py:407-437): points sorted by time, weights
normalised to sum N, ln-flux chi-squared, non-finite chi2 -> logL = -inf.
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence

import numpy as np

from . import abi

# sampler-space parameter name -> (record field path, ) for the typed jet/medium variants
# (fitting/config.py:99-137 registries; Fitter._build_model fitter.py:455-495)
_FIELDS = {
    "theta_c": ("theta_c",), "E_iso": ("E_iso",), "Gamma0": ("Gamma0",), "k_e": ("k_e",), "k_g": ("k_g",),
    "duration": ("duration",), "tau": ("duration",), "theta_w": ("theta_w",), "E_iso_w": ("E_iso_w",),
    "Gamma0_w": ("Gamma0_w",), "sigma0": ("sigma0",), "n_ism": ("n_ism",), "A_star": ("A_star",), "n0": ("n0",),
    "theta_v": ("theta_obs",), "eps_e": ("fwd", "eps_e"), "eps_B": ("fwd", "eps_B"), "p": ("fwd", "p"),
    "xi_e": ("fwd", "xi_e"), "eps_e_r": ("rvs", "eps_e"), "eps_B_r": ("rvs", "eps_B"), "p_r": ("rvs", "p"),
    "xi_e_r": ("rvs", "xi_e"),
}


def time_order(t):
    """The stable time sort of the point data (fitter.py:407-437); per-point columns follow it."""
    return np.argsort(np.asarray(t, dtype=np.float64).reshape(-1), kind="stable")


def consolidate_data(t, nu, flux, err, weights=None):
    """fitter.py:407-437: sort by time, normalise weights to sum N, ln-flux and relative error."""
    t, nu, flux, err = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (t, nu, flux, err))
    w = np.ones_like(t) if weights is None else np.asarray(weights, dtype=np.float64).reshape(-1)
    if np.any(flux <= 0) or np.any(err <= 0):
        raise ValueError("flux and err must be positive")
    order = time_order(t)
    t, nu, flux, err, w = t[order], nu[order], flux[order], err[order], w[order]
    if w.sum() > 0:
        w = w * (len(w) / w.sum())
    return t, nu, np.log(flux), err / flux, w


def band_obs(t, flux, err, nu_min, nu_max, num_points=5, weights=None):
    """One band-integrated data set in the form ``Engine.chi2`` takes (fitter.py BandObs + :525-531: ln flux,
    relative error, weights as given -- the reference normalises only the point-data weights)."""
    t, flux, err = (np.asarray(a, dtype=np.float64).reshape(-1) for a in (t, flux, err))
    w = np.ones_like(t) if weights is None else np.asarray(weights, dtype=np.float64).reshape(-1)
    if np.any(flux <= 0) or np.any(err <= 0):
        raise ValueError("the log-flux likelihood requires strictly positive fluxes and errors")
    order = np.argsort(t, kind="stable")
    return {"t": t[order], "lnF_obs": np.log(flux[order]), "sigma_ln": err[order] / flux[order], "w": w[order],
            "nu_min": float(nu_min), "nu_max": float(nu_max), "num_nu": int(num_points)}


def _chi2_batch(engine, P, points, bands, ext_kernel=None, A_V=None, exposure=None):
    """chi2 of the records ``P`` in one engine call: ``chi2_series`` for points alone, ``chi2`` with bands, and
    ``chi2(extinction=(ext_kernel, A_V))`` with a per-walker A_V.  With ``exposure`` = (expo_time, num_points), one
    single-set ``chi2_multi_bands(exposures=...)``.  The stored arrays are passed as they are."""
    if exposure is not None:
        ext = None if A_V is None else ([ext_kernel], A_V)
        return engine.chi2_multi_bands(P, [points], [bands], np.zeros(P.size, dtype=np.int32), extinction=ext,
                                       exposures=[exposure])
    if A_V is not None:
        return engine.chi2(P, points, bands, extinction=(ext_kernel, A_V))
    if not bands:
        return engine.chi2_series(P, *points)
    return engine.chi2(P, points, bands)


def _ensemble_chi2(engine, P, points, bands, ext_kernel=None, A_V=None, window=None, exposure=None):
    """chi2 of every record of ``P``; +inf for a record the model constructor rejects (the reference maps that exception
    to logL = -inf, samplers.py:63-70).  ``A_V`` (per walker) shifts the point data and is dropped without points.
    ``window``: None evaluates every walker here; else the ensemble is split over the ranks by the cost proxy over the
    span of these times.  The validity mask is computed from the parameters alone, identically on every rank, BEFORE the
    split, and every rank joins the gather even with an empty share: a rejected walker can never desynchronise it."""
    from .engine import Engine

    ok = Engine.valid_mask(P)
    per_walker = (A_V,) if A_V is not None and points is not None else ()

    def evaluate(Q, *av):
        return _chi2_batch(engine, Q, points, bands, ext_kernel, av[0] if av else None, exposure)

    if window is not None:
        from . import parallel

        return parallel.partitioned_chi2(engine, P, window, None, None, None, None, evaluate=evaluate, valid=ok,
                                         per_walker=per_walker)
    out = np.full(P.size, np.inf)
    if ok.any():
        out[ok] = evaluate(P[ok], *(a[ok] for a in per_walker))
    return out


class BatchedLikelihood:
    """``log_prob_batch(samples[n, ndim]) -> logp[n]`` on the GPU.

    names / log_scale describe the sampler-space columns (log10 parameters are exponentiated like
    ``_build_transformer``, fitting/utils.py:110-135); ``template`` is a 1-record ``vag_params``
    array carrying every fixed setting (jet/medium type, distance, redshift, switches).

    A name ``"A_V"`` fits host-galaxy extinction: ``ext_kernel`` (per point, in the caller's order) is the
    extinction law at each point, and a sample's point data are compared as ln F_obs + A_V * ext_kernel
    (``Engine.chi2(extinction=...)``).  Band data are not shifted.

    ``expo_time`` (per point, in the caller's order, each >= 0) compares each point with an exposure with the model
    averaged over ``expo_points`` samples of its exposure, the rule of ``Model.flux_density_exposures``; a point with 0
    is compared with the model at its time (``Engine.chi2_multi_bands(exposures=...)``).  Band data have no exposures.
    """

    def __init__(self, engine, template, names: Sequence[str], log_scale: Sequence[bool], t, nu, flux, err,
                 weights=None, lower=None, upper=None, log_prior: Optional[Callable] = None,
                 log_likelihood_fn: Callable = lambda chi2: -0.5 * chi2, distributed: bool = False, bands=(),
                 ext_kernel=None, expo_time=None, expo_points=10):
        self.engine = engine
        self.template = np.ascontiguousarray(template, dtype=abi.PARAMS_DTYPE).reshape(-1)[:1].copy()
        self.names = list(names)
        self.log_scale = np.asarray(log_scale, dtype=bool)
        for n in self.names:
            if n not in _FIELDS and n != "A_V":
                raise ValueError(f"unknown parameter '{n}' (supported: {sorted(_FIELDS)} and A_V)")
        if "A_V" in self.names and ext_kernel is None:
            raise ValueError("fitting A_V needs ext_kernel, the extinction law at each point")
        if len(np.atleast_1d(t)):
            self.t, self.nu, self.lnF, self.sig, self.w = consolidate_data(t, nu, flux, err, weights)
        else:
            self.t = self.nu = self.lnF = self.sig = self.w = np.zeros(0)
        self.ext_kernel = None
        if ext_kernel is not None:
            ext = np.asarray(ext_kernel, dtype=np.float64).reshape(-1)
            if ext.size != self.t.size:
                raise ValueError(f"ext_kernel has {ext.size} values for {self.t.size} points")
            self.ext_kernel = ext[time_order(t)]
        self.expo_time, self.expo_points = None, int(expo_points)
        if expo_time is not None:
            e = np.asarray(expo_time, dtype=np.float64).reshape(-1)
            if e.size != self.t.size or not self.t.size:
                raise ValueError(f"expo_time has {e.size} values for {self.t.size} points")
            if not np.all(np.isfinite(e) & (e >= 0)):
                raise ValueError("expo_time must be finite and >= 0")
            if np.any(e > 0) and self.expo_points < 2:
                raise ValueError("expo_points must be at least 2 to sample within each exposure time")
            self.expo_time = e[time_order(t)]
        # band-integrated data sets (Fitter.add_flux -> BandObs; fitter.py:525-531 evaluates Model.flux on each)
        self.bands = [band_obs(**b) for b in bands]
        if not self.t.size and not self.bands:
            raise ValueError("no data")
        # the times of the distributed split's cost proxy: the points', or every band's without points
        self._cost_times = self.t if self.t.size else np.concatenate([b["t"] for b in self.bands])
        if self.expo_time is not None:  # and the last sample of each exposure (vag_exposure.cuh)
            k = max(self.expo_points - 1, 1)
            self._cost_times = np.concatenate([self.t, self.t + k * (self.expo_time / k)])
        self.lower = None if lower is None else np.asarray(lower, dtype=np.float64)
        self.upper = None if upper is None else np.asarray(upper, dtype=np.float64)
        self.log_prior = log_prior
        self.log_likelihood_fn = log_likelihood_fn
        self.distributed = distributed

    def to_params(self, samples: np.ndarray) -> np.ndarray:
        samples = np.atleast_2d(np.asarray(samples, dtype=np.float64))
        P = np.repeat(self.template, samples.shape[0])
        for i, name in enumerate(self.names):
            if name == "A_V":  # not a model parameter: it shifts the observed point data (_chi2_batch)
                continue
            col = self._column(samples, i)
            path = _FIELDS[name]
            if len(path) == 1:
                P[path[0]] = col
            else:
                P[path[0]][path[1]] = col
        return P

    def _column(self, samples, i):
        return 10.0 ** samples[:, i] if self.log_scale[i] else samples[:, i]

    def chi2(self, samples: np.ndarray) -> np.ndarray:
        """chi2 of every sample; +inf for a sample the model constructor rejects (``_ensemble_chi2``)."""
        samples = np.atleast_2d(np.asarray(samples, dtype=np.float64))
        pts = (self.t, self.nu, self.lnF, self.sig, self.w) if self.t.size else None
        A_V = self._column(samples, self.names.index("A_V")) if "A_V" in self.names else None
        return _ensemble_chi2(self.engine, self.to_params(samples), pts, self.bands, self.ext_kernel, A_V,
                              self._cost_times if self.distributed else None, self._exposure())

    def _exposure(self):
        """(expo_time, expo_points) in time order, or None"""
        return None if self.expo_time is None else (self.expo_time, self.expo_points)

    def _in_bounds(self, samples: np.ndarray) -> np.ndarray:
        """Indices of the samples inside [lower, upper]."""
        in_bounds = np.ones(samples.shape[0], dtype=bool)
        if self.lower is not None:
            in_bounds &= np.all(samples >= self.lower, axis=1)
        if self.upper is not None:
            in_bounds &= np.all(samples <= self.upper, axis=1)
        return np.nonzero(in_bounds)[0]

    def _log_prob(self, samples: np.ndarray, idx: np.ndarray, chi2: np.ndarray) -> np.ndarray:
        """logp of every sample from the chi2 of the in-bounds ones (``idx``); -inf elsewhere and where not finite."""
        logp = np.full(samples.shape[0], -np.inf)
        if idx.size:
            ll = np.where(np.isfinite(chi2), self.log_likelihood_fn(chi2), -np.inf)
            ll[~np.isfinite(ll)] = -np.inf
            if self.log_prior is not None:
                ll = ll + self.log_prior(samples[idx])
            logp[idx] = ll
        return logp

    def __call__(self, samples: np.ndarray) -> np.ndarray:
        samples = np.atleast_2d(np.asarray(samples, dtype=np.float64))
        idx = self._in_bounds(samples)
        return self._log_prob(samples, idx, self.chi2(samples[idx]) if idx.size else np.zeros(0))

    def flux_quantiles(self, samples: np.ndarray, t, nu, q=(0.16, 0.5, 0.84)):
        """Posterior-predictive band of this fit: ``numpy.quantile`` over the posterior draws ``samples[n, ndim]`` of the
        model's total flux density on the grid (t ascending, nu) at every ``q`` -> (float64[n_q, n_nu, n_t], the number of
        draws used).  Draws the constructors reject are dropped, and so are draws whose ODE failed; bounds are not
        applied (these are posterior draws), and ``A_V`` plays no part (it shifts the data, not the model).  One
        ``Engine.flux_quantiles_multi`` call with one grid."""
        from .engine import Engine

        P = self.to_params(samples)
        P = P[Engine.valid_mask(P)]
        bands, n_used = self.engine.flux_quantiles_multi(P, [(t, nu)], np.zeros(P.size, dtype=np.int32), q)
        return bands[0], int(n_used[0])


_CUDA_STREAM_LEGACY = 0x1  # cudaStreamLegacy (driver_types.h)


def _stream(device):
    """The stream handle of a ``_dev`` call on ``device``: torch's current stream on a GPU, 0 on the CPU.  A NULL stream
    would be the engine's own, unordered with the record assembly before the call.  torch's default stream has the
    handle 0 and is CUDA's legacy default stream, which the C ABI takes as cudaStreamLegacy."""
    import torch

    if device.type != "cuda":
        return 0
    return torch.cuda.current_stream(device).cuda_stream or _CUDA_STREAM_LEGACY


def _rank_share(cost, evaluate, device):
    """Every walker's chi2 (a float64 tensor on ``device``) on every rank: the walkers are split by
    ``parallel.balanced_assignment`` of ``cost``, ``evaluate(mine, idx)`` gives this rank's share (its walkers as a numpy
    array and as a tensor on ``device``), and one ``parallel.gather_indexed_tensor`` collects them, joined even with an
    empty share."""
    import torch

    from . import parallel

    world, rank = parallel.world_rank()
    sets = parallel.balanced_assignment(cost, world)
    mine = sets[rank]
    local = evaluate(mine, torch.as_tensor(mine, dtype=torch.long, device=device))
    return parallel.gather_indexed_tensor(local, sets, len(cost))


def _field_offset(path):
    """Byte offset of a float64 field of ``abi.PARAMS_DTYPE`` (``("fwd", "eps_e")`` for a nested one)."""
    dt, off = abi.PARAMS_DTYPE, 0
    for name in path:
        dt, o = dt.fields[name][:2]
        off += o
    assert dt == np.float64 and off % 8 == 0
    return off


class DeviceLikelihood(BatchedLikelihood):
    """``BatchedLikelihood`` with the data, the walkers and the result in HBM: the same constructor (``device``: where the
    data live, default the engine's GPU) and the same ``__call__(samples[n, ndim]) -> logp[n]``.

    The point data, ``ext_kernel`` and band arrays go to the device once, here.  Per call only the ``n x ndim`` sampler
    columns are uploaded -- exponentiated on the host with ``BatchedLikelihood._column``'s numpy expression (a device
    ``pow`` would not give the same bits, and the theta grid amplifies a last-bit difference).  The records are assembled
    on the device from the template, and ONE ``vag_chi2_dev`` call on the current torch stream validates them (rejected
    walkers: chi2 = +inf), sizes their grids and evaluates every term.  Distributed, each rank evaluates its share of the
    host-side cost-balanced assignment and the chi2 tensors are gathered on the device."""

    def __init__(self, engine, *args, device=None, **kwargs):
        import torch

        super().__init__(engine, *args, **kwargs)
        if self.expo_time is not None:
            raise NotImplementedError("DeviceLikelihood: expo_time is not supported (use BatchedLikelihood)")
        self.device = torch.device("cuda", engine.device) if device is None else torch.device(device)

        def dev(a):
            return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=self.device)

        self._pts = tuple(dev(a) for a in (self.t, self.nu, self.lnF, self.sig, self.w)) if self.t.size else None
        self._ext = dev(self.ext_kernel) if self.ext_kernel is not None else None
        self._bands = [dict(b, **{k: dev(b[k]) for k in ("t", "lnF_obs", "sigma_ln", "w")}) for b in self.bands]
        self._template = torch.as_tensor(self.template.view(np.uint8), device=self.device)
        model = [i for i, n in enumerate(self.names) if n != "A_V"]
        self._cols = torch.as_tensor(model, dtype=torch.long, device=self.device)
        self._slots = torch.as_tensor([_field_offset(_FIELDS[self.names[i]]) // 8 for i in model], dtype=torch.long,
                                      device=self.device)
        self._av = self.names.index("A_V") if "A_V" in self.names and self.t.size else None

    def columns(self, samples: np.ndarray) -> np.ndarray:
        """float64[n, ndim]: the sampler columns as the model sees them (log10 columns exponentiated)."""
        samples = np.atleast_2d(np.asarray(samples, dtype=np.float64))
        out = np.empty_like(samples)
        for i in range(len(self.names)):
            out[:, i] = self._column(samples, i)
        return out

    def records(self, cols):
        """uint8[n * sizeof(vag_params)] on the device: the template repeated, the model columns of ``cols`` (float64
        tensor [n, ndim] from ``columns``) scattered into a float64 view at their fields' offsets."""
        import torch

        n = cols.shape[0]
        rec = self._template.repeat(n)
        view = rec.view(torch.float64).view(n, abi.PARAMS_DTYPE.itemsize // 8)
        view[:, self._slots] = cols[:, self._cols]
        return rec

    def _chi2_dev(self, cols):
        import torch

        n = cols.shape[0]
        chi2 = torch.empty(n, dtype=torch.float64, device=self.device)
        if n == 0:
            return chi2
        rec = self.records(cols)
        points = None if self._pts is None else (*(a.data_ptr() for a in self._pts), self.t.size)
        av = None if self._av is None else cols[:, self._av].contiguous()
        extinction = None if av is None else (self._ext.data_ptr(), av.data_ptr())
        bands = [dict(b, n=b["t"].numel(), **{k: b[k].data_ptr() for k in ("t", "lnF_obs", "sigma_ln", "w")})
                 for b in self._bands]
        self.engine.chi2_dev(rec.data_ptr(), n, points, bands, chi2.data_ptr(), extinction=extinction,
                             stream=_stream(self.device))
        return chi2

    def chi2(self, samples: np.ndarray) -> np.ndarray:
        """chi2 of every sample; +inf for a sample the model constructor rejects (checked on the device)."""
        import torch

        cols = torch.as_tensor(self.columns(samples), device=self.device)
        if not self.distributed:
            return self._chi2_dev(cols).cpu().numpy()
        from . import parallel

        tt = self._cost_times
        cost = parallel.cost_proxy(self.to_params(samples), float(np.min(tt)), float(np.max(tt)))
        return _rank_share(cost, lambda _, idx: self._chi2_dev(cols[idx]), self.device).cpu().numpy()


class LikelihoodStack:
    """K independent fits evaluated together: ``__call__([samples_1, ..., samples_K]) -> [logp_1, ..., logp_K]`` with ONE
    ``Engine.chi2_multi`` call, where each ``BatchedLikelihood`` called alone would make K calls.  Meant for many small
    ensembles -- K emcee samplers stepped in lockstep, a catalogue of light curves, injection-recovery runs -- which
    fill the GPU together where one alone would not.

    Each likelihood keeps its own template, names, point data, bounds, prior, ``log_likelihood_fn`` and optional fitted
    ``A_V``; fit k's walkers are evaluated on fit k's data set.  Bounds, rejected parameter sets and non-finite chi2 give
    -inf as in ``BatchedLikelihood.__call__``.  When only some fits sample ``A_V``, the others run with ext_k = 0 and
    A_V = 0, and lnF_obs + 0 * 0 is lnF_obs exactly.  Fits with ``expo_time`` keep their own exposures and
    ``expo_points``, and the others get zero exposures: the stack then makes one ``chi2_multi_bands(exposures=...)`` call
    instead.  The engine is the first likelihood's.
    Not supported (``NotImplementedError``): band-integrated data (stack such fits with ``BandLikelihoodStack``),
    ``distributed=True`` and ``DeviceLikelihood``."""

    _band_data = False  # whether fits with band-integrated data (or without points) are accepted

    def __init__(self, likelihoods: Sequence[BatchedLikelihood]):
        self.likelihoods = list(likelihoods)
        if not self.likelihoods:
            raise ValueError(f"{type(self).__name__} needs at least one likelihood")
        for k, lk in enumerate(self.likelihoods):
            if isinstance(lk, DeviceLikelihood):
                raise NotImplementedError(f"likelihood {k}: a DeviceLikelihood cannot be stacked (its data live in HBM)")
            if not self._band_data and (lk.bands or not lk.t.size):
                raise NotImplementedError(f"likelihood {k}: band-integrated data cannot be stacked (point data only)")
            if lk.distributed:
                raise NotImplementedError(f"likelihood {k}: distributed=True cannot be stacked")
        self.engine = self.likelihoods[0].engine
        self.datasets = [(lk.t, lk.nu, lk.lnF, lk.sig, lk.w) if lk.t.size else None for lk in self.likelihoods]
        self.fits_av = ["A_V" in lk.names and lk.t.size > 0 for lk in self.likelihoods]
        self.exposures = [lk._exposure() for lk in self.likelihoods]
        if all(e is None for e in self.exposures):
            self.exposures = None

    def _walkers(self, samples):
        """The valid walkers of every fit as one batch: (records, fit of each, A_V of each (0 where the fit has none),
        the validity mask of every fit)."""
        from .engine import Engine

        P, ds, av, ok = [], [], [], []
        for k, (lk, s) in enumerate(zip(self.likelihoods, samples)):
            s = np.atleast_2d(np.asarray(s, dtype=np.float64))
            p = lk.to_params(s)
            good = Engine.valid_mask(p)
            ok.append(good)
            P.append(p[good])
            ds.append(np.full(int(good.sum()), k, dtype=np.int32))
            av.append(lk._column(s, lk.names.index("A_V"))[good] if self.fits_av[k] else np.zeros(int(good.sum())))
        return np.concatenate(P), np.concatenate(ds), np.concatenate(av), ok

    @staticmethod
    def _split(flat, ok):
        """chi2 of the valid walkers back per fit, +inf for the rejected ones."""
        out, lo = [], 0
        for good in ok:
            c = np.full(good.size, np.inf)
            c[good] = flat[lo:lo + int(good.sum())]
            lo += int(good.sum())
            out.append(c)
        return out

    def chi2(self, samples):
        """chi2 of every sample of every fit (a list of K arrays); +inf for parameter sets the constructors reject."""
        P, ds, av, ok = self._walkers(samples)
        extinction = None
        if any(self.fits_av):
            ext = [None if not lk.t.size else lk.ext_kernel if fit else np.zeros(lk.t.size)
                   for lk, fit in zip(self.likelihoods, self.fits_av)]
            extinction = (ext, av)
        return self._split(self._engine_chi2(P, ds, extinction) if P.size else np.zeros(0), ok)

    def _engine_chi2(self, P, dataset_of, extinction):
        """chi2 of the stacked walkers in one engine call: ``chi2_multi`` here, ``chi2_multi_bands`` with bands or
        exposures."""
        if self.exposures is None:
            return self.engine.chi2_multi(P, self.datasets, dataset_of, extinction=extinction)
        return self.engine.chi2_multi_bands(P, self.datasets, [[] for _ in self.datasets], dataset_of, extinction=extinction,
                                            exposures=self.exposures)

    def flux_quantiles(self, samples, grids, q=(0.16, 0.5, 0.84)):
        """Posterior-predictive bands of the K fits in ONE ``Engine.flux_quantiles_multi`` call: fit k's draws
        ``samples[k]`` (through its own ``to_params``) on its own grid ``grids[k]`` = (t ascending, nu).  Returns (a list
        of K float64[n_q, n_nu, n_t] arrays, ``numpy.quantile`` of the total flux over the fit's draws at every ``q``;
        int64[K] draws used per fit).  Draws the constructors reject (``Engine.valid_mask``) are dropped, and so are
        draws whose ODE failed; bounds are not applied (these are posterior draws), and ``A_V`` plays no part (it shifts
        the data, not the model).  Nothing is distributed: quantiles do not decompose over ranks."""
        if len(samples) != len(self.likelihoods) or len(grids) != len(self.likelihoods):
            raise ValueError(f"{len(samples)} sample arrays and {len(grids)} grids for {len(self.likelihoods)} likelihoods")
        P, ds, _, _ = self._walkers(samples)
        return self.engine.flux_quantiles_multi(P, grids, ds, q)

    def __call__(self, samples):
        if len(samples) != len(self.likelihoods):
            raise ValueError(f"{len(samples)} sample arrays for {len(self.likelihoods)} likelihoods")
        samples = [np.atleast_2d(np.asarray(s, dtype=np.float64)) for s in samples]
        idx = [lk._in_bounds(s) for lk, s in zip(self.likelihoods, samples)]
        chi2 = self.chi2([s[i] for s, i in zip(samples, idx)])
        return [lk._log_prob(s, i, c) for lk, s, i, c in zip(self.likelihoods, samples, idx, chi2)]


class BandLikelihoodStack(LikelihoodStack):
    """``LikelihoodStack`` for fits with band-integrated data: fits with points and bands, bands only, or points only, all
    evaluated with ONE ``Engine.chi2_multi_bands`` call -- the points of every fit in one ragged pass and every band of
    every fit in one more, where each ``BatchedLikelihood`` alone makes 1 + (its bands) pipeline runs.  Fit k's walkers
    get fit k's point term and then its band terms in its own order; ``__call__``, the bounds and the -inf rules are
    ``LikelihoodStack``'s.  A bands-only fit that names ``A_V`` ignores it, as ``BatchedLikelihood`` does without points.
    Not supported (``NotImplementedError``): ``distributed=True`` and ``DeviceLikelihood``."""

    _band_data = True

    def __init__(self, likelihoods: Sequence[BatchedLikelihood]):
        super().__init__(likelihoods)
        self.bands = [lk.bands for lk in self.likelihoods]

    def _engine_chi2(self, P, dataset_of, extinction):
        expo = {} if self.exposures is None else {"exposures": self.exposures}
        return self.engine.chi2_multi_bands(P, self.datasets, self.bands, dataset_of, extinction=extinction, **expo)


class DeviceLikelihoodStack(LikelihoodStack):
    """K ``DeviceLikelihood`` fits evaluated together with ONE ``Engine.chi2_multi_bands_dev`` call: the stack of
    ``BandLikelihoodStack`` with the data, the walkers and the result in HBM, and -- with ``distributed=True`` -- spread
    over the GPUs of a box.  Fits may have points, bands or both, with or without a fitted ``A_V``; ``__call__``, ``chi2``,
    the bounds, the per-fit prior and ``log_likelihood_fn`` and the -inf rules are ``LikelihoodStack``'s.

    The members' device point arrays are concatenated once, in fit order (ext_k = 0 for a fit with points and no ``A_V``,
    and lnF_obs + 0 * 0 is lnF_obs exactly), their band arrays stay where they are, and the records' template of every fit
    is a row of one [K, sizeof(vag_params) / 8] float64 table on the device.  Per call the host exponentiates the columns
    (``DeviceLikelihood.columns``) and packs every in-bounds walker into one [n, max_ndim + 1] float64 matrix -- the last
    column is ``A_V``, 0 where a fit has none -- uploaded with the walkers' fits in one copy.  The records are assembled on
    the device by a few launches whatever K: the template rows gathered by fit, then one scatter through a per-fit slot
    table whose padding points at a scratch column.  The call validates the records on the device (rejected: chi2 = +inf).

    ``distributed=True``: every rank gets the same samples, splits all fits' in-bounds walkers with
    ``parallel.balanced_assignment`` of ``parallel.cost_proxy`` (each fit over its own points' and bands' time window),
    evaluates its share with one call and takes part in one ``parallel.gather_indexed_tensor``, even with an empty share.
    The members must share one engine and one device and be built with ``distributed=False``: the stack's flag decides."""

    def __init__(self, likelihoods: Sequence["DeviceLikelihood"], distributed: bool = False):
        import torch

        self.likelihoods = list(likelihoods)
        if not self.likelihoods:
            raise ValueError("DeviceLikelihoodStack needs at least one likelihood")
        first = self.likelihoods[0]
        for k, lk in enumerate(self.likelihoods):
            if not isinstance(lk, DeviceLikelihood):
                raise ValueError(f"likelihood {k}: DeviceLikelihoodStack stacks DeviceLikelihood fits only")
            if lk.engine is not first.engine or lk.device != first.device:
                raise ValueError(f"likelihood {k}: every fit of the stack must use the first fit's engine and device")
            if lk.distributed:
                raise ValueError(f"likelihood {k}: built with distributed=True; the stack's own flag decides")
        self.engine, self.device, self.distributed = first.engine, first.device, distributed
        lks = self.likelihoods
        self.fits_av = [lk._av is not None for lk in lks]
        with_pts = [lk for lk in lks if lk._pts is not None]
        self.n_points = sum(lk.t.size for lk in with_pts)
        self._pts = tuple(torch.cat([lk._pts[i] for lk in with_pts]) for i in range(5)) if with_pts else None
        self._ext = None
        if any(self.fits_av):
            self._ext = torch.cat([lk._ext if fit else torch.zeros(lk.t.size, dtype=torch.float64, device=self.device)
                                   for lk, fit in zip(lks, self.fits_av) if lk._pts is not None])
        self._bands = [dict(b, n=b["t"].numel(), **{k: b[k].data_ptr() for k in ("t", "lnF_obs", "sigma_ln", "w")})
                       for lk in lks for b in lk._bands]
        self.sets = (abi.MultiSet * len(lks))()
        off = b0 = 0
        for k, lk in enumerate(lks):
            self.sets[k] = abi.MultiSet(off, lk.t.size, b0, len(lk._bands))
            off, b0 = off + lk.t.size, b0 + len(lk._bands)
        # each fit's time window (points and bands), for the cost proxy of the distributed split
        self._window = []
        for lk in lks:
            tt = np.concatenate([lk.t] + [b["t"] for b in lk.bands])
            self._window.append((float(np.min(tt)), float(np.max(tt))))
        # records: template table [K, W], per-fit slot table [K, max_ndim + 1] into a row of W + 1 (W: the scratch column)
        self._width = abi.PARAMS_DTYPE.itemsize // 8
        self._ncol = max(len(lk.names) for lk in lks) + 1
        self._templates = torch.as_tensor(np.stack([lk.template.view(np.float64) for lk in lks]), device=self.device)
        slots = np.full((len(lks), self._ncol), self._width, dtype=np.int64)
        for k, lk in enumerate(lks):
            for i, name in enumerate(lk.names):
                if name != "A_V":
                    slots[k, i] = _field_offset(_FIELDS[name]) // 8
        self._slots = torch.as_tensor(slots, device=self.device)

    def records(self, X, fit_of):
        """uint8[n * sizeof(vag_params)] on the device from the packed columns ``X`` ([n, max_ndim + 1] float64) and the
        fit of every walker (int64 [n]): each fit's template with its model columns at their fields' offsets."""
        import torch

        n = X.shape[0]
        rec = torch.empty((n, self._width + 1), dtype=torch.float64, device=self.device)
        rec[:, :self._width] = self._templates[fit_of]
        rec.scatter_(1, self._slots[fit_of], X)
        return rec[:, :self._width].contiguous().view(torch.uint8).view(-1)

    def _pack(self, samples):
        """(the packed columns and the walkers' fits in one float64 host buffer, their number, the fits as int32)"""
        n_k = [s.shape[0] for s in samples]
        n = sum(n_k)
        buf = np.zeros(n * self._ncol + n)
        X = buf[:n * self._ncol].reshape(n, self._ncol)
        fit_of = np.repeat(np.arange(len(n_k), dtype=np.int64), n_k)
        buf[n * self._ncol:] = fit_of.view(np.float64)
        lo = 0
        for k, (lk, s) in enumerate(zip(self.likelihoods, samples)):
            if s.shape[0]:
                X[lo:lo + s.shape[0], :len(lk.names)] = lk.columns(s)  # an A_V column's slot is the scratch column
                if self.fits_av[k]:
                    X[lo:lo + s.shape[0], -1] = lk._column(s, lk._av)
            lo += s.shape[0]
        return buf, n, fit_of.astype(np.int32)

    def _chi2_dev(self, X, fit_of, dataset_of):
        import torch

        n = X.shape[0]
        chi2 = torch.empty(n, dtype=torch.float64, device=self.device)
        if n == 0:
            return chi2
        rec = self.records(X, fit_of)
        points = None if self._pts is None else (*(a.data_ptr() for a in self._pts), self.n_points)
        av = X[:, -1].contiguous() if self._ext is not None else None
        extinction = None if av is None else (self._ext.data_ptr(), av.data_ptr())
        self.engine.chi2_multi_bands_dev(rec.data_ptr(), n, dataset_of, self.sets, points, self._bands, chi2.data_ptr(),
                                         extinction=extinction, stream=_stream(self.device))
        return chi2

    def chi2(self, samples):
        """chi2 of every sample of every fit (a list of K arrays); +inf for parameter sets the constructors reject (checked
        on the device)."""
        import torch

        samples = [np.atleast_2d(np.asarray(s, dtype=np.float64)) for s in samples]
        buf, n, ds = self._pack(samples)
        up = torch.as_tensor(buf, device=self.device)  # the one H2D copy of the call
        X, fit_of = up[:n * self._ncol].view(n, self._ncol), up[n * self._ncol:].view(torch.int64)
        if not self.distributed:
            flat = self._chi2_dev(X, fit_of, ds).cpu().numpy()
        else:
            from . import parallel

            cost = np.concatenate([parallel.cost_proxy(lk.to_params(s), *win) if s.shape[0] else np.zeros(0)
                                   for lk, s, win in zip(self.likelihoods, samples, self._window)])
            evaluate = lambda mine, idx: self._chi2_dev(X[idx], fit_of[idx], ds[mine])  # noqa: E731
            flat = _rank_share(cost, evaluate, self.device).cpu().numpy()
        out, lo = [], 0
        for s in samples:
            out.append(flat[lo:lo + s.shape[0]])
            lo += s.shape[0]
        return out
