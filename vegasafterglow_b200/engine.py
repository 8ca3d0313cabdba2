"""Batched model evaluation on one GPU through the C ABI (include/vag.h).

``Engine`` owns one ``vag_context`` (a CUDA stream + growable HBM workspaces).  Host-array
methods copy inputs/outputs inside the call; ``*_dev`` methods take raw device pointers (e.g.
``torch.Tensor.data_ptr()``) and only enqueue work.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib, abi


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Engine:
    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self._lib.vag_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.vag_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- host buffers -------------------------------------------------------------------------
    @staticmethod
    def _params(params):
        p = np.ascontiguousarray(params, dtype=abi.PARAMS_DTYPE).reshape(-1)
        return p

    def flux_density_grid(self, params, t, nu, return_status=False):
        """Batched ``Model.flux_density_grid`` -> float64[n_models, 5, n_nu, n_t]
        (component order ``abi.COMPONENTS``)."""
        p, t, nu = self._params(params), _f64(t).reshape(-1), _f64(nu).reshape(-1)
        out = (np.zeros if getattr(self, "_present_only", False) else np.empty)((p.size, abi.NCOMP, nu.size, t.size))
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_flux_density_grid(self._h, p.ctypes.data, p.size, t.ctypes.data, t.size,
                                                   nu.ctypes.data, nu.size, out.ctypes.data, st.ctypes.data))
        return (out, st) if return_status else out

    def flux_density_series(self, params, t, nu, return_status=False):
        """Batched ``Model.flux_density`` -> float64[n_models, 5, n]."""
        p, t, nu = self._params(params), _f64(t).reshape(-1), _f64(nu).reshape(-1)
        if t.size != nu.size:  # pybind/pymodel.cpp:376-379
            raise ValueError("time and frequency arrays must have the same size\nIf you intend to get grid-like "
                             "output, use the generic `flux_density_grid` instead")
        out = (np.zeros if getattr(self, "_present_only", False) else np.empty)((p.size, abi.NCOMP, t.size))
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_flux_density_series(self._h, p.ctypes.data, p.size, t.ctypes.data, nu.ctypes.data,
                                                     t.size, out.ctypes.data, st.ctypes.data))
        return (out, st) if return_status else out

    def flux_band(self, params, t, nu_min, nu_max, num_nu, return_status=False):
        """Batched ``Model.flux`` (band-integrated, Boole rule) -> float64[n_models, 5, n_t] [erg cm^-2 s^-1]."""
        p, t = self._params(params), _f64(t).reshape(-1)
        out = np.empty((p.size, abi.NCOMP, t.size))
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_flux_band(self._h, p.ctypes.data, p.size, t.ctypes.data, t.size, float(nu_min),
                                           float(nu_max), int(num_nu), out.ctypes.data, st.ctypes.data))
        return (out, st) if return_status else out

    def flux_density_exposures(self, params, t, nu, expo_time, num_points=10, return_status=False):
        """Batched ``Model.flux_density_exposures`` (pybind/pymodel.cpp:412-496) -> float64[n_models, 5, n]: each point
        is the average of ``num_points`` samples spread over its exposure window, sampled, evaluated and averaged on the
        GPU (``vag_flux_density_exposures``); t need not be sorted."""
        p = self._params(params)
        t, nu, expo_time = (_f64(a).reshape(-1) for a in (t, nu, expo_time))
        if not (t.size == nu.size == expo_time.size):
            raise ValueError("time, frequency, and exposure time arrays must have the same size")
        out = (np.zeros if getattr(self, "_present_only", False) else np.empty)((p.size, abi.NCOMP, t.size))
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_flux_density_exposures(self._h, p.ctypes.data, p.size, t.ctypes.data, nu.ctypes.data,
                                                        expo_time.ctypes.data, t.size, max(int(num_points), 0),
                                                        out.ctypes.data, st.ctypes.data))
        return (out, st) if return_status else out

    def chi2_series(self, params, t, nu, lnF_obs, sigma_ln, w, return_status=False):
        """Batched ``Fitter._evaluate`` for point data -> chi2[n_models] (+inf where non-finite)."""
        p = self._params(params)
        t, nu, lnF_obs, sigma_ln, w = (_f64(a).reshape(-1) for a in (t, nu, lnF_obs, sigma_ln, w))
        if not (t.size == nu.size == lnF_obs.size == sigma_ln.size == w.size):
            raise ValueError("t, nu, lnF_obs, sigma_ln and w must have the same size")
        chi2 = np.empty(p.size)
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_chi2_series(self._h, p.ctypes.data, p.size, t.ctypes.data, nu.ctypes.data,
                                             lnF_obs.ctypes.data, sigma_ln.ctypes.data, w.ctypes.data, t.size,
                                             chi2.ctypes.data, st.ctypes.data))
        return (chi2, st) if return_status else chi2

    def chi2(self, params, points=None, bands=(), return_status=False, extinction=None):
        """Batched ``Fitter._evaluate`` (fitter.py:503-533) -> chi2[n_models]: the point-data term (``points`` =
        (t, nu, lnF_obs, sigma_ln, w), times ascending, or None) plus one term per band-integrated data set
        (``bands``: dicts with t, lnF_obs, sigma_ln, w, nu_min, nu_max, num_nu -- ``Model.flux`` on each).
        ``extinction`` = (ext_k[n_points], A_V[n_models]): a fitted host extinction, which compares model m's point
        fluxes with lnF_obs + A_V[m] * ext_k (band terms unchanged).
        +inf where the sum is not finite or the model's ODE failed (include/vag.h vag_chi2, vag_chi2_ext)."""
        p = self._params(params)
        if points is not None:
            pt = [_f64(a).reshape(-1) for a in points]
            if len(pt) != 5 or len({a.size for a in pt}) != 1:
                raise ValueError("points must be (t, nu, lnF_obs, sigma_ln, w) of one size")
            n_pt = pt[0].size
        else:
            pt, n_pt = [np.zeros(0)] * 5, 0
        ext = av = None
        if extinction is not None:
            if points is None:
                raise ValueError("extinction shifts the point data: it needs points")
            ext, av = (_f64(a).reshape(-1) for a in extinction)
            if ext.size != n_pt:
                raise ValueError(f"ext_k has {ext.size} values for {n_pt} points")
            if av.size != p.size:
                raise ValueError(f"A_V has {av.size} values for {p.size} models")
        arr, _keep = self._band_array(bands, data=True)
        out = np.empty(p.size)
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_chi2_ext(self._h, p.ctypes.data, p.size, *[a.ctypes.data if n_pt else None for a in pt],
                                          None if ext is None else ext.ctypes.data, n_pt,
                                          None if av is None else av.ctypes.data,
                                          C.cast(arr, C.c_void_p) if len(bands) else None, len(bands), out.ctypes.data,
                                          st.ctypes.data))
        return (out, st) if return_status else out

    # ---- several data sets in one batch (include/vag.h vag_flux_density_series_multi, vag_chi2_multi) -------------------
    @staticmethod
    def _concat_sets(datasets, names):
        """Per-data-set column tuples -> (the columns concatenated over the sets, ``abi.SeriesSet`` array, their number)."""
        cols, sizes = [[] for _ in names], []
        for d, ds in enumerate(datasets):
            arrs = [_f64(a).reshape(-1) for a in ds]
            if len(arrs) != len(names) or len({a.size for a in arrs}) != 1:
                raise ValueError(f"data set {d} must be ({', '.join(names)}) of one size")
            for c, a in zip(cols, arrs):
                c.append(a)
            sizes.append(arrs[0].size)
        if not sizes:
            raise ValueError("no data sets")
        sets = (abi.SeriesSet * len(sizes))()
        offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
        for d, (o, n) in enumerate(zip(offsets, sizes)):
            sets[d] = abi.SeriesSet(int(o), int(n))
        return [np.concatenate(c) for c in cols], sets, np.asarray(sizes, dtype=np.int64)

    @staticmethod
    def _dataset_of(dataset_of, n_models):
        ds = np.asarray(dataset_of).reshape(-1)
        if ds.size != n_models:
            raise ValueError(f"dataset_of has {ds.size} entries for {n_models} models")
        if ds.size and not (np.issubdtype(ds.dtype, np.integer) and ds.min() >= -2**31 and ds.max() < 2**31):
            raise ValueError("dataset_of must hold int32 data-set indices")
        return np.ascontiguousarray(ds, dtype=np.int32)

    @staticmethod
    def _extinction(extinction, sizes, n_models):
        """``extinction`` = (ext_k, A_V) of a batch of several data sets -> (ext_k concatenated over the sets, A_V) as float64
        arrays, or (None, None).  ext_k holds one array per data set, None for a set without points; A_V[n_models]."""
        if extinction is None:
            return None, None
        ext_sets, av = extinction
        if len(ext_sets) != len(sizes):
            raise ValueError(f"extinction has {len(ext_sets)} ext_k entries for {len(sizes)} data sets")
        ext = [np.zeros(0) if e is None else _f64(e).reshape(-1) for e in ext_sets]
        for d, (e, n) in enumerate(zip(ext, sizes)):
            if e.size != n:
                raise ValueError(f"data set {d}: ext_k has {e.size} values for {n} points")
        av = _f64(av).reshape(-1)
        if av.size != n_models:
            raise ValueError(f"A_V has {av.size} values for {n_models} models")
        return np.concatenate(ext), av

    def flux_density_series_multi(self, params, datasets, dataset_of, return_status=False):
        """``flux_density_series`` of model m on its own data set ``datasets[dataset_of[m]]`` = (t, nu), t ascending,
        all in one batch.  Returns a list with one float64[5, n_d] array per model (n_d: the size of its data set); the
        arrays are views into one buffer in model order (``vag_flux_density_series_multi``)."""
        p = self._params(params)
        (t, nu), sets, sizes = self._concat_sets(datasets, ("t", "nu"))
        ds = self._dataset_of(dataset_of, p.size)
        n_m = sizes[ds] if p.size else np.zeros(0, dtype=np.int64)
        off = np.concatenate([[0], np.cumsum(n_m)]).astype(np.int64)
        buf = np.empty(abi.NCOMP * int(off[-1]))
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_flux_density_series_multi(self._h, p.ctypes.data, p.size, ds.ctypes.data, C.cast(sets, C.c_void_p),
                                                           len(sets), t.ctypes.data, nu.ctypes.data, t.size, buf.ctypes.data,
                                                           st.ctypes.data))
        out = [buf[abi.NCOMP * off[m]:abi.NCOMP * off[m + 1]].reshape(abi.NCOMP, int(n_m[m])) for m in range(p.size)]
        return (out, st) if return_status else out

    def chi2_multi(self, params, datasets, dataset_of, extinction=None, return_status=False):
        """``chi2_series`` of model m on its own data set ``datasets[dataset_of[m]]`` = (t, nu, lnF_obs, sigma_ln, w), t
        ascending, all in one batch -> chi2[n_models].  ``extinction`` = (ext_k, A_V): one ext_k array per data set (in the
        order of its points) and A_V[n_models]; model m's points are then compared as lnF_obs + A_V[m] * ext_k
        (``vag_chi2_multi``, the rules of ``chi2(extinction=...)``)."""
        p = self._params(params)
        (t, nu, lnF, sig, w), sets, sizes = self._concat_sets(datasets, ("t", "nu", "lnF_obs", "sigma_ln", "w"))
        ds = self._dataset_of(dataset_of, p.size)
        ext, av = self._extinction(extinction, sizes, p.size)
        out = np.empty(p.size)
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_chi2_multi(self._h, p.ctypes.data, p.size, ds.ctypes.data, C.cast(sets, C.c_void_p), len(sets),
                                            t.ctypes.data, nu.ctypes.data, lnF.ctypes.data, sig.ctypes.data, w.ctypes.data,
                                            None if ext is None else ext.ctypes.data, t.size,
                                            None if av is None else av.ctypes.data, out.ctypes.data, st.ctypes.data))
        return (out, st) if return_status else out

    # ---- band-integrated data in a batch of several light curves (vag_flux_band_multi, vag_chi2_multi_bands) ------------
    @staticmethod
    def _band_array(bands, data):
        """``abi.BandObs`` array of band dicts (t, nu_min, nu_max, num_nu; with ``data`` also lnF_obs, sigma_ln, w) and the
        float64 arrays it points into, which must outlive the call."""
        names = ("t", "lnF_obs", "sigma_ln", "w") if data else ("t",)
        arr, keep = (abi.BandObs * max(len(bands), 1))(), []
        for b, band in enumerate(bands):
            cols = [_f64(band[k]).reshape(-1) for k in names]
            if len({a.size for a in cols}) != 1:
                raise ValueError(f"band {b}: arrays {', '.join(names)} must have the same size")
            keep.append(cols)
            ptrs = [a.ctypes.data for a in cols] + [None] * (4 - len(cols))
            arr[b] = abi.BandObs(*ptrs, cols[0].size, float(band["nu_min"]), float(band["nu_max"]), int(band["num_nu"]))
        return arr, keep

    def flux_band_multi(self, params, bands, band_of, return_status=False):
        """``flux_band`` of model m on its own band ``bands[band_of[m]]`` (a dict with t, nu_min, nu_max, num_nu), all in
        one batch.  Returns a list with one float64[5, n_t] array per model (n_t: its band's epochs); the arrays are views
        into one buffer in model order (``vag_flux_band_multi``)."""
        p = self._params(params)
        arr, keep = self._band_array(bands, data=False)
        bo = self._dataset_of(band_of, p.size)
        n_m = np.asarray([keep[b][0].size for b in bo] if p.size and bo.min() >= 0 and bo.max() < len(bands) else
                         np.zeros(p.size), dtype=np.int64)
        off = np.concatenate([[0], np.cumsum(n_m)]).astype(np.int64)
        buf = np.empty(abi.NCOMP * int(off[-1]))
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_flux_band_multi(self._h, p.ctypes.data, p.size, bo.ctypes.data, C.cast(arr, C.c_void_p),
                                                 len(bands), buf.ctypes.data, st.ctypes.data))
        out = [buf[abi.NCOMP * off[m]:abi.NCOMP * off[m + 1]].reshape(abi.NCOMP, int(n_m[m])) for m in range(p.size)]
        return (out, st) if return_status else out

    def chi2_multi_bands(self, params, datasets, bands, dataset_of, extinction=None, return_status=False, exposures=None):
        """``chi2`` of model m on its own data set, all in one batch -> chi2[n_models].  Data set d is its point data
        ``datasets[d]`` = (t, nu, lnF_obs, sigma_ln, w), t ascending, or None when it has none, and its band-integrated data
        ``bands[d]``, a list of ``fitting.band_obs`` dicts (may be empty when it has points).  ``extinction`` = (ext_k, A_V):
        ext_k a list with one array per data set (None for a set without points), A_V[n_models]; model m's points are then
        compared as lnF_obs + A_V[m] * ext_k, its band terms unchanged (``vag_chi2_multi_bands``).  ``exposures``: one
        entry per data set, None or (expo_time, num_points) -- expo_time per point (>= 0, in the order of its points); a
        point with expo_time > 0 is compared with the model averaged over num_points samples of its exposure, as
        ``flux_density_exposures`` computes it (``vag_chi2_multi_bands_exposures``).  None everywhere: the call without."""
        p = self._params(params)
        if len(bands) != len(datasets):
            raise ValueError(f"{len(bands)} band lists for {len(datasets)} data sets")
        cols, n_pts = [[] for _ in range(5)], np.zeros(len(datasets), dtype=np.int64)
        for d, dset in enumerate(datasets):
            if dset is None:
                continue
            arrs = [_f64(a).reshape(-1) for a in dset]
            if len(arrs) != 5 or len({a.size for a in arrs}) != 1:
                raise ValueError(f"data set {d} must be (t, nu, lnF_obs, sigma_ln, w) of one size, or None")
            for c, a in zip(cols, arrs):
                c.append(a)
            n_pts[d] = arrs[0].size
        t, nu, lnF, sig, w = (np.concatenate(c) if c else np.zeros(0) for c in cols)
        pt_off = np.concatenate([[0], np.cumsum(n_pts)]).astype(np.int64)
        flat = [b for bl in bands for b in bl]
        arr, _keep = self._band_array(flat, data=True)
        sets = (abi.MultiSet * max(len(datasets), 1))()
        b0 = 0
        for d in range(len(datasets)):
            sets[d] = abi.MultiSet(int(pt_off[d]), int(n_pts[d]), b0, len(bands[d]))
            b0 += len(bands[d])
        ds = self._dataset_of(dataset_of, p.size)
        ext, av = self._extinction(extinction, n_pts, p.size)
        expo = self._exposures(exposures, n_pts)
        out = np.empty(p.size)
        st = np.zeros(p.size, dtype=np.int32)
        pts = [a.ctypes.data if t.size else None for a in (t, nu, lnF, sig, w)]
        fn, expo_args = self._lib.vag_chi2_multi_bands, ()
        if expo is not None:
            fn, expo_args = self._lib.vag_chi2_multi_bands_exposures, (expo[0].ctypes.data if t.size else None,
                                                                       expo[1].ctypes.data)
        _lib.check(fn(self._h, p.ctypes.data, p.size, ds.ctypes.data, C.cast(sets, C.c_void_p), len(datasets), *pts,
                      None if ext is None else ext.ctypes.data, t.size, None if av is None else av.ctypes.data, *expo_args,
                      C.cast(arr, C.c_void_p) if flat else None, len(flat), out.ctypes.data, st.ctypes.data))
        return (out, st) if return_status else out

    @staticmethod
    def _exposures(exposures, sizes):
        """``exposures`` of a batch of several data sets (one entry per set: None or (expo_time, num_points)) -> (expo_time
        concatenated over the sets, 0 for a set without, int32 num_points[n_sets], 0 for a set without), or None when no
        set has an entry."""
        if exposures is None:
            return None
        if len(exposures) != len(sizes):
            raise ValueError(f"exposures has {len(exposures)} entries for {len(sizes)} data sets")
        if all(e is None for e in exposures):
            return None
        cols, num = [], np.zeros(len(sizes), dtype=np.int32)
        for d, (e, n) in enumerate(zip(exposures, sizes)):
            if e is None:
                cols.append(np.zeros(int(n)))
                continue
            if len(e) != 2:
                raise ValueError(f"data set {d}: exposures must be (expo_time, num_points) or None")
            et, k = _f64(e[0]).reshape(-1), int(e[1])
            if et.size != n:
                raise ValueError(f"data set {d}: expo_time has {et.size} values for {n} points")
            if not -2**31 <= k < 2**31:
                raise ValueError(f"data set {d}: num_points = {k} must fit in a 32-bit int")
            cols.append(et)
            num[d] = k
        return np.concatenate(cols), num

    # ---- a (t x nu) grid per model, and quantiles across models (vag_flux_density_grid_multi, vag_flux_quantiles_multi) --
    @staticmethod
    def _grid_sets(grids):
        """``grids`` = [(t, nu), ...] -> (times and frequencies concatenated over the grids, ``abi.GridSet`` array,
        int64[n_grids, 2] of (n_nu, n_t))."""
        if not len(grids):
            raise ValueError("no grids")
        ts, nus = [], []
        sets = (abi.GridSet * len(grids))()
        shape = np.zeros((len(grids), 2), dtype=np.int64)
        t0 = nu0 = 0
        for d, g in enumerate(grids):
            if len(g) != 2:
                raise ValueError(f"grid {d} must be (t, nu)")
            t, nu = _f64(g[0]).reshape(-1), _f64(g[1]).reshape(-1)
            sets[d] = abi.GridSet(t0, t.size, nu0, nu.size)
            shape[d] = nu.size, t.size
            ts.append(t)
            nus.append(nu)
            t0, nu0 = t0 + t.size, nu0 + nu.size
        return np.concatenate(ts), np.concatenate(nus), sets, shape

    def flux_density_grid_multi(self, params, grids, dataset_of, return_status=False):
        """``flux_density_grid`` of model m on its own grid ``grids[dataset_of[m]]`` = (t, nu), t ascending, all in one
        batch.  Returns a list with one float64[5, n_nu, n_t] array per model; the arrays are views into one buffer in
        model order (``vag_flux_density_grid_multi``)."""
        p = self._params(params)
        t, nu, sets, shape = self._grid_sets(grids)
        ds = self._dataset_of(dataset_of, p.size)
        in_range = p.size and ds.min() >= 0 and ds.max() < len(grids)
        shp = shape[ds] if in_range else np.zeros((p.size, 2), dtype=np.int64)  # (else the call raises)
        off = np.concatenate([[0], np.cumsum(shp[:, 0] * shp[:, 1])]).astype(np.int64)
        buf = np.empty(abi.NCOMP * int(off[-1]))
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_flux_density_grid_multi(self._h, p.ctypes.data, p.size, ds.ctypes.data, C.cast(sets, C.c_void_p),
                                                         len(sets), t.ctypes.data, t.size, nu.ctypes.data, nu.size,
                                                         buf.ctypes.data, st.ctypes.data))
        out = [buf[abi.NCOMP * off[m]:abi.NCOMP * off[m + 1]].reshape(abi.NCOMP, int(shp[m, 0]), int(shp[m, 1]))
               for m in range(p.size)]
        return (out, st) if return_status else out

    def flux_quantiles_multi(self, params, grids, dataset_of, q, return_status=False):
        """Posterior-predictive bands of many fits in one call: for every grid d, ``numpy.quantile`` of the ``total`` flux
        of the models with ``dataset_of == d`` on ``grids[d]`` = (t, nu), at every ``q`` (method "linear"), computed on
        the GPU where the flux is (``vag_flux_quantiles_multi``).  Models whose ODE failed (``abi.ST_ODE_FAIL500``) or
        whose grid exceeded the capacity (``abi.ST_CAPACITY``) are left out.  Returns (a list with one
        float64[n_q, n_nu, n_t] array per grid, int64 n_used[n_grids]: the models each grid's quantiles are over)."""
        p = self._params(params)
        t, nu, sets, shape = self._grid_sets(grids)
        ds = self._dataset_of(dataset_of, p.size)
        qs = _f64(q).reshape(-1)
        cols = shape[:, 0] * shape[:, 1]
        off = np.concatenate([[0], np.cumsum(cols)]).astype(np.int64)
        buf = np.empty(qs.size * int(off[-1]))
        n_used = np.zeros(len(grids), dtype=np.int64)
        st = np.zeros(p.size, dtype=np.int32)
        _lib.check(self._lib.vag_flux_quantiles_multi(self._h, p.ctypes.data, p.size, ds.ctypes.data, C.cast(sets, C.c_void_p),
                                                      len(sets), t.ctypes.data, t.size, nu.ctypes.data, nu.size,
                                                      qs.ctypes.data, qs.size, buf.ctypes.data, n_used.ctypes.data,
                                                      st.ctypes.data))
        bands = [buf[qs.size * off[d]:qs.size * off[d + 1]].reshape(qs.size, int(shape[d, 0]), int(shape[d, 1]))
                 for d in range(len(grids))]
        return (bands, n_used, st) if return_status else (bands, n_used)

    @staticmethod
    def valid_mask(params):
        """bool[n]: which parameter sets pass the constructor checks of the reference (vag_params_validate_batch)."""
        p = np.ascontiguousarray(params, dtype=abi.PARAMS_DTYPE).reshape(-1)
        ok = np.zeros(p.size, dtype=np.int32)
        _lib.check(_lib.load().vag_params_validate_batch(p.ctypes.data, p.size, ok.ctypes.data))
        return ok.astype(bool)

    # ---- device buffers (raw pointers) ---------------------------------------------------------
    def flux_density_grid_dev(self, d_params, n_models, d_t, n_t, d_nu, n_nu, d_out, d_status=0, stream=0):
        _lib.check(self._lib.vag_flux_density_grid_dev(self._h, d_params, n_models, d_t, n_t, d_nu, n_nu, d_out,
                                                       d_status or None, stream or None))

    def flux_density_series_dev(self, d_params, n_models, d_t, d_nu, n, d_out, d_status=0, stream=0):
        _lib.check(self._lib.vag_flux_density_series_dev(self._h, d_params, n_models, d_t, d_nu, n, d_out,
                                                         d_status or None, stream or None))

    def chi2_series_dev(self, d_params, n_models, d_t, d_nu, d_lnF, d_sig, d_w, n, d_chi2, d_status=0, stream=0):
        _lib.check(self._lib.vag_chi2_series_dev(self._h, d_params, n_models, d_t, d_nu, d_lnF, d_sig, d_w, n, d_chi2,
                                                 d_status or None, stream or None))

    def validate_dev(self, d_params, n, d_ok, stream=0):
        """``vag_params_validate_batch_dev``: int32 ok flags into ``d_ok``; returns the planned (theta, phi) capacities.
        Synchronises the stream."""
        caps = (C.c_int * 2)()
        _lib.check(self._lib.vag_params_validate_batch_dev(self._h, d_params, n, d_ok, caps, stream or None))
        return int(caps[0]), int(caps[1])

    def flux_band_dev(self, d_params, n_models, d_t, n_t, nu_min, nu_max, num_nu, d_out, d_status=0, stream=0):
        """``vag_flux_band_dev``: ``Model.flux`` into d_out[n_models, 5, n_t]; parameters checked and grids sized on the
        device (rejected sets: NaN, ``abi.ST_INVALID``)."""
        _lib.check(self._lib.vag_flux_band_dev(self._h, d_params, n_models, d_t, n_t, float(nu_min), float(nu_max),
                                               int(num_nu), d_out, d_status or None, stream or None))

    @staticmethod
    def _band_array_dev(bands):
        """``abi.BandObs`` array of band dicts whose t, lnF_obs, sigma_ln, w are device pointers of length ``n``."""
        arr = (abi.BandObs * max(len(bands), 1))()
        for i, b in enumerate(bands):
            arr[i] = abi.BandObs(b["t"], b["lnF_obs"], b["sigma_ln"], b["w"], int(b["n"]), float(b["nu_min"]),
                                 float(b["nu_max"]), int(b["num_nu"]))
        return arr

    def chi2_dev(self, d_params, n_models, points=None, bands=(), d_chi2=0, d_status=0, extinction=None, stream=0):
        """``vag_chi2_dev``: the likelihood of ``chi2`` on device pointers.  ``points`` = (d_t, d_nu, d_lnF, d_sig, d_w,
        n_points) or None; ``bands``: dicts like ``chi2``'s whose t, lnF_obs, sigma_ln, w are device pointers with their
        length ``n``; ``extinction`` = (d_ext_k, d_A_V).  Rejected parameter sets give chi2 = +inf and ``abi.ST_INVALID``."""
        pts, n_pt = ([None] * 5, 0) if points is None else (list(points[:5]), int(points[5]))
        ext, av = (None, None) if extinction is None else extinction
        arr = self._band_array_dev(bands)
        _lib.check(self._lib.vag_chi2_dev(self._h, d_params, n_models, *pts, ext, n_pt, av,
                                          C.cast(arr, C.c_void_p) if len(bands) else None, len(bands), d_chi2,
                                          d_status or None, stream or None))

    def chi2_multi_bands_dev(self, d_params, n_models, dataset_of, sets, points, bands, d_chi2, d_status=0, extinction=None,
                             stream=0):
        """``vag_chi2_multi_bands_dev``: ``chi2_multi_bands`` on device pointers, each record checked on the device
        (rejected ones: chi2 = +inf, ``abi.ST_INVALID``; they are left out of the batch).  ``dataset_of`` (int32 per
        model) and ``sets`` -- ``(offset, n, band0, n_bands)`` tuples or an ``abi.MultiSet`` array -- are host arrays;
        ``points`` = (d_t, d_nu, d_lnF, d_sig, d_w, n_points_total) of the concatenated points, or None; ``bands``: the
        concatenated band dicts of all sets, as ``chi2_dev``'s (device pointers t, lnF_obs, sigma_ln, w and their length
        ``n``); ``extinction`` = (d_ext_k, d_A_V).  Returns with the work enqueued on ``stream``."""
        pts, n_pt = ([None] * 5, 0) if points is None else (list(points[:5]), int(points[5]))
        ext, av = (None, None) if extinction is None else extinction
        if isinstance(sets, C.Array) and sets._type_ is abi.MultiSet:
            arr_sets, n_sets = sets, len(sets)
        else:
            sets = list(sets)
            arr_sets, n_sets = (abi.MultiSet * max(len(sets), 1))(), len(sets)
            for d, s in enumerate(sets):
                arr_sets[d] = abi.MultiSet(*(int(v) for v in s))
        ds = self._dataset_of(dataset_of, int(n_models))
        arr = self._band_array_dev(bands)
        _lib.check(self._lib.vag_chi2_multi_bands_dev(self._h, d_params, int(n_models), ds.ctypes.data,
                                                      C.cast(arr_sets, C.c_void_p) if n_sets else None, n_sets, *pts, ext,
                                                      n_pt, av, C.cast(arr, C.c_void_p) if len(bands) else None, len(bands),
                                                      d_chi2, d_status or None, stream or None))

    def synchronize(self):
        _lib.check(self._lib.vag_synchronize(self._h))

    def set_capacity(self, cap_theta, cap_phi):
        _lib.check(self._lib.vag_set_capacity(self._h, int(cap_theta), int(cap_phi)))

    def set_output_mode(self, present_only: bool, alias_total: bool = False):
        """True: host-buffer calls skip the planes of components no model of the batch has (vag.h VAG_OUT_PRESENT);
        alias_total: additionally skip `total` when it equals the batch's only component (``last_total_alias()``)."""
        _lib.check(self._lib.vag_set_output_mode(self._h, (2 if alias_total else 1) if present_only else 0))
        self._present_only = bool(present_only)

    def set_series_mode(self, mode: int):
        """Evaluation of series requests with <= 8 distinct frequencies (vag.h vag_set_series_mode): 0 auto (default),
        1 per-point spectra always, 2 banded whenever possible."""
        _lib.check(self._lib.vag_set_series_mode(self._h, int(mode)))

    def set_grid_lanes(self, lanes: int):
        """Lanes per model of the grid builder (vag.h vag_set_grid_lanes): 0 by batch size (default), or 4 / 8 / 16 / 32 for
        every batch.  The grid is the same bit for bit at every width."""
        _lib.check(self._lib.vag_set_grid_lanes(self._h, int(lanes)))

    def last_total_alias(self):
        """Index into ``abi.COMPONENTS`` of the plane that holds `total` after the last host call, or -1."""
        return int(self._lib.vag_last_total_alias(self._h))

    def debug_set_ode_limits(self, max_steps=0, max_fails=0):
        """Test hook (include/vag.h vag_debug_set_ode_limits): 0 restores the reference limits."""
        _lib.check(self._lib.vag_debug_set_ode_limits(self._h, int(max_steps), int(max_fails)))

    def set_profiling(self, on=True):
        _lib.check(self._lib.vag_set_profiling(self._h, 1 if on else 0))

    def last_stage_ms(self):
        ms = (C.c_float * 8)()
        self._lib.vag_last_stage_ms(self._h, ms)
        names = ("grid", "dynamics", "radiation", "eats", "finish")
        return {k: float(ms[i]) for i, k in enumerate(names)}

    def last_work(self):
        """Work counters of the last profiled pass (include/vag.h vag_last_work)."""
        w = (C.c_double * 8)()
        self._lib.vag_last_work(self._h, w)
        names = ("rows_fwd", "rows_pair", "cells", "eats_cells", "eats_rows", "quad_attempts_theta", "quad_phi_evals", "sum_n_theta")
        return {k: float(w[i]) for i, k in enumerate(names)}

    def measure_fp64_peak(self):
        v = C.c_double()
        _lib.check(self._lib.vag_measure_fp64_peak(self._h, C.byref(v)))
        return float(v.value)

    LIBM_FUNCS = ("exp", "exp2", "log", "log2", "log10", "pow", "sin", "cos")

    def selftest_libm(self, fn, x, y=None):
        """Device evaluation of one libm-exact function of csrc/vag_libm.cuh (include/vag.h vag_selftest_libm)."""
        x = _f64(x).reshape(-1)
        out = np.empty_like(x)
        yv = None if y is None else _f64(y).reshape(-1)
        _lib.check(self._lib.vag_selftest_libm(self._h, self.LIBM_FUNCS.index(fn), x.ctypes.data,
                                               None if yv is None else yv.ctypes.data, out.ctypes.data, x.size))
        return out

    def last_launch_count(self):
        return int(self._lib.vag_last_launch_count(self._h))

    def details(self, param, t_min, t_max):
        """Stage tables of one model (code units) -- the analogue of ``Model.details``."""
        p = self._params(param)
        assert p.size == 1
        info = np.zeros(1, dtype=abi.GRID_INFO_DTYPE)
        f = self._lib.vag_details
        _lib.check(f(self._h, p.ctypes.data, t_min, t_max, info.ctypes.data, *([None] * 7)))
        i = info[0]
        n_phi, n_theta, n_t, n_reps = (int(i[k]) for k in ("n_phi", "n_theta", "n_t", "n_reps"))
        d = {
            "info": i,
            "theta": np.zeros(n_theta),
            "phi": np.zeros(n_phi),
            "reps": np.zeros(n_reps, dtype=np.int32),
            "t_rows": np.zeros((n_reps, n_t)),
            "fwd_shock": np.zeros((7, n_reps, n_t)),
            "rvs_shock": np.zeros((7, n_reps, n_t)),
            "inj_idx": np.zeros(n_reps, dtype=np.int32),
        }
        _lib.check(f(self._h, p.ctypes.data, t_min, t_max, info.ctypes.data, d["theta"].ctypes.data,
                     d["phi"].ctypes.data, d["reps"].ctypes.data, d["t_rows"].ctypes.data,
                     d["fwd_shock"].ctypes.data, d["rvs_shock"].ctypes.data, d["inj_idx"].ctypes.data))
        return d

    def details_ic(self, param, t_min, t_max, n_reps, n_t):
        """Electron / inverse-Compton records of the ssc=True shocks: (fwd, rvs) each [7, n_reps, n_t] -- gamma_m, gamma_c,
        gamma_a, gamma_M, gamma_m_hat, gamma_c_hat, Y_T (include/vag.h vag_details_ic); zero for shocks without ssc."""
        p = self._params(param)
        assert p.size == 1
        fwd = np.zeros((7, n_reps, n_t))
        rvs = np.zeros((7, n_reps, n_t))
        _lib.check(self._lib.vag_details_ic(self._h, p.ctypes.data, t_min, t_max, fwd.ctypes.data, rvs.ctypes.data))
        return fwd, rvs

    def details_photons(self, param, t_min, t_max, n_reps, n_t):
        """Photon tables of one model: (fwd, rvs) each [6, n_reps, n_t] -- log2 nu_m, nu_c, nu_a, nu_M, I_nu_max (code
        units) and 1/nu_M (include/vag.h vag_details_photons)."""
        p = self._params(param)
        assert p.size == 1
        fwd = np.zeros((6, n_reps, n_t))
        rvs = np.zeros((6, n_reps, n_t))
        _lib.check(self._lib.vag_details_photons(self._h, p.ctypes.data, t_min, t_max, fwd.ctypes.data, rvs.ctypes.data))
        return fwd, rvs
