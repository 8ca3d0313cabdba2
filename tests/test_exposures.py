"""Exposure-averaged flux densities on the GPU: vag_flux_density_exposures (Engine / Model.flux_density_exposures) and
exposure-averaged points in the ragged likelihood (vag_chi2_multi_bands_exposures, BatchedLikelihood(expo_time=...),
the likelihood stacks).

GPU tier: the reference fixture; equality with the host composition the call replaces (series on the sorted samples,
np.add.at, / k) on a mixed batch in every series mode and both output modes, with unsorted times and shared sample times;
launch counts; with no exposure the chi-squared equals vag_chi2_multi_bands; with exposures it equals a numpy restatement
and, for a set of exposures only, the values of vag_flux_density_exposures; stacks against each fit alone; an ODE failure;
a long banded set of samples; the 32768-model pass boundary; argument checks.
CPU tier: the sample plan and averaging body of csrc/vag_exposure.cuh against numpy; BatchedLikelihood's checks; the
stacks with a recording engine.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests.test_multi_band import XRAY, _band
from tests.test_multi_band import _datasets as _band_datasets
from tests.test_multi_dataset import _LOG, _NAMES, UNSPLIT_MODELS, _light_curve, _models, _padded, _raw_points, _samples
from vegasafterglow_b200 import abi, configs, fitting

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "vegasafterglow_b200", "csrc")


# ---- the rule, restated in numpy ----------------------------------------------------------------------------------------
def _expand(t, nu, e, k):
    """The samples of one set (vag_exposure.cuh): (sorted times, their frequencies, the point of each, its count)."""
    ts, of = [], []
    for i in range(t.size):
        if e[i] > 0:
            ts.append(t[i] + np.arange(k, dtype=np.float64) * (e[i] / (k - 1)))
            of.append(np.full(k, i))
        else:
            ts.append(t[i:i + 1])
            of.append(np.array([i]))
    ts, of = np.concatenate(ts), np.concatenate(of)
    order = np.argsort(ts, kind="stable")
    return ts[order], nu[of[order]], of[order], np.bincount(of, minlength=t.size)


def _average(f, of, count):
    """f[..., samples] -> the averages [..., points]: np.add.at in sorted order, then / count."""
    out = np.zeros(f.shape[:-1] + (count.size,))
    np.add.at(out, (Ellipsis, of), f)
    return out / count


def _host_composition(engine, P, t, nu, e, k):
    """What Engine.flux_density_exposures computed before: the series on the sorted samples, np.add.at, / k."""
    kk = np.arange(k, dtype=np.float64)
    ts = (t[:, None] + kk[None, :] * (e / (k - 1))[:, None]).reshape(-1)
    nus, idx = np.repeat(nu, k), np.repeat(np.arange(t.size), k)
    order = np.argsort(ts, kind="stable")
    f, st = engine.flux_density_series(P, ts[order], nus[order], return_status=True)
    out = np.zeros((f.shape[0], abi.NCOMP, t.size))
    np.add.at(out, (slice(None), slice(None), idx[order]), f)
    out /= float(k)
    return out, st


def _chi2_rule(F, lnF, sig, w, ext=None, av=0.0):
    obs = lnF if ext is None else lnF + av * ext
    return np.sum(w * ((obs - np.log(np.maximum(F, 1e-300))) / sig) ** 2)


# ---- GPU tier -----------------------------------------------------------------------------------------------------------
def _mixed_batch():
    """FS tophat, FS+RS, Gaussian off-axis and SSC models"""
    P = np.concatenate([configs.random_draw(6, seed=1), configs.random_draw(6, seed=2, rvs=True),
                        configs.random_draw(6, seed=3, jet="gaussian", theta_obs_max=0.4),
                        configs.random_draw(3, seed=4, ssc=True, kn=True)])
    P["t_resol"] = 3.0
    return P


def _exposure_points():
    """Unsorted times in three bands; point 1's samples include t of point 4 (150 = 100 + 5 * 10) and point 5 starts at
    point 1's last sample (190)."""
    t = np.array([3e4, 100.0, 2e3, 7e5, 150.0, 190.0, 1e4, 5e2, 2e5])
    nu = np.array([1e9, 4.84e14, 1e18, 1e9, 4.84e14, 1e18, 4.84e14, 1e9, 1e18])
    e = np.array([5e3, 90.0, 400.0, 1e5, 30.0, 1.0, 2e3, 50.0, 3e4])
    return t, nu, e


@pytest.mark.gpu
def test_reference_fixture_through_the_device_average(engine):
    from tests.helpers import load_golden

    g = load_golden("method_exposures")
    f, st = engine.flux_density_exposures(g["params"], g["t"], g["nu"], g["expo"], int(g["num_points"]), return_status=True)
    assert not (st & abi.ST_ODE_FAIL500).any()
    for c, theirs in zip((0, 1, 3), g["flux"]):
        err = np.max(np.abs(f[0, c] - theirs) / np.abs(theirs))
        assert err <= 1e-6, (c, err)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("present_only", [False, True])
def test_flux_density_exposures_equals_the_host_composition(engine, mode, present_only):
    P = _mixed_batch()
    t, nu, e = _exposure_points()
    k = 10
    try:
        engine.set_series_mode(mode)
        engine.set_output_mode(present_only)
        want, q = _host_composition(engine, P, t, nu, e, k)
        n_series = engine.last_launch_count()
        got, st = engine.flux_density_exposures(P, t, nu, e, k, return_status=True)
        assert engine.last_launch_count() == n_series + 1
    finally:
        engine.set_series_mode(0)
        engine.set_output_mode(False)
    assert np.array_equal(st, q)
    assert np.array_equal(got, want, equal_nan=True)
    assert np.isfinite(got[:, 0]).all() and (got[:, 0] > 0).all()


@pytest.mark.gpu
def test_mirror_uses_the_device_average(engine):
    from vegasafterglow_b200 import VegasAfterglowC_b200 as va

    m = va.Model(jet=va.TophatJet(0.1, 1e52, 300, duration=1e3), medium=va.ISM(1), observer=va.Observer(1e27, 0.5, 0),
                 fwd_rad=va.Radiation(0.1, 1e-3, 2.3), rvs_rad=va.Radiation(0.1, 1e-2, 2.5))
    P = configs.make(duration=1e3, lumi_dist=1e27, z=0.5, rvs=(0.1, 1e-2, 2.5))
    t, nu, e = _exposure_points()
    fe = m.flux_density_exposures(t, nu, e, 7)
    want, _ = _host_composition(engine, P, t, nu, e, 7)
    assert np.array_equal(fe.total, want[0, 0]) and np.array_equal(fe.rvs.sync, want[0, 3])
    for bad, word in (((t, nu, -e, 7), "expo_time[0] must be finite and > 0"), ((t, nu, e, 1), "num_points"),
                      ((t, nu[:3], e, 7), "same size")):
        with pytest.raises(ValueError, match=word.replace("[", r"\[").replace("]", r"\]")):
            m.flux_density_exposures(*bad)


def _expanded_sets(pts, exposures):
    """The sets of samples of vag_chi2_multi_bands_exposures: per set (t, nu, point of each sample, counts) or None."""
    out = []
    for p, ex in zip(pts, exposures):
        if p is None:
            out.append(None)
            continue
        e, k = ex if ex is not None else (np.zeros(p[0].size), 2)
        out.append(_expand(p[0], p[1], e, k))
    return out


def _restated_point_chi2(engine, P, ds, pts, exposures, ext=None, A_V=None):
    """The point term of every model whose set has points: flux_density_series_multi on the sets of samples (the same
    batch as the point pass), averaged, then the chi-squared rule with A_V."""
    X = _expanded_sets(pts, exposures)
    keep = [d for d in range(len(pts)) if pts[d] is not None]
    remap = {d: i for i, d in enumerate(keep)}
    m_pt = np.nonzero([pts[d] is not None for d in ds])[0]
    flux = engine.flux_density_series_multi(P[m_pt], [X[d][:2] for d in keep], np.array([remap[d] for d in ds[m_pt]]))
    out = {}
    for j, m in enumerate(m_pt):
        d = ds[m]
        F = _average(flux[j][0], X[d][2], X[d][3])
        e_k = None if ext is None else ext[d]
        out[m] = _chi2_rule(F, pts[d][2], pts[d][3], pts[d][4], e_k, 0.0 if A_V is None else A_V[m])
    return out


def _raw_multi_expo(engine, P, ds, sets, pts, expo, num, bands=(), ext=None, A_V=None):
    """engine.chi2_multi_bands's arguments to vag_chi2_multi_bands_exposures with sentinel outputs -> (rc, untouched)"""
    P = np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE)
    ds = np.ascontiguousarray(ds, dtype=np.int32)
    arr = (abi.MultiSet * max(len(sets), 1))(*[abi.MultiSet(*s) for s in sets])
    t, nu = pts
    lnF, sig, w = np.zeros(t.size), np.ones(t.size), np.ones(t.size)
    keep = [[np.asarray(b["t"], dtype=np.float64), np.zeros(len(b["t"])), np.ones(len(b["t"])), np.ones(len(b["t"]))]
            for b in bands]
    barr = (abi.BandObs * max(len(bands), 1))(*[abi.BandObs(*[a.ctypes.data for a in k], k[0].size, b["nu_min"], b["nu_max"],
                                                            b["num_nu"]) for k, b in zip(keep, bands)])
    chi2 = np.full(P.size, 7.0)
    st = np.full(P.size, 99, dtype=np.int32)
    rc = engine._lib.vag_chi2_multi_bands_exposures(
        engine._h, P.ctypes.data, P.size, ds.ctypes.data, C.cast(arr, C.c_void_p) if sets else None, len(sets),
        *[a.ctypes.data for a in (t, nu, lnF, sig, w)], None if ext is None else ext.ctypes.data, t.size,
        None if A_V is None else A_V.ctypes.data, None if expo is None else expo.ctypes.data,
        None if num is None else num.ctypes.data, C.cast(barr, C.c_void_p) if bands else None, len(bands),
        chi2.ctypes.data, st.ctypes.data)
    return rc, bool((chi2 == 7.0).all() and (st == 99).all())


def _chi2_batch():
    P, _ = _models(n_per_kind=300, seed=30)
    ds = np.random.default_rng(31).integers(0, 4, P.size).astype(np.int32)  # set 4: no model
    pts, bands = _band_datasets(3)  # 0 points + bands, 1 bands only, 2 and 3 points only, 4 unused
    rng = np.random.default_rng(32)
    ext = [None if p is None else rng.uniform(0.0, 1.7, p[0].size) for p in pts]
    ext[2] = np.zeros(pts[2][0].size)  # A_V on sets 0 and 3 only
    A_V = rng.uniform(0.0, 2.0, P.size)
    return P, ds, pts, bands, ext, A_V


@pytest.mark.gpu
@pytest.mark.parametrize("extinction", [False, True])
def test_without_exposures_equals_chi2_multi_bands(engine, extinction):
    P, ds, pts, bands, ext, A_V = _chi2_batch()
    kw = dict(extinction=(ext, A_V)) if extinction else {}
    zero = [None if p is None else (np.zeros(p[0].size), 10) for p in pts]
    want, q = engine.chi2_multi_bands(P, pts, bands, ds, return_status=True, **kw)
    n_plain = engine.last_launch_count()
    got, st = engine.chi2_multi_bands(P, pts, bands, ds, return_status=True, exposures=zero, **kw)
    assert engine.last_launch_count() == n_plain + 1
    assert np.array_equal(got, want) and np.array_equal(st, q)
    assert np.isfinite(got).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [1, 2])
def test_with_exposures_equals_numpy_restatement(engine, mode):
    P, ds, pts, bands, ext, A_V = _chi2_batch()
    rng = np.random.default_rng(33)
    e0 = rng.uniform(0.05, 0.5, pts[0][0].size) * pts[0][0]
    e0[::3] = 0.0  # points without an exposure among points with one
    exposures = [(e0, 5), None, None, (0.3 * pts[3][0], 3), None]
    try:
        engine.set_series_mode(mode)
        got, st = engine.chi2_multi_bands(P, pts, bands, ds, extinction=(ext, A_V), exposures=exposures,
                                          return_status=True)
        n_expo = engine.last_launch_count()
        # the launches of vag_chi2_multi_bands on the sets of samples, + 1
        X = _expanded_sets(pts, exposures)
        x_pts = [None if x is None else (x[0], x[1], *(np.zeros(x[0].size),) * 2, np.ones(x[0].size)) for x in X]
        engine.chi2_multi_bands(P, x_pts, bands, ds)
        assert n_expo == engine.last_launch_count() + 1
        point = _restated_point_chi2(engine, P, ds, pts, exposures, ext, A_V)
        band_only = engine.chi2_multi_bands(P, [None] * len(pts), [b if b else [_band([1e4], *XRAY, 5)] for b in bands], ds)
    finally:
        engine.set_series_mode(0)
    for m in range(P.size):
        d = ds[m]
        want = point.get(m, 0.0) + (band_only[m] if bands[d] else 0.0)
        np.testing.assert_allclose(got[m], want, rtol=1e-12, atol=0, err_msg=str((m, d)))
    assert np.isfinite(got).all() and not (st & abi.ST_ODE_FAIL500).any()


@pytest.mark.gpu
def test_a_set_of_exposures_gives_the_values_of_flux_density_exposures(engine):
    t, nu, lnF, sig, w = _light_curve(np.logspace(3, 6, 12), np.tile([1e9, 4.84e14, 1e18], 4), 40)
    e = 0.2 * t
    P = configs.random_draw(UNSPLIT_MODELS, seed=41)
    P["t_resol"] = 3.0
    ds = np.zeros(P.size, dtype=np.int32)
    try:
        engine.set_series_mode(1)
        got = engine.chi2_multi_bands(P, [(t, nu, lnF, sig, w)], [[]], ds, exposures=[(e, 6)])
        F = engine.flux_density_exposures(P, t, nu, e, 6)
    finally:
        engine.set_series_mode(0)
    want = np.array([_chi2_rule(F[m, 0], lnF, sig, w) for m in range(P.size)])
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)


def _expo_fits(engine, n_walkers):
    """Four fits: points with exposures (k = 10), an X-ray band and A_V; bands only; points with exposures (k = 3),
    some zero; points without exposures."""
    specs = [(configs.make(lumi_dist=1e28, z=0.3), True, _raw_points(1), [_band(np.logspace(3, 5.5, 8), *XRAY, 5, 1)], 10),
             (configs.make(jet="gaussian", rvs=(0.1, 0.01, 2.3), lumi_dist=1e28, z=0.3, theta_obs=0.05), False, None,
              [_band(np.logspace(3.5, 6, 6), *XRAY, 5, 2)], None),
             (configs.make(lumi_dist=3e27, z=0.1), False, _raw_points(3, 12, (1e9, 5e9, 4.84e14, 1e17)), [], 3),
             (configs.make(lumi_dist=1e28, z=0.3), False, _raw_points(4, 8, (5e9, 1e17)), [], None)]
    fits, samples = [], []
    for k, (tmpl, av, pts, bands, kk) in enumerate(specs):
        tmpl["t_resol"] = 3.0
        s = _samples(n_walkers, 70 + k, av)
        names, log = _NAMES + (["A_V"] if av else []), _LOG + ([False] if av else [])
        t, nu, flux, err, ext = pts if pts is not None else (np.zeros(0),) * 5
        raw_bands = [dict(t=b["t"], flux=np.exp(b["lnF_obs"]), err=np.exp(b["lnF_obs"]) * b["sigma_ln"], nu_min=b["nu_min"],
                          nu_max=b["nu_max"], num_points=b["num_nu"]) for b in bands]
        expo = None
        if kk is not None:
            expo = 0.25 * t
            expo[::4] = 0.0
        fits.append(fitting.BatchedLikelihood(engine, tmpl, names, log, t, nu, flux, err, bands=raw_bands,
                                              ext_kernel=ext if av else None, expo_time=expo, expo_points=kk or 10))
        samples.append(s)
    return fits, samples


@pytest.mark.gpu
def test_stacks_equal_each_likelihood_alone(engine):
    fits, samples = _expo_fits(engine, UNSPLIT_MODELS)
    try:
        engine.set_series_mode(1)
        want = [lk(s) for lk, s in zip(fits, samples)]
        got = fitting.BandLikelihoodStack(fits)(samples)
        point_fits = [fits[0], fits[2], fits[3]]
        got_pts = fitting.LikelihoodStack([fitting.BatchedLikelihood(engine, lk.template, lk.names, lk.log_scale, lk.t, lk.nu,
                                                                     np.exp(lk.lnF), np.exp(lk.lnF) * lk.sig, lk.w,
                                                                     ext_kernel=lk.ext_kernel, expo_time=lk.expo_time,
                                                                     expo_points=lk.expo_points)
                                           for lk in point_fits])([samples[0], samples[2], samples[3]])
        want_pts = [fitting.BatchedLikelihood(engine, lk.template, lk.names, lk.log_scale, lk.t, lk.nu, np.exp(lk.lnF),
                                              np.exp(lk.lnF) * lk.sig, lk.w, ext_kernel=lk.ext_kernel,
                                              expo_time=lk.expo_time, expo_points=lk.expo_points)(s)
                    for lk, s in zip(point_fits, [samples[0], samples[2], samples[3]])]
    finally:
        engine.set_series_mode(0)
    for g, w in zip(got + got_pts, want + want_pts):
        np.testing.assert_allclose(g, w, rtol=1e-12, atol=0)
        assert np.isfinite(w).sum() >= UNSPLIT_MODELS // 2


@pytest.mark.gpu
def test_ode_failure_gives_inf(engine):
    P, ds, pts, bands, ext, A_V = _chi2_batch()
    exposures = [(0.2 * pts[0][0], 4), None, (0.1 * pts[2][0], 2), None, None]
    try:
        engine.debug_set_ode_limits(0, 1)
        got, st = engine.chi2_multi_bands(P, pts, bands, ds, exposures=exposures, return_status=True)
    finally:
        engine.debug_set_ode_limits(0, 0)
    fail = (st & abi.ST_ODE_FAIL500) != 0
    assert fail[np.isin(ds, (0, 2))].any()
    assert np.isposinf(got[fail]).all() and np.isfinite(got[~fail]).all()


@pytest.mark.gpu
def test_long_banded_set_of_samples(engine):
    t, nu, lnF, sig, w = _light_curve(np.repeat(np.logspace(2.5, 6.5, 100), 3), np.tile([1e9, 4.84e14, 1e18], 100), 50)
    e = 0.05 * t
    P = configs.random_draw(256, seed=51, rvs=True)
    ds = np.zeros(P.size, dtype=np.int32)
    pts, exposures = [(t, nu, lnF, sig, w)], [(e, 10)]
    try:
        engine.set_series_mode(2)
        got, st = engine.chi2_multi_bands(P, pts, [[]], ds, exposures=exposures, return_status=True)
        want = _restated_point_chi2(engine, P, ds, pts, exposures)
    finally:
        engine.set_series_mode(0)
    assert _expanded_sets(pts, exposures)[0][0].size == 3000
    np.testing.assert_allclose(got, [want[m] for m in range(P.size)], rtol=1e-12, atol=0)
    assert np.isfinite(got).all()


@pytest.mark.gpu
def test_pass_boundary(engine):
    P = configs.random_draw(32768 + 64, seed=61)
    P["t_resol"] = 3.0
    t, nu, lnF, sig, w = _light_curve([1e3, 1e4], [1e9, 1e17], 60)
    ds = np.zeros(P.size, dtype=np.int32)
    args = ([(t, nu, lnF, sig, w)], [[]])
    expo = [(np.array([100.0, 0.0]), 3)]
    got = engine.chi2_multi_bands(P, *args, ds, exposures=expo)
    first = engine.chi2_multi_bands(P[:32768], *args, ds[:32768], exposures=expo)
    second = engine.chi2_multi_bands(P[32768:], *args, ds[32768:], exposures=expo)
    assert np.array_equal(got, np.concatenate([first, second]))
    assert np.isfinite(got).all()


@pytest.mark.gpu
def test_arguments_are_validated_before_any_work(engine):
    P = configs.random_draw(4, seed=1)
    # vag_flux_density_exposures
    t, nu, e = _exposure_points()

    def flux(t=t, nu=nu, e=e, k=5, n=None):
        out = np.full((P.size, abi.NCOMP, t.size), 7.0)
        st = np.full(P.size, 99, dtype=np.int32)
        rc = engine._lib.vag_flux_density_exposures(engine._h, P.ctypes.data, P.size, t.ctypes.data, nu.ctypes.data,
                                                    e.ctypes.data, t.size if n is None else n, k, out.ctypes.data,
                                                    st.ctypes.data)
        return rc, bool((out == 7.0).all() and (st == 99).all())

    assert flux()[0] == abi.VAG_OK
    neg, nan_t, inf_nu = e.copy(), t.copy(), nu.copy()
    neg[2], nan_t[3], inf_nu[4] = -1.0, np.nan, np.inf
    cases = {"num_points must be at least 2": dict(k=1), "expo_time[2] must be finite and > 0, got -1.0": dict(e=neg),
             "time array must be non-empty": dict(n=0), "observation times must be finite": dict(t=nan_t),
             "observation frequencies must be finite": dict(nu=inf_nu), "32-bit int": dict(k=2**31),
             "observation times must be finite and > 0": dict(t=np.full(t.size, 1.7e308), e=np.full(t.size, 1.7e308))}
    for word, kw in cases.items():
        rc, untouched = flux(**kw)
        msg = engine._lib.vag_last_error().decode()
        assert rc == abi.VAG_ERR_INVALID and untouched and word in msg, (word, msg)
    with pytest.raises(ValueError, match="same size"):
        engine.flux_density_exposures(P, t, nu[:3], e)
    # vag_chi2_multi_bands_exposures
    tp = np.array([1e3, 1e4, 1e5, 2e3, 2e4, 2e5])
    pts = (tp, np.full(tp.size, 1e9))
    sets = [(0, 3, 0, 0), (3, 3, 0, 1), (0, 0, 1, 1)]
    xb = dict(t=[1e3, 1e4], nu_min=XRAY[0], nu_max=XRAY[1], num_nu=5)
    ds = np.array([0, 1, 2, 0])
    expo, num = np.array([0.0, 10.0, 0.0, 0.0, 0.0, 0.0]), np.array([2, 0, 0], dtype=np.int32)
    assert _raw_multi_expo(engine, P, ds, sets, pts, expo, num, [xb, xb])[0] == abi.VAG_OK
    bad_e, big_e, late = expo.copy(), expo.copy(), (np.array([1e3, 1e4, 1.7e308, 2e3, 2e4, 2e5]), pts[1])
    bad_e[4], big_e[2] = -2.0, 1.7e308
    cases = {"point 4: expo_time": dict(expo=bad_e), "data set 1: num_expo = 0": dict(expo=expo[::-1].copy()),
             "expo_time is NULL": dict(expo=None), "num_expo is NULL": dict(num=None),
             "data set 0: point 2: its last sample time is not finite": dict(pts=late, expo=big_e),
             "32-bit int": dict(num=np.array([2**31 - 1, 0, 0], dtype=np.int32)),
             "no data sets": dict(sets=[]), "model 2: dataset_of": dict(ds=np.array([0, 1, 3, 0]))}
    for word, kw in cases.items():
        args = dict(P=P, ds=ds, sets=sets, pts=pts, expo=expo, num=num, bands=[xb, xb])
        args.update(kw)
        rc, untouched = _raw_multi_expo(engine, args.pop("P"), args.pop("ds"), args.pop("sets"), args.pop("pts"),
                                        args.pop("expo"), args.pop("num"), **args)
        msg = engine._lib.vag_last_error().decode()
        assert rc == abi.VAG_ERR_INVALID and untouched and word in msg, (word, msg)
    with pytest.raises(ValueError, match="data set 0: expo_time has 2 values"):
        engine.chi2_multi_bands(P, [_light_curve([1e3, 1e4, 1e5], [1e9] * 3, 0)], [[]], np.zeros(4, dtype=np.int32),
                                exposures=[(np.zeros(2), 3)])
    # a failed call leaves the engine usable
    assert _raw_multi_expo(engine, P, ds, sets, pts, expo, num, [xb, xb])[0] == abi.VAG_OK
    assert flux()[0] == abi.VAG_OK


# ---- CPU tier -----------------------------------------------------------------------------------------------------------
_SHIM = r"""
#include "vag_exposure.cuh"
// one set: the samples (t, nu), the plan (s0[n + 1], pos[samples]) and the averages of f[comp][samples] per point
extern "C" int expo_plan(const double* t, const double* nu, const double* e, int n, int k, double* ts, double* nus,
                         int* s0, int* pos) {
    vag::ExpoPlan P;
    vag::expo_plan_append(t, nu, e, (size_t)n, k, P);
    for (size_t i = 0; i < P.t.size(); ++i) { ts[i] = P.t[i]; nus[i] = P.nu[i]; pos[i] = P.pos[i]; }
    for (size_t i = 0; i < P.s0.size(); ++i) s0[i] = P.s0[i];
    return (int)P.t.size();
}
extern "C" void expo_average(const double* f, int n_s, const int* s0, const int* pos, int n, int n_comp, double* out) {
    for (int c = 0; c < n_comp; ++c)
        for (int i = 0; i < n; ++i) out[c * n + i] = vag::expo_mean(f + (size_t)c * n_s, pos + s0[i], s0[i + 1] - s0[i]);
}
"""


@pytest.fixture(scope="module")
def expo_host(tmp_path_factory):
    d = tmp_path_factory.mktemp("expo")
    src, so = d / "expo.cpp", d / "libexpo.so"
    src.write_text(_SHIM)
    # the host emulation's flags (oracle/hostemu/emu.py), contraction included: the plan must not depend on it
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=fast", "-fPIC", "-shared",
                           "-I", CSRC, str(src), "-o", str(so)])
    lib = C.CDLL(str(so))
    lib.expo_plan.argtypes = [C.c_void_p] * 3 + [C.c_int] * 2 + [C.c_void_p] * 4
    lib.expo_average.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    return lib


def _host_plan(lib, t, nu, e, k):
    n_max = t.size * k
    ts, nus, pos = np.empty(n_max), np.empty(n_max), np.empty(n_max, dtype=np.int32)
    s0 = np.empty(t.size + 1, dtype=np.int32)
    n_s = lib.expo_plan(t.ctypes.data, nu.ctypes.data, e.ctypes.data, t.size, k, ts.ctypes.data, nus.ctypes.data,
                        s0.ctypes.data, pos.ctypes.data)
    return ts[:n_s], nus[:n_s], s0, pos[:n_s]


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_header_plan_and_average_equal_numpy(expo_host, seed):
    rng = np.random.default_rng(seed)
    n, k = 40, [10, 2, 7][seed]
    t = 10 ** rng.uniform(2, 6, n)
    t[5], t[6] = 100.0, 150.0  # point 5's samples at 100 + j 10 include point 6's time
    nu = rng.choice([1e9, 4.84e14, 1e18], n)
    e = t * rng.uniform(0.01, 0.6, n) * (rng.uniform(size=n) > 0.3)  # about a third without an exposure
    e[5] = 10.0 * (k - 1)
    ts, nus, s0, pos = _host_plan(expo_host, t, nu, e, k)
    want_t, want_nu, of, count = _expand(t, nu, e, k)
    assert np.array_equal(ts, want_t) and np.array_equal(nus, want_nu)
    assert np.array_equal(np.diff(s0), count)
    f = 10 ** rng.uniform(-30, -25, (abi.NCOMP, ts.size))
    out = np.empty((abi.NCOMP, n))
    expo_host.expo_average(np.ascontiguousarray(f).ctypes.data, ts.size, s0.ctypes.data, pos.ctypes.data, n, abi.NCOMP,
                           out.ctypes.data)
    assert np.array_equal(out, _average(f, of, count))
    if seed == 0:  # all exposures: the composition the engine used to restate, sample for sample
        e_all = np.maximum(e, 1.0)
        kk = np.arange(k, dtype=np.float64)
        ts_np = np.sort((t[:, None] + kk[None, :] * (e_all / (k - 1))[:, None]).reshape(-1), kind="stable")
        assert np.array_equal(_host_plan(expo_host, t, nu, e_all, k)[0], ts_np)


def test_batched_likelihood_checks_exposures():
    t, nu, flux, err, _ = _raw_points(1)
    args = (object(), configs.make(), _NAMES, _LOG, t, nu, flux, err)
    with pytest.raises(ValueError, match="expo_time has 3 values"):
        fitting.BatchedLikelihood(*args, expo_time=np.ones(3))
    with pytest.raises(ValueError, match="finite and >= 0"):
        fitting.BatchedLikelihood(*args, expo_time=-np.ones(t.size))
    with pytest.raises(ValueError, match="expo_points"):
        fitting.BatchedLikelihood(*args, expo_time=np.ones(t.size), expo_points=1)
    lk = fitting.BatchedLikelihood(*args, expo_time=np.arange(t.size, dtype=np.float64), expo_points=4, distributed=True)
    order = fitting.time_order(t)
    assert np.array_equal(lk.expo_time, np.arange(t.size, dtype=np.float64)[order])  # sorted with the data
    assert lk._cost_times.max() == np.max(lk.t + 3 * (lk.expo_time / 3))  # the window spans the last samples
    with pytest.raises(NotImplementedError, match="expo_time"):
        fitting.DeviceLikelihood(*args, device="cpu", expo_time=np.ones(t.size))


class _RecordingEngine:
    device = 0

    def __init__(self):
        self.calls = []

    def chi2_multi(self, P, datasets, dataset_of, extinction=None):
        self.calls.append(("chi2_multi", dict(extinction=extinction)))
        return np.zeros(P.size)

    def chi2_multi_bands(self, P, datasets, bands, dataset_of, **kw):
        self.calls.append(("chi2_multi_bands", dict(kw, datasets=datasets, bands=bands, dataset_of=np.array(dataset_of))))
        return np.zeros(P.size)


def test_stacks_pass_each_fits_exposures():
    eng = _RecordingEngine()
    t1, nu1, f1, e1, _ = _raw_points(1)
    t2, nu2, f2, e2, _ = _raw_points(2, 6, (1e9, 1e17))
    x1 = np.linspace(0, 50, t1.size)
    plain = fitting.BatchedLikelihood(eng, configs.make(), _NAMES, _LOG, t2, nu2, f2, e2)
    with_e = fitting.BatchedLikelihood(eng, configs.make(), _NAMES, _LOG, t1, nu1, f1, e1, expo_time=x1, expo_points=6)
    bands_only = fitting.BatchedLikelihood(eng, configs.make(), _NAMES, _LOG, [], [], [], [],
                                           bands=[dict(t=[1e3, 1e4], flux=[1.0, 1.0], err=[0.1, 0.1], nu_min=1e9,
                                                       nu_max=1e10)])
    samples = [_samples(5, 1), _samples(6, 2), _samples(4, 3)]
    # without exposures: the calls of today
    fitting.LikelihoodStack([plain, plain])(samples[:2])
    fitting.BandLikelihoodStack([plain, bands_only])(samples[:2])
    assert [c[0] for c in eng.calls] == ["chi2_multi", "chi2_multi_bands"] and "exposures" not in eng.calls[1][1]
    eng.calls.clear()
    fitting.LikelihoodStack([plain, with_e])(samples[:2])
    fitting.BandLikelihoodStack([with_e, bands_only, plain])(samples)
    for (name, call), fits in zip(eng.calls, ([plain, with_e], [with_e, bands_only, plain])):
        assert name == "chi2_multi_bands"
        expo = call["exposures"]
        assert len(expo) == len(fits)
        for ex, lk in zip(expo, fits):
            if lk is with_e:
                assert np.array_equal(ex[0], x1[fitting.time_order(t1)]) and ex[1] == 6
            else:
                assert ex is None
        assert all(b == [] for b, lk in zip(call["bands"], fits) if lk is not bands_only)
