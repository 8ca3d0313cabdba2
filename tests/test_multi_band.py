"""Band-integrated data in a batch of several light curves (vag_flux_band_multi, vag_chi2_multi_bands,
Engine.flux_band_multi / chi2_multi_bands, fitting.BandLikelihoodStack).

GPU tier, bit for bit unless stated: the ragged band flux against vag_flux_band of each band alone (2, 3, 4, 5 and 9
nodes, a one-epoch band, disjoint early and late windows, an unused band, SSC models on a radio and on an X-ray band);
the chi-squared against vag_chi2 / vag_chi2_ext of each data set alone (points + bands, bands only, points only, with
A_V and a NaN A_V, Boost's 500-rejection limit lowered so that band runs fail); a batch without bands against
vag_chi2_multi; a batch over the 32768-evaluation pass boundary; launch counts; argument validation;
BandLikelihoodStack against each BatchedLikelihood alone.
CPU tier: BandLikelihoodStack with a recording engine, and the vag_multi_set layout against the header.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests.test_multi_dataset import (_LOG, _NAMES, UNSPLIT_MODELS, _light_curve, _models, _padded, _raw_points, _samples,
                                      _with_mode)
from vegasafterglow_b200 import abi, configs, fitting

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _band(t, nu_min, nu_max, num_nu, seed=0):
    """A band-integrated data set (fitting.band_obs) of a synthetic decaying light curve."""
    t = np.asarray(t, dtype=np.float64)
    rng = np.random.default_rng(seed)
    flux = 1e-12 * (t / 1e4) ** -1.2 * np.exp(0.1 * rng.standard_normal(t.size))
    return fitting.band_obs(t, flux, 0.2 * flux, nu_min, nu_max, num_nu, weights=rng.uniform(0.5, 2.0, t.size))


XRAY = (7.25e16, 2.4e18)  # 0.3-10 keV


def _bands():
    return [
        _band(np.logspace(3, 5, 10), 1e9, 5e9, 2, 0),         # 0: radio, trapezoid
        _band(np.logspace(2, 4, 8), 4e14, 7.5e14, 3, 1),      # 1: optical, Simpson, early window
        _band(np.logspace(5, 7, 6), 1e15, 1e16, 4, 2),        # 2: 3/8 rule, late window (disjoint from 1)
        _band(np.logspace(3, 6, 12), *XRAY, 5, 3),            # 3: X-ray, Boole
        _band(np.logspace(3, 6, 7), 1e10, 1e18, 9, 4),        # 4: two frequency tiles (8 + 1)
        _band([3e4], 1e17, 1e18, 5, 5),                        # 5: one epoch
        _band(np.logspace(3, 5, 5), 1e12, 1e13, 7, 6),        # 6: used by no model
    ]


RADIO, XRAY_BAND, UNUSED_BAND = 0, 3, 6


def _band_batch(seed=0):
    """(params, band_of): a shuffled mixed batch over every band but the unused one; the SSC models on radio / X-ray.
    t_resol = 2: with the nine-node band the batch stages an 8-wide frequency tile, and at t_resol = 3 (lattices of up to
    ~35 nodes) 8 staged rows would not fit the 27 KB of shared memory that 8 CTAs per SM leave -- the batch would stage 7
    rows per pass where a two-node band's own call stages 8, and round differently (vag.h)."""
    P, is_ssc = _models(seed=seed)
    P["t_resol"] = 2.0
    used = [b for b in range(len(_bands())) if b != UNUSED_BAND]
    bo = np.asarray(used, dtype=np.int32)[np.random.default_rng(seed + 7).integers(0, len(used), P.size)]
    ssc_idx = np.nonzero(is_ssc)[0]
    bo[ssc_idx[::2]] = RADIO
    bo[ssc_idx[1::2]] = XRAY_BAND
    return P, bo


# ---- GPU tier -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_flux_band_multi_equals_each_band_alone(engine):
    P, bo = _band_batch()
    bands = _bands()
    assert 2 * P.size >= UNSPLIT_MODELS
    got, st = engine.flux_band_multi(P, bands, bo, return_status=True)
    for b in np.unique(bo):
        Q, B, idx = P[bo == b], bands[b], np.nonzero(bo == b)[0]
        f, q = engine.flux_band(_padded(Q), B["t"], B["nu_min"], B["nu_max"], B["num_nu"], return_status=True)
        assert np.array_equal(st[idx], q[:idx.size]), b
        for j, m in enumerate(idx):
            assert got[m].shape == (abi.NCOMP, B["t"].size)
            assert np.array_equal(got[m], f[j], equal_nan=True), (b, m)
    ssc = abi.COMPONENTS.index("fwd_ssc")
    assert all((got[m][ssc] > 0).all() for m in np.nonzero(P["fwd"]["ssc"] == 1)[0])


def _datasets(seed):
    """Five data sets: 0 points + two bands, 1 bands only, 2 points only, 3 points only (A_V below), 4 unused."""
    pts = [_light_curve(np.logspace(3, 6, 12), np.tile([1e9, 4.84e14, 1e18], 4), seed),
           None,
           _light_curve(np.logspace(2.5, 5, 9), np.tile([5e9, 1e14, 1e17], 3), seed + 1),
           _light_curve(np.logspace(4, 6.5, 8), np.tile([4.84e14, 1e17], 4), seed + 2),
           _light_curve(np.logspace(3, 4, 4), np.full(4, 1e9), seed + 3)]
    bands = [[_band(np.logspace(3, 6, 10), *XRAY, 5, seed), _band(np.logspace(3.5, 5, 6), 4e14, 7.5e14, 3, seed + 1)],
             [_band(np.logspace(2.5, 5.5, 8), *XRAY, 5, seed + 2), _band(np.logspace(4, 6, 5), 1e9, 5e9, 2, seed + 3)],
             [], [],
             [_band(np.logspace(3, 4, 3), 1e10, 1e18, 9, seed + 4)]]
    return pts, bands


def _chi2_batch(seed):
    P, _ = _models(seed=seed)
    ds = np.random.default_rng(seed + 8).integers(0, 4, P.size).astype(np.int32)  # set 4: no model
    return P, ds


@pytest.mark.gpu
def test_chi2_multi_bands_equals_each_data_set_alone(engine):
    P, ds = _chi2_batch(10)
    pts, bands = _datasets(0)
    rng = np.random.default_rng(3)
    ext = [None if p is None else rng.uniform(0.0, 1.7, p[0].size) for p in pts]
    A_V = rng.uniform(0.0, 2.0, P.size)
    A_V[np.nonzero(ds == 0)[0][:3]] = np.nan  # +inf
    A_V[ds == 1] = np.nan  # a set without points: A_V is not read

    def ref(d, extinction):
        Q = P[ds == d]
        kw = {}
        if extinction and pts[d] is not None:
            kw["extinction"] = (ext[d], np.tile(A_V[ds == d], -(-UNSPLIT_MODELS // Q.size)))
        c, q = engine.chi2(_padded(Q), pts[d], bands[d], return_status=True, **kw)
        return c[:Q.size], q[:Q.size]

    def run(extinction):
        got = engine.chi2_multi_bands(P, pts, bands, ds, extinction=(ext, A_V) if extinction else None, return_status=True)
        return got, {d: ref(d, extinction) for d in range(4)}

    for limits in ((0, 0), (0, 1)):  # then Boost's 500-rejection limit lowered to 1: VAG_ST_ODE_FAIL500 in band runs too
        for extinction in (False, True):
            try:
                engine.debug_set_ode_limits(*limits)
                (got, st), want = _with_mode(engine, 1, lambda: run(extinction))
            finally:
                engine.debug_set_ode_limits(0, 0)
            for d, (c, q) in want.items():
                assert np.array_equal(got[ds == d], c) and np.array_equal(st[ds == d], q), (limits, extinction, d)
            fail = (st & abi.ST_ODE_FAIL500) != 0
            assert np.isposinf(got[fail]).all()
            nan_av = np.isnan(A_V) & (ds != 1) & extinction
            assert np.isposinf(got[nan_av]).all()
            if limits[1]:
                assert fail[ds == 1].any()  # a bands-only set: the failure comes from a band run
            else:
                assert np.isfinite(got[~nan_av]).all()


@pytest.mark.gpu
def test_without_bands_equals_chi2_multi(engine):
    P, ds = _chi2_batch(20)
    pts, _ = _datasets(1)
    pts[1] = pts[4]  # every set has points
    got = engine.chi2_multi_bands(P, pts, [[] for _ in pts], ds, return_status=True)
    want = engine.chi2_multi(P, pts, ds, return_status=True)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.gpu
def test_pass_boundary(engine):
    n = (32768 + 64) // 3  # three bands per model: 32832 evaluations, the second pass 64 of them
    P = configs.random_draw(n, seed=21)
    P["t_resol"] = 3.0
    bands = [_band(np.logspace(3, 6, 6), *XRAY, 5, 7), _band(np.logspace(3, 5, 4), 4e14, 7.5e14, 3, 8),
             _band(np.logspace(4, 6, 5), 1e9, 5e9, 2, 9)]
    got, st = engine.chi2_multi_bands(P, [None], [bands], np.zeros(n, dtype=np.int32), return_status=True)
    want, q = engine.chi2(P, None, bands, return_status=True)
    assert np.array_equal(st, q)
    first = 3 * np.arange(n) + 2 < 32768  # every evaluation of the model in the first pass
    assert not first.all() and first.sum() > 10000
    assert np.array_equal(got[first], want[first])
    # the second pass is a batch of 64 evaluations, whose rows k_eats splits into partial sums: to rounding
    np.testing.assert_allclose(got[~first], want[~first], rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_sets_or_bands(engine):
    P = configs.random_draw(64, seed=41, rvs=True)
    pts, bands = _datasets(2)
    pts, bands = pts + [pts[0], pts[2]], bands + [bands[1], bands[0]]  # seven sets, 0 to 2 bands each

    def count(n_sets):
        ds = (np.arange(P.size) % n_sets).astype(np.int32)
        sub_pts, sub_bands = pts[:n_sets], bands[:n_sets]
        engine.chi2_multi_bands(P, sub_pts, sub_bands, ds)
        total = engine.last_launch_count()
        # the documented formula: the point pass (vag_chi2_multi on the models with points) + the band pass
        # (vag_flux_band_multi on every evaluation) + the gather and the band chi-squared
        with_pts = np.array([sub_pts[d] is not None for d in ds])
        keep = [d for d in range(n_sets) if sub_pts[d] is not None]
        remap = {d: i for i, d in enumerate(keep)}
        engine.chi2_multi(P[with_pts], [sub_pts[d] for d in keep], np.array([remap[d] for d in ds[with_pts]]))
        l_pts = engine.last_launch_count()
        flat = [b for bl in sub_bands for b in bl]
        first = np.cumsum([0] + [len(bl) for bl in sub_bands])
        band_of = np.array([first[d] + j for d in ds for j in range(len(sub_bands[d]))], dtype=np.int32)
        engine.flux_band_multi(np.repeat(P, [len(sub_bands[d]) for d in ds]), flat, band_of)
        l_bands = engine.last_launch_count()
        assert total == l_pts + l_bands + 2
        return total

    assert count(2) == count(7)


def _raw(engine, P, ds, sets, t, n_points=None, bands=None, ext=None, A_V=None, null_points=False):
    """vag_chi2_multi_bands on the given arrays with sentinel outputs -> (return code, outputs untouched)"""
    P = np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE)
    ds = np.ascontiguousarray(ds, dtype=np.int32)
    arr = (abi.MultiSet * max(len(sets), 1))(*[abi.MultiSet(*s) for s in sets])
    n = t.size if n_points is None else n_points
    nu, lnF, sig, w = np.full(t.size, 1e9), np.zeros(t.size), np.ones(t.size), np.ones(t.size)
    bands = bands or []
    keep = [[np.asarray(b["t"], dtype=np.float64), np.zeros(len(b["t"])), np.ones(len(b["t"])), np.ones(len(b["t"]))]
            for b in bands]
    barr = (abi.BandObs * max(len(bands), 1))(*[abi.BandObs(*[a.ctypes.data for a in k], k[0].size, b["nu_min"], b["nu_max"],
                                                            b["num_nu"]) for k, b in zip(keep, bands)])
    chi2 = np.full(P.size, 7.0)
    st = np.full(P.size, 99, dtype=np.int32)
    ptrs = [None] * 5 if null_points else [a.ctypes.data for a in (t, nu, lnF, sig, w)]
    rc = engine._lib.vag_chi2_multi_bands(engine._h, P.ctypes.data, P.size, ds.ctypes.data,
                                          C.cast(arr, C.c_void_p) if sets else None, len(sets), *ptrs,
                                          None if ext is None else ext.ctypes.data, n, None if A_V is None else A_V.ctypes.data,
                                          C.cast(barr, C.c_void_p) if bands else None, len(bands), chi2.ctypes.data,
                                          st.ctypes.data)
    return rc, bool((chi2 == 7.0).all() and (st == 99).all())


@pytest.mark.gpu
def test_arguments_are_validated_before_any_work(engine):
    P = configs.random_draw(4, seed=1)
    t = np.array([1e3, 1e4, 1e5, 2e3, 2e4, 2e5])
    xb = dict(t=[1e3, 1e4], nu_min=XRAY[0], nu_max=XRAY[1], num_nu=5)
    ok_bands = [xb, dict(xb, num_nu=3)]
    ok_sets = [(0, 3, 0, 1), (3, 3, 0, 0), (0, 0, 1, 1)]
    ds = np.array([0, 1, 2, 0])
    assert _raw(engine, P, ds, ok_sets, t, bands=ok_bands)[0] == abi.VAG_OK
    bad_P = P.copy()
    bad_P["Gamma0"][2] = 1.0
    ext = np.zeros(t.size)
    bad_ext = ext.copy()
    bad_ext[1] = np.inf
    # word in the message -> arguments
    cases = {
        "no data": dict(sets=[(0, 3, 0, 1), (3, 3, 0, 0), (0, 0, 1, 0)]),
        "points [": dict(sets=[(0, 3, 0, 1), (4, 3, 0, 0), (0, 0, 1, 1)]),
        "bands [": dict(sets=[(0, 3, 0, 1), (3, 3, 0, 0), (0, 0, 1, 2)]),
        "ascending": dict(sets=[(0, 4, 0, 1), (4, 2, 0, 0), (0, 0, 1, 1)]),
        "empty (n = 0)": dict(bands=[xb, dict(xb, t=[])]),
        "band 1: time array must be in ascending order": dict(bands=[xb, dict(xb, t=[1e4, 1e3])]),
        "finite": dict(bands=[xb, dict(xb, t=[1e3, np.inf])]),
        "num_nu": dict(bands=[xb, dict(xb, num_nu=1)]),
        "nu_max": dict(bands=[xb, dict(xb, nu_max=1e16)]),
        "model 2: dataset_of": dict(ds=np.array([0, 1, 3, 0])),
        "model 2: Gamma0": dict(P=bad_P),
        "both": dict(ext=ext),
        "ext_k": dict(ext=bad_ext, A_V=np.zeros(P.size)),
        "extinction needs point data": dict(sets=[(0, 0, 0, 1)], ds=np.zeros(4), n_points=0, ext=ext, A_V=np.zeros(4)),
        "point data arrays": dict(null_points=True),
        "no data sets": dict(sets=[]),
    }
    for word, kw in cases.items():
        args = dict(P=P, ds=ds, sets=ok_sets, t=t, bands=ok_bands)
        args.update(kw)
        rc, untouched = _raw(engine, args.pop("P"), args.pop("ds"), args.pop("sets"), args.pop("t"), **args)
        assert rc == abi.VAG_ERR_INVALID, word
        assert untouched, word
        msg = engine._lib.vag_last_error().decode()
        assert word in msg, (word, msg)
    _raw(engine, P, ds, [(0, 3, 0, 1), (3, 3, 0, 0), (0, 0, 1, 0)], t, bands=ok_bands)
    assert "data set 2" in engine._lib.vag_last_error().decode()
    # flux_band_multi: the band and the model are named
    with pytest.raises(ValueError, match="model 1: band_of"):
        engine.flux_band_multi(P, [xb], [0, 1, 0, 0])
    with pytest.raises(ValueError, match="band 1: empty"):
        engine.flux_band_multi(P, [xb, dict(xb, t=[])], [0, 0, 0, 0])
    # a failed call leaves the engine usable
    assert _raw(engine, P, ds, ok_sets, t, bands=ok_bands)[0] == abi.VAG_OK
    assert len(engine.flux_band_multi(P, [xb], [0, 0, 0, 0])) == 4


# ---- BandLikelihoodStack ----------------------------------------------------------------------------------------------
def _band_fits(engine, n_walkers, gpu=True):
    """Three fits: tophat FS with points, an X-ray band and A_V; a Gaussian FS+RS fit with two bands only that names A_V
    (ignored without points); tophat FS with points and a radio band, no A_V."""
    def raw_band(t, nu_min, nu_max, num, seed):
        b = _band(t, nu_min, nu_max, num, seed)
        return dict(t=b["t"], flux=np.exp(b["lnF_obs"]), err=np.exp(b["lnF_obs"]) * b["sigma_ln"], nu_min=nu_min,
                    nu_max=nu_max, num_points=num)

    specs = [(configs.make(lumi_dist=1e28, z=0.3), True, _raw_points(1), [raw_band(np.logspace(3, 5.5, 8), *XRAY, 5, 1)]),
             (configs.make(jet="gaussian", rvs=(0.1, 0.01, 2.3), lumi_dist=1e28, z=0.3, theta_obs=0.05), True, None,
              [raw_band(np.logspace(3.5, 6, 6), *XRAY, 5, 2), raw_band(np.logspace(3, 5, 5), 4e14, 7.5e14, 3, 3)]),
             (configs.make(lumi_dist=3e27, z=0.1), False, _raw_points(3, 12, (1e9, 5e9, 4.84e14, 1e17)),
              [raw_band(np.logspace(4, 6, 4), 1e9, 5e9, 2, 4)])]
    fits, samples = [], []
    for k, (tmpl, av, pts, bands) in enumerate(specs):
        if gpu:
            tmpl["t_resol"] = 3.0
        s = _samples(n_walkers, 60 + k, av)
        lo, hi = np.min(s, axis=0), np.max(s, axis=0)
        hi[1] = np.quantile(s[:, 1], 0.9)
        names, log = _NAMES + (["A_V"] if av else []), _LOG + ([False] if av else [])
        t, nu, flux, err, ext = pts if pts is not None else (np.zeros(0),) * 5
        fits.append(fitting.BatchedLikelihood(engine, tmpl, names, log, t, nu, flux, err, lower=lo, upper=hi,
                                              log_prior=lambda x, k=k: -0.5 * k * x[:, 2], bands=bands,
                                              ext_kernel=ext if av else None))
        samples.append(s)
    return fits, samples


@pytest.mark.gpu
def test_band_likelihood_stack_equals_each_likelihood_alone(engine):
    fits, samples = _band_fits(engine, 2 * UNSPLIT_MODELS)
    try:
        engine.set_series_mode(1)
        want = [lk(s) for lk, s in zip(fits, samples)]
        got = fitting.BandLikelihoodStack(fits)(samples)
    finally:
        engine.set_series_mode(0)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
        assert np.isneginf(w).sum() > 100 and np.isfinite(w).sum() >= UNSPLIT_MODELS


# ---- CPU tier: BandLikelihoodStack with a recording engine ----------------------------------------------------------
def _stand_in(P, lnF, ext, A_V, bands):
    """Not a likelihood: a value that depends on the model, on its points, its bands (in order) and A_V."""
    v = np.log10(P["E_iso"]) + P["Gamma0"] + P["theta_c"] + lnF.sum() + A_V * (1.0 + ext.sum())
    for i, b in enumerate(bands):
        v = v + (i + 1) * b["lnF_obs"].sum() + b["num_nu"]
    return v


class _RecordingEngine:
    device = 0

    def __init__(self):
        self.calls = []

    def chi2_series(self, P, t, nu, lnF, sig, w):
        return _stand_in(P, lnF, np.zeros(1), np.zeros(P.size), ())

    def chi2(self, P, pts, bands, extinction=None):
        ext, A_V = extinction if extinction is not None else (np.zeros(1), np.zeros(P.size))
        return _stand_in(P, np.zeros(1) if pts is None else pts[2], ext, A_V, bands)

    def chi2_multi_bands(self, P, datasets, bands, dataset_of, extinction=None):
        self.calls.append(dict(n=P.size, datasets=datasets, bands=bands, dataset_of=np.array(dataset_of),
                               extinction=extinction))
        out = np.empty(P.size)
        for m in range(P.size):
            d = dataset_of[m]
            lnF = np.zeros(1) if datasets[d] is None else datasets[d][2]
            ext, av = (np.zeros(1), 0.0)
            if extinction is not None and datasets[d] is not None:
                ext, av = extinction[0][d], extinction[1][m]
            out[m] = _stand_in(P[m:m + 1], lnF, ext, np.array([av]), bands[d])[0]
        return out


def test_band_likelihood_stack_is_one_call_split_back_per_fit():
    eng = _RecordingEngine()
    fits, samples = _band_fits(eng, 40, gpu=False)
    got = fitting.BandLikelihoodStack(fits)(samples)
    want = [lk(s) for lk, s in zip(fits, samples)]
    assert len(eng.calls) == 1
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
        assert np.isneginf(w).any() and np.isfinite(w).any()
    call = eng.calls[0]
    counts = [int(np.isfinite(lk.chi2(s[lk._in_bounds(s)])).sum()) for lk, s in zip(fits, samples)]
    assert np.array_equal(call["dataset_of"], np.repeat(np.arange(3), counts)) and call["n"] == sum(counts)
    assert call["datasets"][1] is None  # the bands-only fit
    for k, lk in enumerate(fits):
        if lk.t.size:
            assert all(np.array_equal(a, b) for a, b in zip(call["datasets"][k], (lk.t, lk.nu, lk.lnF, lk.sig, lk.w)))
        assert len(call["bands"][k]) == len(lk.bands)
        assert all(a is b for a, b in zip(call["bands"][k], lk.bands))  # the fit's bands, in its order
    ext, A_V = call["extinction"]
    assert np.array_equal(ext[0], fits[0].ext_kernel) and ext[1] is None and not ext[2].any()
    assert A_V[call["dataset_of"] == 0].all() and not A_V[call["dataset_of"] != 0].any()


def test_band_likelihood_stack_rejects_what_it_cannot_stack():
    eng = _RecordingEngine()
    t, nu, flux, err, _ = _raw_points(1)
    args = (configs.make(), _NAMES, _LOG, t, nu, flux, err)
    plain = fitting.BatchedLikelihood(eng, *args)
    with pytest.raises(NotImplementedError, match="distributed"):
        fitting.BandLikelihoodStack([fitting.BatchedLikelihood(eng, *args, distributed=True), plain])
    with pytest.raises(NotImplementedError, match="DeviceLikelihood"):
        fitting.BandLikelihoodStack([plain, fitting.DeviceLikelihood(eng, *args, device="cpu")])


def test_multi_set_layout_matches_header(tmp_path):
    src = tmp_path / "sets.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu %%zu %%zu\\n", '
                   'offsetof(vag_multi_set, offset), offsetof(vag_multi_set, n), offsetof(vag_multi_set, band0), '
                   'offsetof(vag_multi_set, n_bands), sizeof(vag_multi_set)); return 0;}'
                   % os.path.join(ROOT, "include", "vag.h"))
    exe = tmp_path / "sets"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = tuple(int(v) for v in subprocess.check_output([str(exe)]).split())
    M = abi.MultiSet
    assert got == (M.offset.offset, M.n.offset, M.band0.offset, M.n_bands.offset, C.sizeof(M))
