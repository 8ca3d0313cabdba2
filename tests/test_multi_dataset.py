"""Several light curves in one batch: every model has its own data set (vag_flux_density_series_multi, vag_chi2_multi,
Engine.flux_density_series_multi / chi2_multi, fitting.LikelihoodStack).

GPU tier: on a shuffled mixed batch over seven data sets (one point; ten distinct frequencies; early and late windows
that do not overlap; a set no model uses; a config-5-like set; a radio-only set), the ragged call equals the
single-request call of each data set's models on that data set, status included; the same for chi2 with and without a
fitted A_V; a batch across the 32768-model pass boundary; the SSC band of each model; launch counts; argument
validation; LikelihoodStack against each BatchedLikelihood alone.
CPU tier: LikelihoodStack with a recording engine, and the vag_series_set layout against the header.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from vegasafterglow_b200 import abi, configs, fitting

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# k_eats cuts the rows of a model into partial sums below 2368 (model x shock) CTAs on 148 SMs, and how many depends on
# the batch size (vag_b200.cu run_flux_pass): a ragged batch and the single-data-set batch of a part of its models would
# round differently.  Reference calls are therefore padded to this many models (by repeating them), where neither splits.
UNSPLIT_MODELS = 2368


# ---- data ------------------------------------------------------------------------------------------------------------
def _light_curve(t, nu, seed):
    """(t, nu, lnF_obs, sigma_ln, w) of a synthetic power-law light curve, sorted by time."""
    rng = np.random.default_rng(seed)
    t, nu = np.asarray(t, dtype=np.float64), np.asarray(nu, dtype=np.float64)
    flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
    return fitting.consolidate_data(t, nu, flux, 0.2 * flux, rng.uniform(0.5, 2.0, t.size))


def _grid_set(t_lo, t_hi, n_epochs, bands, seed):
    t = np.repeat(np.logspace(np.log10(t_lo), np.log10(t_hi), n_epochs), len(bands))
    return _light_curve(t, np.tile(bands, n_epochs), seed)


WIDE = 1  # the data set with more than 8 distinct frequencies
UNUSED = 4
RADIO = 6  # narrower band than the batch's union: SSC tables sized per data set


def _datasets():
    return [
        _light_curve([3e4], [4.84e14], 0),                                       # 0: one point
        _light_curve(np.logspace(3, 6, 20), np.tile(np.logspace(9, 18, 10), 2), 1),  # 1: ten distinct frequencies
        _grid_set(1e2, 1e4, 10, [1e9, 4.84e14, 1e18], 2),                         # 2: early window
        _grid_set(1e5, 1e7, 8, [5e9, 1e14, 4.84e14, 1e17], 3),                    # 3: late window, disjoint from 2
        _grid_set(1e3, 1e5, 6, [1e9, 5e9, 4.84e14, 1e17, 1e18], 4),               # 4: used by no model
        _grid_set(10 ** 2.5, 10 ** 6.5, 20, [1e9, 5e9, 4.84e14, 1e17, 1e18], 5),  # 5: config-5-like
        _grid_set(1e3, 1e6, 10, [1e9, 5e9], 6),                                   # 6: radio only
    ]


def _models(n_per_kind=400, seed=0):
    """Tophat FS, FS+RS, Gaussian off-axis and spreading models and a few SSC+KN ones, shuffled; short time lattices
    (t_resol = 3) keep every call at the full 8 staged rows per pass, so that the ragged call and the single-data-set
    calls stage the same rows (vag.h)."""
    sp = configs.random_draw(n_per_kind, seed=seed + 4)
    sp["spreading"] = 1
    ssc = configs.random_draw(16, seed=seed + 5, ssc=True, kn=True)
    P = np.concatenate([configs.random_draw(n_per_kind, seed=seed + 1), configs.random_draw(n_per_kind, seed=seed + 2, rvs=True),
                        configs.random_draw(n_per_kind, seed=seed + 3, jet="gaussian", theta_obs_max=0.4), sp, ssc])
    P["t_resol"] = 3.0
    is_ssc = np.zeros(P.size, dtype=bool)
    is_ssc[-ssc.size:] = True
    perm = np.random.default_rng(seed + 6).permutation(P.size)
    return P[perm], is_ssc[perm]


def _batch(with_wide=True, seed=0):
    """(params, data sets, dataset_of): every set but UNUSED has models; half of the SSC models use the radio-only set."""
    P, is_ssc = _models(seed=seed)
    sets = _datasets()
    used = [d for d in range(len(sets)) if d != UNUSED and (with_wide or d != WIDE)]
    ds = np.asarray(used, dtype=np.int32)[np.random.default_rng(seed + 7).integers(0, len(used), P.size)]
    ssc_idx = np.nonzero(is_ssc)[0]
    ds[ssc_idx[::2]] = RADIO
    ds[ssc_idx[1::2]] = 5
    if not with_wide:  # a batch without the wide set: banded in series mode 2
        sets[WIDE] = sets[0]
    return P, sets, ds


def _padded(P):
    return np.tile(P, -(-UNSPLIT_MODELS // P.size))


def _per_set(engine, P, sets, ds, call):
    """{d: result of call(models of set d, padded, set d)} restricted to those models"""
    out = {}
    for d in np.unique(ds):
        Q = P[ds == d]
        out[int(d)] = call(_padded(Q), sets[d], Q.size)
    return out


# ---- GPU tier -----------------------------------------------------------------------------------------------------------
# case -> (series mode of the ragged call, with the wide set, series mode of the reference calls).  With the ten-frequency
# set in the batch, mode 2 runs every model per point (vag.h), so its references are per point too.
CASES = {"per_point": (1, True, 1), "banded": (2, False, 2), "wide_set_runs_per_point": (2, True, 1)}


def _with_mode(engine, mode, fn):
    try:
        engine.set_series_mode(mode)
        return fn()
    finally:
        engine.set_series_mode(0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_flux_equals_each_data_set_alone(engine, case):
    mode, with_wide, ref_mode = CASES[case]
    P, sets, ds = _batch(with_wide)
    assert 2 * P.size >= UNSPLIT_MODELS  # FS+RS models in the batch: 2 shocks per model
    got, st = _with_mode(engine, mode, lambda: engine.flux_density_series_multi(P, [s[:2] for s in sets], ds,
                                                                                 return_status=True))

    def ref(Q, s, n):
        f, q = engine.flux_density_series(Q, s[0], s[1], return_status=True)
        return f[:n], q[:n]

    want = _with_mode(engine, ref_mode, lambda: _per_set(engine, P, sets, ds, ref))
    for d, (f, q) in want.items():
        idx = np.nonzero(ds == d)[0]
        assert np.array_equal(st[idx], q), d
        for j, m in enumerate(idx):
            assert got[m].shape == (abi.NCOMP, sets[d][0].size)
            assert np.array_equal(got[m], f[j], equal_nan=True), (d, m)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_chi2_equals_each_data_set_alone(engine, case):
    mode, with_wide, ref_mode = CASES[case]
    P, sets, ds = _batch(with_wide, seed=10)
    got, st = _with_mode(engine, mode, lambda: engine.chi2_multi(P, sets, ds, return_status=True))

    def ref(Q, s, n):
        c, q = engine.chi2_series(Q, *s, return_status=True)
        return c[:n], q[:n]

    want = _with_mode(engine, ref_mode, lambda: _per_set(engine, P, sets, ds, ref))
    for d, (c, q) in want.items():
        assert np.array_equal(got[ds == d], c) and np.array_equal(st[ds == d], q), d
    assert np.isfinite(got).all()


@pytest.mark.gpu
def test_chi2_with_extinction_equals_chi2_ext(engine):
    P, sets, ds = _batch(seed=20)
    rng = np.random.default_rng(3)
    ext = [rng.uniform(0.0, 1.7, s[0].size) for s in sets]
    A_V = rng.uniform(0.0, 2.0, P.size)
    A_V[np.nonzero(ds == 5)[0][:3]] = np.nan

    def run():
        got = engine.chi2_multi(P, sets, ds, extinction=(ext, A_V), return_status=True)

        def ref(Q, s, n, d):
            sub = A_V[ds == d]
            c, q = engine.chi2(Q, s, (), return_status=True, extinction=(ext[d], np.tile(sub, -(-UNSPLIT_MODELS // sub.size))))
            return c[:n], q[:n]

        want = {int(d): ref(_padded(P[ds == d]), sets[d], int((ds == d).sum()), int(d)) for d in np.unique(ds)}
        return got, want

    for limits in ((0, 0), (0, 1)):  # then Boost's 500-rejection limit lowered to 1: VAG_ST_ODE_FAIL500
        try:
            engine.debug_set_ode_limits(*limits)
            (got, st), want = _with_mode(engine, 1, run)
        finally:
            engine.debug_set_ode_limits(0, 0)
        for d, (c, q) in want.items():
            assert np.array_equal(got[ds == d], c) and np.array_equal(st[ds == d], q), d
        assert np.isposinf(got[np.isnan(A_V)]).all()
        fail = (st & abi.ST_ODE_FAIL500) != 0
        assert np.isposinf(got[fail]).all()
        if limits[1]:
            assert fail.any()


@pytest.mark.gpu
def test_pass_boundary(engine):
    n = 32768 + 64
    P = configs.random_draw(n, seed=21)
    sets = [_grid_set(1e3, 1e6, 4, [1e9, 1e17], 8), _grid_set(1e4, 1e7, 3, [4.84e14], 9)]
    ds = ((np.arange(n) // 16) % 2).astype(np.int32)
    assert ds[32767] != ds[32768]
    A_V = np.random.default_rng(4).uniform(0, 2, n)
    ext = [np.linspace(0.0, 1.2, s[0].size) for s in sets]

    def run():
        got = engine.chi2_multi(P, sets, ds, extinction=(ext, A_V), return_status=True)
        flux = engine.flux_density_series_multi(P, [s[:2] for s in sets], ds)
        want = {d: engine.chi2(P[ds == d], sets[d], (), return_status=True, extinction=(ext[d], A_V[ds == d])) for d in (0, 1)}
        want_f = {d: engine.flux_density_series(P[ds == d], *sets[d][:2]) for d in (0, 1)}
        return got, flux, want, want_f

    (got, st), flux, want, want_f = _with_mode(engine, 1, run)
    for d in (0, 1):
        idx = np.nonzero(ds == d)[0]
        assert np.array_equal(got[idx], want[d][0]) and np.array_equal(st[idx], want[d][1])
        f = np.stack([flux[m] for m in idx])
        first = idx < 32768
        assert np.array_equal(f[first], want_f[d][first])
        # the second pass is a batch of 64 models, whose rows k_eats splits into partial sums (UNSPLIT_MODELS): to rounding
        np.testing.assert_allclose(f[~first], want_f[d][~first], rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_ssc_tables_span_each_models_own_band(engine):
    # SSC models on a radio-only set in a batch whose other set reaches 1e18 Hz.  Batches this small split their rows,
    # and the split count depends on the batch size: the comparison is to 1e-12 relative, not bit for bit.
    P = configs.random_draw(6, seed=31, ssc=True, kn=True)
    sets = _datasets()
    radio, wide = sets[RADIO], sets[5]
    ds = np.array([0, 1, 0, 1, 0, 1], dtype=np.int32)
    got = engine.flux_density_series_multi(P, [radio[:2], wide[:2]], ds)
    own = engine.flux_density_series(P[ds == 0], *radio[:2])
    # the same models with the radio points evaluated inside a request that spans the union band
    t_u, nu_u = np.concatenate([radio[0], wide[0]]), np.concatenate([radio[1], wide[1]])
    order = np.argsort(t_u, kind="stable")
    union = engine.flux_density_series(P[ds == 0], t_u[order], nu_u[order])[:, :, np.argsort(order)[:radio[0].size]]
    ssc = abi.COMPONENTS.index("fwd_ssc")
    mine = np.stack([got[m] for m in np.nonzero(ds == 0)[0]])
    assert (own[:, ssc] > 0).all()
    np.testing.assert_allclose(mine, own, rtol=1e-12, atol=0)
    assert not np.allclose(union[:, ssc], own[:, ssc], rtol=1e-12, atol=0), "the union band builds the same tables"


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_the_number_of_sets(engine):
    P = configs.random_draw(64, seed=41, rvs=True)
    sets = _datasets()
    engine.chi2_series(P, *sets[5])
    single = engine.last_launch_count()
    engine.chi2_multi(P, [sets[5]], np.zeros(P.size, dtype=np.int32))
    one = engine.last_launch_count()
    engine.chi2_multi(P, sets, (np.arange(P.size) % 7).astype(np.int32))
    seven = engine.last_launch_count()
    assert one == seven == single


def _raw_chi2_multi(engine, P, ds, sets, t, nu, ext=None, A_V=None, n_points=None):
    """vag_chi2_multi on the given arrays with sentinel outputs -> (return code, outputs untouched)"""
    P = np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE)
    ds = np.ascontiguousarray(ds, dtype=np.int32)
    arr = (abi.SeriesSet * max(len(sets), 1))(*[abi.SeriesSet(o, n) for o, n in sets])
    n = t.size if n_points is None else n_points
    lnF, sig, w = np.zeros(t.size), np.ones(t.size), np.ones(t.size)
    chi2 = np.full(P.size, 7.0)
    st = np.full(P.size, 99, dtype=np.int32)
    rc = engine._lib.vag_chi2_multi(engine._h, P.ctypes.data, P.size, ds.ctypes.data, C.cast(arr, C.c_void_p) if sets else None,
                                    len(sets), t.ctypes.data, nu.ctypes.data, lnF.ctypes.data, sig.ctypes.data, w.ctypes.data,
                                    None if ext is None else ext.ctypes.data, n,
                                    None if A_V is None else A_V.ctypes.data, chi2.ctypes.data, st.ctypes.data)
    return rc, bool((chi2 == 7.0).all() and (st == 99).all())


@pytest.mark.gpu
def test_arguments_are_validated_before_any_work(engine):
    P = configs.random_draw(4, seed=1)
    t = np.array([1e3, 1e4, 1e5, 2e3, 2e4, 2e5])
    nu = np.full(t.size, 1e9)
    ok_sets = [(0, 3), (3, 3)]
    ds = np.array([0, 1, 1, 0])
    assert _raw_chi2_multi(engine, P, ds, ok_sets, t, nu)[0] == abi.VAG_OK
    bad_t = t.copy()
    bad_t[5] = np.inf  # last of set 1: still ascending
    neg_t = t.copy()
    neg_t[3] = -1.0
    bad_nu = nu.copy()
    bad_nu[5] = 0.0
    bad_P = P.copy()
    bad_P["Gamma0"][2] = 1.0
    ext = np.zeros(t.size)
    bad_ext = ext.copy()
    bad_ext[1] = np.inf
    cases = {
        "dataset_of": dict(ds=np.array([0, 1, 2, 0])),
        "dataset_of ": dict(ds=np.array([0, -1, 1, 0])),
        "outside": dict(sets=[(0, 3), (4, 3)]),
        "empty": dict(sets=[(0, 3), (3, 0)]),
        "ascending": dict(sets=[(0, 4), (4, 2)]),
        "finite": dict(t=bad_t),
        "> 0": dict(t=neg_t),
        "frequencies": dict(nu=bad_nu),
        "Gamma0": dict(P=bad_P),
        "both": dict(ext=ext),
        "ext_k": dict(ext=bad_ext, A_V=np.zeros(P.size)),
        "no data sets": dict(sets=[]),
    }
    for word, kw in cases.items():
        args = dict(P=P, ds=ds, sets=ok_sets, t=t, nu=nu)
        args.update(kw)
        rc, untouched = _raw_chi2_multi(engine, args.pop("P"), args.pop("ds"), args.pop("sets"), args.pop("t"), args.pop("nu"),
                                        **args)
        assert rc == abi.VAG_ERR_INVALID, word
        assert untouched, word
        msg = engine._lib.vag_last_error().decode()
        assert word.strip() in msg, (word, msg)
    # messages name the data set / the model
    rc, _ = _raw_chi2_multi(engine, P, ds, [(0, 3), (3, 0)], t, nu)
    assert "data set 1" in engine._lib.vag_last_error().decode()
    rc, _ = _raw_chi2_multi(engine, P, np.array([0, 1, 5, 0]), ok_sets, t, nu)
    assert "model 2" in engine._lib.vag_last_error().decode()
    with pytest.raises(ValueError, match="data set 1"):
        engine.flux_density_series_multi(P, [(t[:3], nu[:3]), (t[3:][::-1], nu[3:])], ds)


# ---- LikelihoodStack --------------------------------------------------------------------------------------------------
_NAMES = ["E_iso", "Gamma0", "theta_c", "n_ism", "eps_e", "eps_B", "p"]
_LOG = [True, True, False, True, True, True, False]


def _samples(n, seed, av=False):
    rng = np.random.default_rng(seed)
    cols = [rng.uniform(51, 54, n), rng.uniform(1.7, 3, n), rng.uniform(0.03, 0.4, n), rng.uniform(-3, 1, n),
            rng.uniform(-2, 0.4, n), rng.uniform(-4, -1, n), rng.uniform(2.1, 2.8, n)]
    return np.column_stack(cols + ([rng.uniform(0, 2, n)] if av else []))


def _raw_points(seed, n_epochs=10, bands=(1e9, 4.84e14, 1e18), t_lo=1e3):
    rng = np.random.default_rng(seed)
    t = np.repeat(np.logspace(np.log10(t_lo), np.log10(t_lo) + 3, n_epochs), len(bands))
    nu = np.tile(bands, n_epochs)
    flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
    perm = rng.permutation(t.size)  # the likelihood sorts by time itself
    return t[perm], nu[perm], flux[perm], 0.2 * flux[perm], rng.uniform(0, 1.5, t.size)[perm]


def _fits(engine, n_walkers, gpu=True):
    """Three fits: tophat FS with A_V, Gaussian FS+RS without, tophat FS with A_V and a different light curve; each has
    out-of-bounds walkers and walkers the constructors reject (eps_e = 10^s > 1)."""
    specs = [(configs.make(lumi_dist=1e28, z=0.3), True, _raw_points(1)),
             (configs.make(jet="gaussian", rvs=(0.1, 0.01, 2.3), lumi_dist=1e28, z=0.3, theta_obs=0.05), False,
              _raw_points(2, 8, (5e9, 1e17), 1e4)),
             (configs.make(lumi_dist=3e27, z=0.1), True, _raw_points(3, 12, (1e9, 5e9, 4.84e14, 1e17)))]
    fits, samples = [], []
    for k, (tmpl, av, (t, nu, flux, err, ext)) in enumerate(specs):
        if gpu:
            tmpl["t_resol"] = 3.0
        s = _samples(n_walkers, 50 + k, av)
        lo, hi = np.min(s, axis=0), np.max(s, axis=0)
        hi[1] = np.quantile(s[:, 1], 0.9)
        names, log = _NAMES + (["A_V"] if av else []), _LOG + ([False] if av else [])
        fits.append(fitting.BatchedLikelihood(engine, tmpl, names, log, t, nu, flux, err, lower=lo, upper=hi,
                                              log_prior=lambda x, k=k: -0.5 * k * x[:, 2], ext_kernel=ext if av else None))
        samples.append(s)
    return fits, samples


@pytest.mark.gpu
def test_likelihood_stack_equals_each_likelihood_alone(engine):
    fits, samples = _fits(engine, 2 * UNSPLIT_MODELS)
    try:
        engine.set_series_mode(1)
        want = [lk(s) for lk, s in zip(fits, samples)]
        got = fitting.LikelihoodStack(fits)(samples)
    finally:
        engine.set_series_mode(0)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
        assert np.isneginf(w).sum() > 100 and np.isfinite(w).sum() >= UNSPLIT_MODELS


# ---- CPU tier: LikelihoodStack with a recording engine --------------------------------------------------------------
def _stand_in_chi2(P, lnF, ext, A_V):
    """Not a likelihood: a value that depends on the model, on its data set and on A_V."""
    return np.log10(P["E_iso"]) + P["Gamma0"] + P["theta_c"] + lnF.sum() + A_V * (1.0 + ext.sum())


class _RecordingEngine:
    device = 0

    def __init__(self):
        self.calls = []

    def chi2_series(self, P, t, nu, lnF, sig, w):
        return _stand_in_chi2(P, lnF, np.zeros(1), np.zeros(P.size))

    def chi2(self, P, pts, bands, extinction=None):
        ext, A_V = extinction if extinction is not None else (np.zeros(1), np.zeros(P.size))
        return _stand_in_chi2(P, pts[2], ext, A_V)

    def chi2_multi(self, P, datasets, dataset_of, extinction=None):
        self.calls.append(dict(n=P.size, datasets=datasets, dataset_of=np.array(dataset_of), extinction=extinction))
        out = np.empty(P.size)
        for m in range(P.size):
            d = dataset_of[m]
            ext, av = (extinction[0][d], extinction[1][m]) if extinction is not None else (np.zeros(1), 0.0)
            out[m] = _stand_in_chi2(P[m:m + 1], datasets[d][2], ext, np.array([av]))[0]
        return out


def test_likelihood_stack_is_one_call_split_back_per_fit():
    eng = _RecordingEngine()
    fits, samples = _fits(eng, 40, gpu=False)
    got = fitting.LikelihoodStack(fits)(samples)
    want = [lk(s) for lk, s in zip(fits, samples)]
    assert len(eng.calls) == 1
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
        assert np.isneginf(w).any() and np.isfinite(w).any()
    call = eng.calls[0]
    # dataset_of: the valid in-bounds walkers of fit 0, then of fit 1, then of fit 2
    counts = [int(np.isfinite(lk.chi2(s[lk._in_bounds(s)])).sum()) for lk, s in zip(fits, samples)]
    assert np.array_equal(call["dataset_of"], np.repeat(np.arange(3), counts)) and call["n"] == sum(counts)
    for k, lk in enumerate(fits):
        assert all(np.array_equal(a, b) for a, b in zip(call["datasets"][k], (lk.t, lk.nu, lk.lnF, lk.sig, lk.w)))
    ext, A_V = call["extinction"]
    assert np.array_equal(ext[0], fits[0].ext_kernel) and np.array_equal(ext[2], fits[2].ext_kernel)
    assert ext[1].shape == fits[1].t.shape and not ext[1].any()  # the fit without A_V: ext_k = 0
    assert not A_V[call["dataset_of"] == 1].any() and A_V[call["dataset_of"] != 1].all()


def test_likelihood_stack_without_av_passes_no_extinction():
    eng = _RecordingEngine()
    fits, samples = _fits(eng, 20, gpu=False)
    fitting.LikelihoodStack([fits[1]])([samples[1]])
    assert eng.calls[0]["extinction"] is None


def test_likelihood_stack_rejects_what_it_cannot_stack():
    eng = _RecordingEngine()
    t, nu, flux, err, _ = _raw_points(1)
    args = (configs.make(), _NAMES, _LOG, t, nu, flux, err)
    plain = fitting.BatchedLikelihood(eng, *args)
    tb = np.logspace(3.2, 5.5, 6)
    band = dict(t=tb, flux=1e-12 * tb ** 0, err=2e-13 * tb ** 0, nu_min=7.25e16, nu_max=2.4e18, num_points=5)
    with pytest.raises(NotImplementedError, match="band"):
        fitting.LikelihoodStack([plain, fitting.BatchedLikelihood(eng, *args, bands=[band])])
    with pytest.raises(NotImplementedError, match="distributed"):
        fitting.LikelihoodStack([fitting.BatchedLikelihood(eng, *args, distributed=True), plain])
    with pytest.raises(NotImplementedError, match="DeviceLikelihood"):
        fitting.LikelihoodStack([plain, fitting.DeviceLikelihood(eng, *args, device="cpu")])


def test_series_set_layout_matches_header(tmp_path):
    src = tmp_path / "sets.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu\\n", '
                   'offsetof(vag_series_set, offset), offsetof(vag_series_set, n), sizeof(vag_series_set)); return 0;}'
                   % os.path.join(ROOT, "include", "vag.h"))
    exe = tmp_path / "sets"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    off, n, size = (int(v) for v in subprocess.check_output([str(exe)]).split())
    assert (off, n, size) == (abi.SeriesSet.offset.offset, abi.SeriesSet.n.offset, C.sizeof(abi.SeriesSet))
