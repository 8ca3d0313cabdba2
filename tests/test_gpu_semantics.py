"""GPU tier: likelihood with band-integrated terms, failure semantics, limits of the batched entry points."""
import numpy as np
import pytest

from tests.helpers import load_golden
from vegasafterglow_b200 import abi, configs, fitting

pytestmark = pytest.mark.gpu


def _manual_chi2(lnF, F, sig, w):
    return np.sum(w * ((lnF - np.log(np.maximum(F, 1e-300))) / sig) ** 2, axis=-1)


def test_chi2_with_band_terms_equals_manual_formula(engine):
    # Fitter._evaluate (fitter.py:503-533): point term on flux_density + one term per band on Model.flux; the manual
    # formula is tests/python/test_fit_smoke.py:119-127
    P = configs.random_draw(12, seed=3, rvs=True)
    rng = np.random.default_rng(1)
    t = np.sort(np.tile(np.logspace(3, 6, 6), 2))
    nu = np.tile([1e9, 4.84e14], 6)
    truth = engine.flux_density_series(P[:1], t, nu)[0, 0]
    pts = fitting.consolidate_data(t, nu, truth * (1 + 0.05 * rng.standard_normal(t.size)), 0.1 * truth,
                                   rng.uniform(0.5, 2, t.size))
    bands = []
    for (lo, hi, num, tb) in ((7.25e16, 2.4e18, 5, np.logspace(3.2, 5.5, 7)), (1e9, 1e11, 9, np.array([2e4, 3e5]))):
        fb = engine.flux_band(P[:1], tb, lo, hi, num)[0, 0]
        bands.append(fitting.band_obs(tb, fb * (1 + 0.1 * rng.standard_normal(tb.size)), 0.2 * fb, lo, hi, num,
                                      weights=rng.uniform(0.5, 2, tb.size)))
    chi2, st = engine.chi2(P, pts, bands, return_status=True)
    assert (st == 0).all()
    manual = _manual_chi2(pts[2], engine.flux_density_series(P, pts[0], pts[1])[:, 0], pts[3], pts[4])
    for b in bands:
        manual = manual + _manual_chi2(b["lnF_obs"], engine.flux_band(P, b["t"], b["nu_min"], b["nu_max"], b["num_nu"])[:, 0],
                                       b["sigma_ln"], b["w"])
    np.testing.assert_allclose(chi2, manual, rtol=1e-12)
    np.testing.assert_array_equal(engine.chi2(P, pts, ()), engine.chi2_series(P, *pts))
    only_bands = engine.chi2(P, None, bands)
    np.testing.assert_allclose(only_bands, chi2 - engine.chi2_series(P, *pts), rtol=1e-9)
    # the sampler-side object routes band data the same way
    lk = fitting.BatchedLikelihood(engine, P[:1], ["E_iso"], [True], t, nu, np.exp(pts[2]), pts[3] * np.exp(pts[2]),
                                   weights=pts[4], bands=[dict(t=b["t"], flux=np.exp(b["lnF_obs"]),
                                                               err=b["sigma_ln"] * np.exp(b["lnF_obs"]), nu_min=b["nu_min"],
                                                               nu_max=b["nu_max"], num_points=b["num_nu"], weights=b["w"])
                                                          for b in bands])
    s = np.log10(P["E_iso"][:4])[:, None]
    Q = np.repeat(P[:1], 4)
    Q["E_iso"] = P["E_iso"][:4]
    np.testing.assert_allclose(lk.chi2(s), engine.chi2(Q, pts, bands), rtol=1e-12)


def test_band_flux_matches_reference_fixture(engine):
    g = np.load(__import__("os").path.join(__import__("tests.helpers", fromlist=["GOLDEN_DIR"]).GOLDEN_DIR, "method_flux_band.npz"))
    p = abi.upgrade_params(g["params"])
    for num in (2, 5, 12):
        fb = engine.flux_band(p, g["t"], float(g["nu_min"]), float(g["nu_max"]), num)
        ref = g[f"num_{num}"]
        np.testing.assert_allclose(fb[0, 0], ref[0], rtol=1e-6)
        np.testing.assert_allclose(fb[0, 1], ref[1], rtol=1e-6)
        np.testing.assert_allclose(fb[0, 3], ref[2], rtol=1e-6)


def test_ode_failure_semantics(engine):
    # reference: a row that exhausts max_ode_steps keeps the Shock-constructor defaults beyond the last saved node and a
    # warning is printed (forward-shock.tpp:196-200, reverse-shock.tpp:555-566) -- a finite, smaller flux, no exception;
    # 500 consecutive rejections throw inside Boost (max_step_checker.hpp:99-106) -> the samplers' logL = -inf.
    P = np.concatenate([configs.random_draw(6, seed=5), configs.random_draw(6, seed=6, rvs=True)])
    g = load_golden("series_rs_tophat_ism")
    t, nu = g["t"], g["nu"]
    f0, st0 = engine.flux_density_series(P, t, nu, return_status=True)
    assert (st0 == 0).all()
    obs = (np.log(f0[0, 0]), np.full(t.size, 0.1), np.ones(t.size))
    try:
        engine.debug_set_ode_limits(max_steps=20)
        f, st = engine.flux_density_series(P, t, nu, return_status=True)
        assert ((st & abi.ST_ODE_STEP_CAP) != 0).all() and (st & ~abi.ST_ODE_STEP_CAP == 0).all()
        assert np.isfinite(f).all() and (f >= 0).all()
        assert (f[:, 0, -1] == 0).all() and (f0[:, 0, -1] > 0).all()  # late epochs lie beyond the truncated solve
        chi2 = engine.chi2_series(P, t, nu, *obs)
        assert np.isfinite(chi2).all() and (chi2 > 1e6).all()          # ln(1e-300) terms: huge but finite, as in the reference
        engine.debug_set_ode_limits(max_fails=1)
        f, st = engine.flux_density_series(P, t, nu, return_status=True)
        hit = (st & abi.ST_ODE_FAIL500) != 0
        assert hit[6:].any(), "a reverse-shock solve rejects at least one step"
        chi2 = engine.chi2_series(P, t, nu, *obs)
        assert np.isinf(chi2[hit]).all() and np.isfinite(chi2[~hit]).all()
        assert np.isinf(engine.chi2(P, (t, nu, *obs), ())[hit]).all()
    finally:
        engine.debug_set_ode_limits(0, 0)
    f1, st1 = engine.flux_density_series(P, t, nu, return_status=True)
    assert (st1 == 0).all() and np.array_equal(f1, f0)  # small batches are deterministic too (k_sum_splits)


def test_capacity_overflow_gives_nan_and_inf(engine):
    import torch

    P = configs.random_draw(4, seed=9, jet="gaussian", theta_obs_max=0.4)
    t, nu = np.logspace(3, 6, 8), np.array([1e9, 1e17])
    dev = torch.device("cuda:0")
    d_p = torch.from_numpy(P.view(np.uint8).copy()).to(dev)
    d_t, d_nu = torch.from_numpy(t).to(dev), torch.from_numpy(nu).to(dev)
    d_out = torch.empty((P.size, abi.NCOMP, nu.size, t.size), dtype=torch.float64, device=dev)
    d_st = torch.zeros(P.size, dtype=torch.int32, device=dev)
    try:
        engine.set_capacity(40, 2)
        engine.flux_density_grid_dev(d_p.data_ptr(), P.size, d_t.data_ptr(), t.size, d_nu.data_ptr(), nu.size, d_out.data_ptr(),
                                     d_st.data_ptr())
        engine.synchronize()
        assert ((d_st.cpu().numpy() & abi.ST_CAPACITY) != 0).all()
        assert torch.isnan(d_out).all()
        # a host-buffer call in between sizes its own batch and must not disturb the configured device capacity
        assert np.isfinite(engine.flux_density_grid(P, t, nu)).all()
        engine.set_capacity(384, 128)
        engine.flux_density_grid(configs.random_draw(2, seed=1), t, nu)  # tight per-batch capacities (tophat on axis)
        engine.flux_density_grid_dev(d_p.data_ptr(), P.size, d_t.data_ptr(), t.size, d_nu.data_ptr(), nu.size, d_out.data_ptr(),
                                     d_st.data_ptr())
        engine.synchronize()
        assert int(d_st.abs().sum()) == 0
        np.testing.assert_allclose(d_out.cpu().numpy(), engine.flux_density_grid(P, t, nu), rtol=1e-13)
    finally:
        engine.set_capacity(384, 128)


def test_batches_beyond_one_pass(engine):
    # more than MAX_MODELS_PER_PASS (and than the 65535 limit of gridDim.y): consecutive passes, same rows
    n = 70001
    P = np.tile(configs.random_draw(257, seed=12), n // 257 + 1)[:n]
    t, nu = np.array([1e3, 1e4, 1e5]), np.array([1e14])
    f, st = engine.flux_density_grid(P, t, nu, return_status=True)
    assert f.shape == (n, abi.NCOMP, 1, 3) and (st == 0).all() and np.isfinite(f).all()
    small = engine.flux_density_grid(P[:257], t, nu)
    np.testing.assert_allclose(f[:257], small, rtol=1e-13)
    np.testing.assert_allclose(f[-257:], np.roll(small, -(n - 257) % 257, axis=0), rtol=1e-13)


def test_observation_arrays_are_validated(engine):
    p, t, nu = configs.C1()
    for bad_t in ([0.0, 1e3], [-1.0, 1e3], [1e3, np.inf], [np.nan, 1e3]):
        with pytest.raises(ValueError):
            engine.flux_density_grid(p, np.array(bad_t), nu)
    for bad_nu in ([0.0], [-1e9], [np.inf]):
        with pytest.raises(ValueError, match="frequenc"):
            engine.flux_density_grid(p, t, np.array(bad_nu))
    with pytest.raises(ValueError, match="nu_max"):
        engine.flux_band(p, t, 1e10, 1e9, 5)
    with pytest.raises(ValueError, match="no data"):
        engine.chi2(p, None, ())
