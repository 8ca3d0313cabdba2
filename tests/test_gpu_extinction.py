"""Fitted host-galaxy extinction: a per-walker A_V shifts the observed point data to lnF_obs + A_V * ext_k inside the
chi-squared kernel (vag_chi2_ext), so an ensemble with a sampled A_V stays one batched call.

GPU tier: Engine.chi2(extinction=...) against a same-batch oracle (one call per distinct A_V with the shift computed
in numpy), status and +inf rules, validation, the second pass of a batch beyond 32768 models, GpuFitterEvaluator on
the device.  CPU tier: GpuFitterEvaluator and BatchedLikelihood with recording engines, the walker partition with a
per-walker column under gloo, and -- where the reference checkout exists -- the shift convention against Fitter._evaluate.
"""
import os
import shutil
import subprocess
import sys
import textwrap
import types

import numpy as np
import pytest

from vegasafterglow_b200 import abi, configs, fitting, parallel

from tests.test_integration_patch import REF_PKG, _stub_samplers  # noqa: E402  the reference checkout's package

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- data ------------------------------------------------------------------------------------------------------------
def _points(seed=0):
    """Config-5-like point data: 5 bands x 20 epochs, power-law fluxes with noise; a finite ext_k for every point."""
    rng = np.random.default_rng(seed)
    t = np.sort(np.tile(np.logspace(2.5, 6.5, 20), 5))
    nu = np.tile([1e9, 5e9, 4.84e14, 1e17, 1e18], 20)
    flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
    pts = fitting.consolidate_data(t, nu, flux, 0.2 * flux, rng.uniform(0.5, 2.0, t.size))
    ext = rng.uniform(0.0, 1.7, t.size)
    return pts, ext


def _xray_band():
    tb = np.logspace(3.2, 5.5, 6)
    fb = 1e-12 * (tb / 1e4) ** -1.2
    return fitting.band_obs(tb, fb, 0.2 * fb, 7.25e16, 2.4e18, 5)


def _mixed_batch():
    P = np.concatenate([configs.random_draw(16, seed=11), configs.random_draw(16, seed=12, rvs=True),
                        configs.random_draw(16, seed=13, jet="gaussian", theta_obs_max=0.4)])
    return P[np.random.default_rng(5).permutation(P.size)]


def _same_batch_oracle(engine, P, pts, bands, ext, A_V):
    """One Engine.chi2 per distinct A_V on the whole batch, the shift computed in numpy; the rows of that value."""
    chi2, st = np.full(P.size, np.nan), np.full(P.size, -1, dtype=np.int32)
    for av in np.unique(A_V):
        sel = A_V == av
        c, s = engine.chi2(P, (pts[0], pts[1], pts[2] + av * ext, pts[3], pts[4]), bands, return_status=True)
        chi2[sel], st[sel] = c[sel], s[sel]
    return chi2, st


# ---- GPU tier ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("series_mode", [0, 1, 2])
def test_extinction_equals_the_same_batch_oracle(engine, series_mode):
    P = _mixed_batch()
    pts, ext = _points()
    bands = [_xray_band()]
    A_V = np.tile([0.0, 0.37, 1.13, 1.9], P.size // 4)[np.random.default_rng(2).permutation(P.size)]
    try:
        engine.set_series_mode(series_mode)
        chi2, st = engine.chi2(P, pts, bands, return_status=True, extinction=(ext, A_V))
        want, want_st = _same_batch_oracle(engine, P, pts, bands, ext, A_V)
    finally:
        engine.set_series_mode(0)
    assert np.isfinite(chi2).all()
    assert np.array_equal(chi2, want)
    assert np.array_equal(st, want_st)


@pytest.mark.gpu
def test_zero_extinction_is_the_plain_likelihood(engine):
    P = _mixed_batch()
    pts, ext = _points(1)
    for bands in ((), [_xray_band()]):
        plain, st0 = engine.chi2(P, pts, bands, return_status=True)
        n0 = engine.last_launch_count()
        shifted, st1 = engine.chi2(P, pts, bands, return_status=True, extinction=(ext, np.zeros(P.size)))
        assert engine.last_launch_count() == n0
        assert np.array_equal(shifted, plain) and np.array_equal(st1, st0)


@pytest.mark.gpu
def test_non_finite_av_and_ode_failure_give_inf(engine):
    from tests.helpers import load_golden

    P = np.concatenate([configs.random_draw(6, seed=5), configs.random_draw(6, seed=6, rvs=True)])
    g = load_golden("series_rs_tophat_ism")
    t, nu = g["t"], g["nu"]
    pts = (t, nu, np.log(np.full(t.size, 1e-27)), np.full(t.size, 0.1), np.ones(t.size))
    ext = np.linspace(0.0, 1.5, t.size)
    A_V = np.linspace(0.1, 1.2, P.size)
    base = engine.chi2(P, pts, (), extinction=(ext, A_V))
    bad = A_V.copy()
    bad[4] = np.nan
    chi2 = engine.chi2(P, pts, (), extinction=(ext, bad))
    assert np.isinf(chi2[4]) and chi2[4] > 0
    assert np.array_equal(np.delete(chi2, 4), np.delete(base, 4))
    try:
        engine.debug_set_ode_limits(max_fails=1)
        chi2, st = engine.chi2(P, pts, (), return_status=True, extinction=(ext, A_V))
    finally:
        engine.debug_set_ode_limits(0, 0)
    hit = (st & abi.ST_ODE_FAIL500) != 0
    assert hit[6:].any(), "a reverse-shock solve rejects at least one step"
    assert np.isposinf(chi2[hit]).all() and np.isfinite(chi2[~hit]).all()


@pytest.mark.gpu
def test_extinction_arguments_are_validated(engine):
    P = configs.random_draw(3, seed=1)
    pts, ext = _points()
    A_V = np.ones(P.size)
    with pytest.raises(ValueError, match="ext_k"):
        engine.chi2(P, pts, (), extinction=(ext[:-1], A_V))
    with pytest.raises(ValueError, match="A_V"):
        engine.chi2(P, pts, (), extinction=(ext, A_V[:-1]))
    for v in (np.nan, np.inf):
        e = ext.copy()
        e[7] = v
        with pytest.raises(ValueError, match="finite"):
            engine.chi2(P, pts, (), extinction=(e, A_V))
    with pytest.raises(ValueError, match="points"):
        engine.chi2(P, None, [_xray_band()], extinction=(ext, A_V))


@pytest.mark.gpu
def test_chi2_ext_arguments_are_checked_before_any_work(engine):
    import ctypes as C

    P = np.ascontiguousarray(configs.random_draw(3, seed=1), dtype=abi.PARAMS_DTYPE)
    pts, ext = _points()
    pts = [np.ascontiguousarray(a, dtype=np.float64) for a in pts]
    A_V = np.ones(P.size)
    bad_ext = ext.copy()
    bad_ext[7] = np.inf
    bt, bl, bs, bw = np.array([1e3, 1e4]), np.zeros(2), np.ones(2), np.ones(2)
    xb = dict(t=bt.ctypes.data, lnF_obs=bl.ctypes.data, sigma_ln=bs.ctypes.data, w=bw.ctypes.data, n=bt.size,
              nu_min=7.25e16, nu_max=2.4e18, num_nu=5)

    def call(n_points=pts[0].size, ext=None, A_V=None, **band):
        b = dict(xb, **band)
        arr = (abi.BandObs * 1)(abi.BandObs(b["t"], b["lnF_obs"], b["sigma_ln"], b["w"], b["n"], b["nu_min"], b["nu_max"],
                                            b["num_nu"]))
        chi2 = np.full(P.size, 7.0)
        st = np.full(P.size, 99, dtype=np.int32)
        rc = engine._lib.vag_chi2_ext(engine._h, P.ctypes.data, P.size, *[a.ctypes.data for a in pts],
                                      None if ext is None else ext.ctypes.data, n_points,
                                      None if A_V is None else A_V.ctypes.data, C.cast(arr, C.c_void_p), 1, chi2.ctypes.data,
                                      st.ctypes.data)
        return rc, bool((chi2 == 7.0).all() and (st == 99).all())

    assert call(ext=ext, A_V=A_V) == (abi.VAG_OK, False)
    # word in the message -> arguments
    cases = {
        "band 0: empty (n = 0)": dict(n=0),
        "band 0: data arrays must not be NULL": dict(lnF_obs=None),
        "band 0: nu_max": dict(nu_max=1e16),
        "band 0: num_nu": dict(num_nu=1),
        "both": dict(ext=ext),
        "extinction needs point data": dict(n_points=0, ext=ext, A_V=A_V),
        "finite": dict(ext=bad_ext, A_V=A_V),
    }
    for word, kw in cases.items():
        rc, untouched = call(**kw)
        assert rc == abi.VAG_ERR_INVALID, word
        assert untouched, word
        msg = engine._lib.vag_last_error().decode()
        assert word in msg, (word, msg)


@pytest.mark.gpu
def test_extinction_across_the_pass_boundary(engine):
    # 32768 models per pass: the second pass must read A_V from its own offset
    n = 32768 + 64
    P = configs.random_draw(n, seed=21)
    t = np.array([1e3, 1e4, 1e5, 1e6])
    nu = np.array([1e9, 4.84e14, 1e17, 1e18])
    pts = fitting.consolidate_data(t, nu, 1e-27 * (t / 1e4) ** -1.0, 0.2e-27 * (t / 1e4) ** -1.0)
    ext = np.array([0.0, 1.3, 0.4, 0.05])
    A_V = np.array([0.2, 0.9, 1.6])[(np.arange(n) // 16) % 3]
    assert A_V[32767] != A_V[32768] and A_V[32768] != A_V[0]
    chi2, st = engine.chi2(P, pts, (), return_status=True, extinction=(ext, A_V))
    want, want_st = _same_batch_oracle(engine, P, pts, (), ext, A_V)
    assert np.array_equal(chi2, want) and np.array_equal(st, want_st)


# ---- stand-in Fitter (the attributes GpuFitterEvaluator reads) ---------------------------------------------------------
_NAMES = ("E_iso", "Gamma0", "theta_c", "n_ism", "eps_e", "eps_B", "p", "eps_e_r", "eps_B_r", "p_r")
_LOG = (True, True, False, True, True, True, False, True, True, False)


def _to_params(theta):
    kw = {n: (10.0 ** v if lg else v) for n, lg, v in zip(_NAMES, _LOG, theta[:-1])}
    return types.SimpleNamespace(theta_v=0.0, A_V=theta[-1], **kw)


def _stand_in_fitter(pts, ext, band_obs=(), ext_law="smc"):
    t, nu, lnF, sig, w = pts
    return types.SimpleNamespace(
        _custom_extinction=False, _consolidate_data=lambda: None, _to_params=_to_params, _all_t=t, _all_nu=nu,
        _all_log_flux=lnF, _all_log_err=sig, _all_weights=w, _band_obs=list(band_obs), _ext_law=ext_law, _ext_kernel=ext,
        _custom_jet=False, _custom_medium=False, jet="tophat", medium="ism", magnetar=False, lumi_dist=1e26, z=0.1,
        fwd_ssc=False, kn=False, rvs_shock=True, rvs_ssc=False, resolution=None, rtol=None, radiative_fireball=False)


def _thetas(n, seed):
    rng = np.random.default_rng(seed)
    return np.column_stack([rng.uniform(51, 54, n), rng.uniform(1.7, 3, n), rng.uniform(0.03, 0.4, n),
                            rng.uniform(-3, 1, n), rng.uniform(-2, -0.5, n), rng.uniform(-4, -1, n),
                            rng.uniform(2.1, 2.8, n), rng.uniform(-2, -0.5, n), rng.uniform(-4, -1, n),
                            rng.uniform(2.1, 2.8, n), rng.uniform(0, 2, n)])


class _CountingLib:
    """The engine's library with every vag_chi2* call recorded."""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        f = getattr(self._lib, name)
        if not name.startswith("vag_chi2"):
            return f

        def counted(*args):
            self.calls.append(name)
            return f(*args)

        return counted


@pytest.mark.gpu
def test_fitter_evaluator_is_one_call_on_the_device(engine, monkeypatch):
    from vegasafterglow_b200.integration import GpuFitterEvaluator, params_from_fitter

    pts, ext = _points(3)
    tb = np.logspace(3.2, 5.5, 6)
    band = types.SimpleNamespace(t=tb, flux=1e-12 * (tb / 1e4) ** -1.2, err=2e-13 * (tb / 1e4) ** -1.2, nu_min=7.25e16,
                                 nu_max=2.4e18, num_points=5, weights=None)
    fitter = _stand_in_fitter(pts, ext, [band])
    th = _thetas(24, 4)
    ev = GpuFitterEvaluator(fitter, engine)
    counting = _CountingLib(engine._lib)
    with monkeypatch.context() as m:
        m.setattr(engine, "_lib", counting)
        chi2 = ev.chi2(th)
    assert counting.calls == ["vag_chi2_ext"]
    # the grouped computation this replaces: one evaluation per distinct A_V, i.e. per walker
    P = params_from_fitter(fitter, [_to_params(x) for x in th])
    want = np.array([engine.chi2(P[i:i + 1], (pts[0], pts[1], pts[2] + th[i, -1] * ext, pts[3], pts[4]), ev.bands)[0]
                     for i in range(len(th))])
    assert np.isfinite(want).all()
    np.testing.assert_allclose(chi2, want, rtol=1e-9)


# ---- CPU tier ------------------------------------------------------------------------------------------------------------
class _RecordingEngine:
    def __init__(self):
        self.calls = []

    def chi2(self, P, points, bands, extinction=None):
        self.calls.append(("chi2", len(P), points, len(bands), extinction))
        return np.arange(len(P), dtype=np.float64) + 1.0

    def chi2_series(self, P, *points):
        self.calls.append(("chi2_series", len(P), points, 0, None))
        return np.arange(len(P), dtype=np.float64) + 1.0


@pytest.mark.parametrize("distributed", [False, True])
def test_fitter_evaluator_passes_av_in_walker_order(distributed):
    from vegasafterglow_b200.integration import GpuFitterEvaluator

    pts, ext = _points(4)
    th = _thetas(9, 6)
    th[3, 4] = 0.5  # eps_e = 10^0.5 > 1: the model constructor rejects the walker
    eng = _RecordingEngine()
    chi2 = GpuFitterEvaluator(_stand_in_fitter(pts, ext), eng, distributed=distributed).chi2(th)
    assert len(eng.calls) == 1
    name, n, points, n_bands, extinction = eng.calls[0]
    assert name == "chi2" and n == 8 and n_bands == 0 and points[2] is pts[2]
    ok = np.arange(9) != 3
    assert extinction[0] is ext
    np.testing.assert_array_equal(extinction[1], th[ok, -1])  # one process: every valid walker, in walker order
    np.testing.assert_array_equal(chi2[ok], np.arange(8) + 1.0)
    assert np.isposinf(chi2[3])


def test_fitter_evaluator_with_band_data_only_applies_no_extinction():
    from vegasafterglow_b200.integration import GpuFitterEvaluator

    tb = np.logspace(3.2, 5.5, 6)
    band = types.SimpleNamespace(t=tb, flux=1e-12 * np.ones(6), err=2e-13 * np.ones(6), nu_min=7.25e16, nu_max=2.4e18,
                                 num_points=5, weights=None)
    empty = (np.zeros(0),) * 5
    eng = _RecordingEngine()
    ev = GpuFitterEvaluator(_stand_in_fitter(empty, np.zeros(0), [band]), eng)
    chi2 = ev.chi2(_thetas(4, 7))
    assert ev.ext_kernel is None and np.isfinite(chi2).all()
    assert [(c[0], c[1], c[2], c[3], c[4]) for c in eng.calls] == [("chi2", 4, None, 1, None)]


def test_fitter_without_extinction_law_keeps_the_plain_call():
    from vegasafterglow_b200.integration import GpuFitterEvaluator

    pts, ext = _points(4)
    eng = _RecordingEngine()
    GpuFitterEvaluator(_stand_in_fitter(pts, ext, ext_law=None), eng).chi2(_thetas(5, 8))
    assert [c[0] for c in eng.calls] == ["chi2_series"] and eng.calls[0][4] is None


def test_likelihood_fits_av_with_a_sorted_ext_kernel():
    t = np.array([1e5, 1e3, 1e4, 1e3])
    nu = np.array([1e9, 4.84e14, 1e17, 1e9])
    flux, err = np.array([1.0, 2.0, 3.0, 4.0]), np.array([0.1, 0.2, 0.3, 0.4])
    ext = np.array([0.5, 1.5, 2.5, 3.5])
    tmpl = configs.make()
    with pytest.raises(ValueError, match="ext_kernel"):
        fitting.BatchedLikelihood(None, tmpl, ["E_iso", "A_V"], [True, False], t, nu, flux, err)
    with pytest.raises(ValueError, match="ext_kernel"):
        fitting.BatchedLikelihood(None, tmpl, ["E_iso", "A_V"], [True, False], t, nu, flux, err, ext_kernel=ext[:3])
    eng = _RecordingEngine()
    lk = fitting.BatchedLikelihood(eng, tmpl, ["E_iso", "A_V", "p"], [True, False, False], t, nu, flux, err,
                                   ext_kernel=ext)
    # the stable time order of consolidate_data: 1e3 (index 1), 1e3 (index 3), 1e4, 1e5
    np.testing.assert_array_equal(lk.t, [1e3, 1e3, 1e4, 1e5])
    np.testing.assert_array_equal(lk.ext_kernel, [1.5, 3.5, 2.5, 0.5])
    s = np.array([[52.0, 0.3, 2.2], [53.0, 1.7, 2.4], [52.5, 0.0, 2.6]])
    P = lk.to_params(s)
    Q = np.repeat(configs.make(), 3)
    Q["E_iso"], Q["fwd"]["p"] = 10.0 ** s[:, 0], s[:, 2]
    assert P.tobytes() == Q.tobytes()  # A_V is not a model parameter
    lk.chi2(s)
    (name, n, points, n_bands, extinction), = eng.calls
    assert name == "chi2" and n == 3 and points[0] is lk.t
    assert extinction[0] is lk.ext_kernel
    np.testing.assert_array_equal(extinction[1], s[:, 1])
    eng.calls.clear()
    lk.distributed = True
    lk.chi2(s)
    (_, _, _, _, extinction), = eng.calls
    np.testing.assert_array_equal(extinction[1], s[:, 1])


_GLOO_WORKER = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, {root!r})
    import numpy as np, torch.distributed as dist
    from vegasafterglow_b200 import configs, parallel
    from oracle.hostemu import emu
    rank = int(sys.argv[1])
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2)
    P = configs.random_draw(7, seed=3, rvs=True)
    ts = np.sort(np.tile(np.logspace(3, 6, 4), 2)); nus = np.tile([1e9, 4.84e14], 4)
    lnF = np.log(np.full(ts.size, 1e-27)); sig = np.full(ts.size, 0.1); w = np.ones(ts.size)
    ext = np.tile([0.0, 1.4], 4)
    A_V = 0.1 + 0.2 * np.arange(7)
    seen = []
    def host_eval(block, av):  # test-only evaluator: the kernel bodies executed on the host, the shift in numpy
        seen.append(av.copy())
        f, _ = emu.flux_density_series(block, ts, nus)
        d = (lnF + av[:, None] * ext - np.log(np.maximum(f[:, 0], 1e-300))) / sig
        return np.sum(w * d * d, axis=1)
    full = host_eval(P, A_V)
    seen.clear()
    chi2 = parallel.partitioned_chi2(None, P, ts, nus, lnF, sig, w, evaluate=host_eval, per_walker=(A_V,))
    assert np.array_equal(chi2, full), (chi2, full)
    mine = parallel.balanced_assignment(parallel.cost_proxy(P, ts.min(), ts.max()), 2)[rank]
    assert np.array_equal(seen[-1], A_V[mine])
    chi2c = parallel.partitioned_chi2(None, P, ts, nus, lnF, sig, w, evaluate=host_eval, balance=False, per_walker=(A_V,))
    assert np.array_equal(chi2c, full)
    lo, hi = parallel.partition(7, 2, rank)
    assert np.array_equal(seen[-1], A_V[lo:hi])
    dist.destroy_process_group()
    print("ok", rank)
""")


def test_per_walker_columns_follow_the_partition_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER.format(root=ROOT, port=28517 + os.getpid() % 1000))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
             for r in range(2)]
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        assert "ok" in out


# ---- against the reference's own Fitter, where a checkout exists ------------------------------------------------------
@pytest.fixture(scope="module")
def refpkg(tmp_path_factory):
    """The reference's Python package assembled in a temp directory around the pybind module oracle/_ref."""
    from oracle import ref

    if not os.path.isdir(REF_PKG):
        pytest.skip("needs the reference checkout")
    if not ref.available():
        pytest.skip("oracle/_ref not built")
    base = tmp_path_factory.mktemp("refpkg_ext")
    pkg = base / "VegasAfterglow"
    pkg.mkdir()
    for name in os.listdir(REF_PKG):
        if name not in ("fitting", "__pycache__"):
            os.symlink(os.path.join(REF_PKG, name), pkg / name)
    (pkg / "fitting").mkdir()
    for name in os.listdir(os.path.join(REF_PKG, "fitting")):
        if name.endswith(".py"):
            shutil.copy(os.path.join(REF_PKG, "fitting", name), pkg / "fitting" / name)
    so = [f for f in os.listdir(os.path.join(ROOT, "oracle", "_ref")) if f.startswith("VegasAfterglowC")][0]
    os.symlink(os.path.join(ROOT, "oracle", "_ref", so), pkg / so)
    stubs = _stub_samplers()  # emcee / bilby are absent: minimal stand-ins
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    sys.path.insert(0, str(base))
    for k in [k for k in sys.modules if k == "VegasAfterglow" or k.startswith("VegasAfterglow.")]:
        del sys.modules[k]
    if ref._pymod is not None:  # the pybind module may be loaded only once per process: reuse an earlier load
        sys.modules["VegasAfterglow.VegasAfterglowC"] = ref._pymod
    import VegasAfterglow.fitting as fitting_mod

    ref._pymod = sys.modules["VegasAfterglow.VegasAfterglowC"]
    yield fitting_mod
    sys.path.remove(str(base))
    for k, v in saved.items():
        if v is None:
            sys.modules.pop(k, None)
        else:
            sys.modules[k] = v


class _ReferenceBackedEngine:
    """Engine stand-in answered by the unmodified reference: the shifted point data evaluated walker by walker."""

    def __init__(self):
        self.calls = []

    def chi2(self, P, points, bands, extinction=None):
        from oracle import ref

        assert not bands
        self.calls.append(len(P))
        t, nu, lnF, sig, w = points
        ext, A_V = extinction
        return np.array([ref.chi2_series(P[i:i + 1], t, nu, lnF + A_V[i] * ext, sig, w, n_threads=1)[0]
                         for i in range(len(P))])


def _reference_fitter_with_extinction(fm):
    """A tophat Fitter with optical and X-ray points and a built-in extinction law; None if the reference offers no
    built-in law through its constructor."""
    import inspect

    keys = [k for k in inspect.signature(fm.Fitter).parameters if "ext" in k.lower()]
    for key in keys:
        for law in ("smc", "SMC", "mw", "MW", "lmc", "LMC"):
            try:
                f = fm.Fitter(z=0.1, lumi_dist=1e27, jet="tophat", medium="ism", **{key: law})
            except (TypeError, ValueError, KeyError):
                continue
            if getattr(f, "_ext_law", None) is not None:
                return f
    return None


def test_fitted_extinction_matches_the_reference_fitter(refpkg):
    from VegasAfterglow import ParamDef, Scale

    from vegasafterglow_b200.integration import GpuFitterEvaluator

    f = _reference_fitter_with_extinction(refpkg)
    if f is None:
        pytest.skip("the reference Fitter takes no built-in extinction law")
    t = np.logspace(3, 6, 6)
    rng = np.random.default_rng(3)
    for nu, amp in ((1e9, 1e-27), (4.84e14, 3e-28), (6.0e14, 2e-28), (1e18, 1e-30)):
        f.add_flux_density(nu, t, amp * (t / 1e4) ** -1.0 * (1 + 0.05 * rng.standard_normal(t.size)), amp * 0.1 * np.ones(t.size))
    defs = [ParamDef("E_iso", 1e51, 1e54, Scale.log), ParamDef("Gamma0", 50, 800, Scale.log),
            ParamDef("theta_c", 0.03, 0.4, Scale.linear), ParamDef("n_ism", 1e-3, 10, Scale.log),
            ParamDef("eps_e", 1e-2, 0.5, Scale.log), ParamDef("eps_B", 1e-4, 0.1, Scale.log),
            ParamDef("p", 2.1, 2.8, Scale.linear), ParamDef("theta_v", 0.0, 0.0, Scale.fixed),
            ParamDef("A_V", 0.0, 2.0, Scale.linear)]
    f.fit(defs, sampler="emcee", nwalkers=8, nsteps=1, nburn=0, npool=1, top_k=1)  # sets the parameter transformer
    th = np.array([[52.3, 2.4, 0.12, -0.5, -1.2, -2.5, 2.35, 0.0], [53.1, 2.1, 0.3, 0.5, -0.7, -3.0, 2.6, 0.8],
                   [52.7, 2.2, 0.2, -1.0, -1.0, -2.0, 2.2, 1.7]])
    eng = _ReferenceBackedEngine()
    ev = GpuFitterEvaluator(f, eng)
    want = np.array([f._evaluate(f._to_params(x)) for x in th])
    np.testing.assert_allclose(ev.chi2(th), want, rtol=1e-9)
    assert eng.calls == [3]
