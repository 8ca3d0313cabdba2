"""The likelihood on device buffers, planned on the device: vag_chi2_dev / vag_flux_band_dev / vag_params_validate_batch_dev
and fitting.DeviceLikelihood.

GPU tier: vag_chi2_dev and vag_flux_band_dev against their host-buffer counterparts bit for bit (every term combination,
series modes 0/1/2, the 32768-model pass boundary), launch counts, device validation and capacities against the host's on
a seeded fuzz, rejected walkers, a walker beyond the default capacity, DeviceLikelihood against BatchedLikelihood.
CPU tier: record assembly, the reason-code validation against the previous messages, DeviceLikelihood under gloo.
"""
import ctypes as C
import math
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from vegasafterglow_b200 import abi, configs, fitting

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLANNING_LAUNCHES = 2  # k_plan before the call's work, k_reject after it

_F8 = [(n,) for n in abi.PARAMS_DTYPE.names if abi.PARAMS_DTYPE[n] == np.float64] + \
      [(s, n) for s in ("fwd", "rvs") for n in abi.RADIATION_DTYPE.names if abi.RADIATION_DTYPE[n] == np.float64]


def _field(P, path):
    return P[path[0]] if len(path) == 1 else P[path[0]][path[1]]


# ---- seeded fuzz of parameter sets ------------------------------------------------------------------------------------
_SPECIAL = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1.0, np.nextafter(1.0, 2.0), np.nextafter(1.0, 0.0), np.pi / 2,
                     np.nextafter(np.pi / 2, 4.0), np.pi, np.nextafter(np.pi, 4.0), -1.0, 1e308, 5e-324, 0.5, 3.0])


def fuzz_records(n=100_000, seed=0):
    """Every jet and medium type, switches on and off, and in every float64 field now and then one of _SPECIAL
    (NaN, +-inf, 0, 1 and 1 + ulp, pi/2 and pi and one ulp above, ...).  The first records are named boundary cases."""
    rng = np.random.default_rng(seed)
    P = abi.default_params(n)
    P["jet_type"] = rng.integers(0, 6, n)
    P["medium_type"] = rng.integers(0, 2, n)
    P["spreading"] = rng.integers(0, 2, n)
    P["theta_c"] = rng.uniform(0.02, 0.4, n)
    P["E_iso"] = 10.0 ** rng.uniform(50, 54, n)
    P["Gamma0"] = 10.0 ** rng.uniform(0.3, 3.3, n)
    P["k_e"], P["k_g"] = rng.uniform(0.5, 4, n), rng.uniform(0.5, 4, n)
    P["theta_w"] = P["theta_c"] + rng.uniform(0.01, 0.5, n)
    P["E_iso_w"], P["Gamma0_w"] = 10.0 ** rng.uniform(48, 52, n), 10.0 ** rng.uniform(0.3, 2.5, n)
    P["n_ism"], P["A_star"] = 10.0 ** rng.uniform(-3, 1, n), 10.0 ** rng.uniform(-2, 0, n)
    P["lumi_dist"], P["z"] = 10.0 ** rng.uniform(26, 28.5, n), rng.uniform(0, 2, n)
    P["theta_obs"] = np.where(rng.random(n) < 0.5, 0.0, rng.uniform(0, 1.5, n))
    P["has_rvs"] = rng.integers(0, 2, n)
    P["has_magnetar"] = rng.random(n) < 0.2
    P["magnetar_L0"], P["magnetar_t0"], P["magnetar_q"] = 1e46, 1e3, 2.0
    for k, lo, hi in (("theta_resol", 0.05, 2.0), ("phi_resol", 0.02, 0.5), ("t_resol", 2, 20), ("rtol", 1e-8, 1e-3)):
        P[k] = np.where(rng.random(n) < 0.7, 0.0, rng.uniform(lo, hi, n))
    for path in _F8:
        col = _field(P, path)
        hit = rng.random(n) < 0.02
        col[hit] = rng.choice(_SPECIAL, hit.sum())
    hit = rng.random(n) < 0.01
    P["jet_type"][hit] = rng.choice([-1, 6, 7], hit.sum())
    hit = rng.random(n) < 0.01
    P["medium_type"][hit] = rng.choice([-1, 2], hit.sum())
    # named boundaries: accepted theta_c = pi/2 and Gamma0 = 1 + ulp; rejected Gamma0 = 1, wind n0 = 0, rtol = 1
    base = configs.make()
    named = np.repeat(base, 5)
    named["theta_c"][0] = np.pi / 2
    named["Gamma0"][1] = np.nextafter(1.0, 2.0)
    named["Gamma0"][2] = 1.0
    named["medium_type"][3], named["A_star"][3], named["n0"][3] = abi.MEDIUM_WIND, 0.1, 0.0
    named["rtol"][4] = 1.0
    P[:5] = named
    return P


# ---- the previous host validation, message for message (the checks vag_params_validate made before they were
# restated as a reason code shared with the device) ------------------------------------------------------------------
def _previous_validate(p):
    fin = math.isfinite

    def fp(x):
        return fin(x) and x > 0

    def rng_oi(v, lo, hi):
        return fin(v) and lo < v <= hi

    jt, mt = int(p["jet_type"]), int(p["medium_type"])
    if jt < 0 or jt > 5:
        return "jet_type must be one of VAG_JET_* (0..5)"
    if mt < 0 or mt > 1:
        return "medium_type must be 0 (ISM) or 1 (wind)"
    if not rng_oi(p["theta_c"], 0.0, math.pi / 2):
        return "theta_c must be in (0, pi/2]"
    has_core, has_wing = jt != abi.JET_POWERLAW_WING, jt >= abi.JET_TWO_COMPONENT
    if has_core and not fp(p["E_iso"]):
        return "E_iso must be finite and > 0"
    if has_core and not (fin(p["Gamma0"]) and p["Gamma0"] > 1.0):
        return "Gamma0 must be > 1"
    if not fp(p["duration"]):
        return "duration must be finite and > 0"
    if jt in (abi.JET_POWERLAW, abi.JET_STEP_POWERLAW, abi.JET_POWERLAW_WING) and (not fp(p["k_e"]) or not fp(p["k_g"])):
        return "k_e and k_g must be finite and > 0"
    if has_wing:
        if not fp(p["E_iso_w"]):
            return "E_iso_w must be finite and > 0"
        if not (fin(p["Gamma0_w"]) and p["Gamma0_w"] > 1.0):
            return "Gamma0_w must be > 1"
    if jt == abi.JET_TWO_COMPONENT:
        if not rng_oi(p["theta_w"], 0.0, math.pi / 2):
            return "theta_w must be in (0, pi/2]"
        if not p["theta_w"] > p["theta_c"]:
            return ("theta_w (wing angle) must be greater than theta_c (core angle), got theta_w=%f, theta_c=%f"
                    % (p["theta_w"], p["theta_c"]))
    if not (fin(p["sigma0"]) and p["sigma0"] >= 0):
        return "sigma0 must be finite and >= 0"
    if p["has_magnetar"]:
        for k, name in (("magnetar_L0", "L0"), ("magnetar_t0", "t0"), ("magnetar_q", "q")):
            if not fp(p[k]):
                return f"{name} must be finite and > 0"
        if jt == abi.JET_POWERLAW_WING:
            return "PowerLawWing takes no magnetar (pybind/pybind.cpp:220-223)"
    if mt == abi.MEDIUM_ISM:
        if not (fin(p["n_ism"]) and p["n_ism"] >= 0):
            return "n_ism must be finite and >= 0"
    else:
        if not fp(p["A_star"]):
            return "A_star must be finite and > 0"
        if not (fin(p["n_ism"]) and p["n_ism"] >= 0):
            return "n_ism must be finite and >= 0"
        if not p["n0"] > 0:
            return "n0 must be > 0 (or +inf for no floor)"
        if not fin(p["wind_k_m"]):
            return "k_m must be finite and > 0"
    if not fp(p["lumi_dist"]):
        return "lumi_dist must be finite and > 0"
    if not (fin(p["z"]) and p["z"] >= 0):
        return "z must be finite and >= 0"
    if not (fin(p["theta_obs"]) and 0 <= p["theta_obs"] <= math.pi):
        return "theta_obs must be in [0, pi]"
    if not fin(p["phi_obs"]):
        return "phi_obs must be finite"
    for who, r, on in (("fwd_rad", p["fwd"], True), ("rvs_rad", p["rvs"], bool(p["has_rvs"]))):
        if not on:
            continue
        for k in ("eps_e", "eps_B", "xi_e"):
            if not rng_oi(r[k], 0.0, 1.0):
                return f"{who}.{k} must be in (0, 1]"
        if not (fin(r["p"]) and r["p"] > 1.0):
            return f"{who}.p must be > 1"
    if p["rtol"] > 0 and not p["rtol"] < 1:
        return "rtol must be in (0, 1)"
    if not all(fin(p[k]) for k in ("rtol", "phi_resol", "theta_resol", "t_resol")):
        return "resolutions and rtol must be finite"
    return None


def test_validation_codes_and_messages_are_unchanged():
    from vegasafterglow_b200 import _lib

    lib = _lib.load()
    P = fuzz_records(100_000, seed=7)
    n_bad = 0
    for i in range(P.size):
        rec = P[i:i + 1]
        rc = lib.vag_params_validate(rec.ctypes.data)
        want = _previous_validate(P[i])
        if want is None:
            assert rc == abi.VAG_OK, (i, P[i])
        else:
            n_bad += 1
            assert rc == abi.VAG_ERR_INVALID and lib.vag_last_error().decode() == want, (i, want)
    assert 0.2 * P.size < n_bad < 0.8 * P.size  # the fuzz exercises both outcomes


# ---- record assembly ------------------------------------------------------------------------------------------------
_NAMES = ["E_iso", "Gamma0", "theta_c", "n_ism", "eps_e", "eps_B", "p", "A_V", "theta_v", "p_r"]
_LOG = [True, True, False, True, True, True, False, False, False, False]


def _template():
    return configs.make(rvs=(0.1, 0.01, 2.3), lumi_dist=1e28, z=0.3)


def _samples(n, seed):
    rng = np.random.default_rng(seed)
    return np.column_stack([rng.uniform(51, 54, n), rng.uniform(1.7, 3, n), rng.uniform(0.03, 0.4, n),
                            rng.uniform(-3, 1, n), rng.uniform(-2, 0.4, n), rng.uniform(-4, -1, n),
                            rng.uniform(2.1, 2.8, n), rng.uniform(0, 2, n), rng.uniform(0, 0.01, n),
                            rng.uniform(2.1, 2.8, n)])


def _point_data(seed=0):
    rng = np.random.default_rng(seed)
    t = np.sort(np.tile(np.logspace(2.5, 6.5, 12), 3))
    nu = np.tile([1e9, 4.84e14, 1e18], 12)
    flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
    return t, nu, flux, 0.2 * flux, rng.uniform(0.0, 1.7, t.size)


def _band():
    tb = np.logspace(3.2, 5.5, 6)
    fb = 1e-12 * (tb / 1e4) ** -1.2
    return dict(t=tb, flux=fb, err=0.2 * fb, nu_min=7.25e16, nu_max=2.4e18, num_points=5)


def test_records_assembled_from_columns_equal_to_params():
    import torch

    t, nu, flux, err, ext = _point_data()
    lk = fitting.DeviceLikelihood(None, _template(), _NAMES, _LOG, t, nu, flux, err, ext_kernel=ext, device="cpu")
    s = _samples(37, 3)
    rec = lk.records(torch.as_tensor(lk.columns(s)))
    assert rec.dtype == torch.uint8 and rec.numel() == 37 * abi.PARAMS_DTYPE.itemsize
    assert rec.numpy().tobytes() == lk.to_params(s).tobytes()


class _PointerEngine:
    """Engine stand-in for CPU tensors: reads the records and A_V behind the pointers and writes a chi2 that depends on
    every model field and on A_V (not a likelihood: it only has to tell walkers apart)."""

    device = 0

    def __init__(self):
        self.calls = []

    def chi2_dev(self, d_params, n, points, bands, d_chi2, d_status=0, extinction=None, stream=0):
        P = np.frombuffer((C.c_char * (n * abi.PARAMS_DTYPE.itemsize)).from_address(d_params), dtype=abi.PARAMS_DTYPE)
        av = np.zeros(n) if extinction is None else np.ctypeslib.as_array((C.c_double * n).from_address(extinction[1]))
        out = np.ctypeslib.as_array((C.c_double * n).from_address(d_chi2))
        self.calls.append(n)
        ok = np.array([_previous_validate(p) is None for p in P])
        out[:] = np.where(ok, np.log10(P["E_iso"]) + P["Gamma0"] + P["theta_c"] + P["fwd"]["eps_e"] + av, np.inf)


_GLOO_WORKER = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, {root!r})
    import numpy as np, torch.distributed as dist
    from tests.test_device_likelihood import _NAMES, _LOG, _template, _samples, _point_data, _band, _PointerEngine
    from vegasafterglow_b200 import fitting
    rank = int(sys.argv[1])
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2)
    t, nu, flux, err, ext = _point_data()
    s = _samples(23, 5)
    lo, hi = np.min(s, axis=0), np.max(s, axis=0)
    hi[0] = np.quantile(s[:, 0], 0.8)  # some walkers out of bounds
    args = (_template(), _NAMES, _LOG, t, nu, flux, err)
    kw = dict(bands=[_band()], ext_kernel=ext, lower=lo, upper=hi, device="cpu")
    single = fitting.DeviceLikelihood(_PointerEngine(), *args, **kw)(s)
    eng = _PointerEngine()
    split = fitting.DeviceLikelihood(eng, *args, distributed=True, **kw)(s)
    assert np.array_equal(split, single), (split, single)
    assert np.isneginf(single).any() and np.isfinite(single).any()
    assert 0 < eng.calls[0] < 23
    dist.destroy_process_group()
    print("ok", rank)
""")


def test_device_likelihood_distributed_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER.format(root=ROOT, port=29317 + os.getpid() % 1000))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
             for r in range(2)]
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        assert "ok" in out


# ---- GPU tier ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host_caps(tmp_path_factory):
    """The host's caps_for (vag_pipeline.cuh), compiled from the header into a temporary library."""
    d = tmp_path_factory.mktemp("caps")
    src = d / "caps.cpp"
    src.write_text('#include "vag_pipeline.cuh"\n'
                   'extern "C" void caps_for_batch(const vag_params* p, size_t n, int* out) {\n'
                   '    const vag::Caps c = vag::caps_for(p, n); out[0] = c.theta; out[1] = c.phi; }\n')
    so = d / "caps.so"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I", os.path.join(ROOT, "vegasafterglow_b200", "csrc"),
                           str(src), "-o", str(so)])
    lib = C.CDLL(str(so))

    def caps(P):
        P = np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE)
        out = (C.c_int * 2)()
        lib.caps_for_batch(C.c_void_p(P.ctypes.data), C.c_size_t(P.size), out)
        return int(out[0]), int(out[1])

    return caps


def _dev(a):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a), device="cuda:0")


def _records(P):
    return _dev(np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE).view(np.uint8))


def _mixed_batch():
    P = np.concatenate([configs.random_draw(16, seed=11), configs.random_draw(16, seed=12, rvs=True),
                        configs.random_draw(16, seed=13, jet="gaussian", theta_obs_max=0.4)])
    return P[np.random.default_rng(5).permutation(P.size)]


def _chi2_pair(engine, P, pts, bands, ext=None, A_V=None):
    """(chi2, status, launches) of vag_chi2_ext on host buffers and of vag_chi2_dev on device buffers"""
    extinction = None if ext is None else (ext, A_V)
    want, want_st = engine.chi2(P, pts, bands, return_status=True, extinction=extinction)
    return (want, want_st, engine.last_launch_count()), _chi2_dev(engine, P, pts, bands, ext, A_V)


def _chi2_dev(engine, P, pts, bands, ext=None, A_V=None):
    """(chi2, status, launches) of vag_chi2_dev on device copies of the host arrays"""
    import torch

    keep = []
    dpts = None
    if pts is not None:
        keep += [_dev(a) for a in pts]
        dpts = (*(a.data_ptr() for a in keep), pts[0].size)
    dbands = []
    for b in bands:
        arrs = {k: _dev(b[k]) for k in ("t", "lnF_obs", "sigma_ln", "w")}
        keep.append(arrs)
        dbands.append(dict(b, n=b["t"].size, **{k: v.data_ptr() for k, v in arrs.items()}))
        assert b["t"].size
    dext = None
    if ext is not None:
        e, a = _dev(ext), _dev(A_V)
        keep += [e, a]
        dext = (e.data_ptr(), a.data_ptr())
    rec = _records(P)
    chi2 = torch.empty(P.size, dtype=torch.float64, device="cuda:0")
    st = torch.empty(P.size, dtype=torch.int32, device="cuda:0")
    engine.chi2_dev(rec.data_ptr(), P.size, dpts, dbands, chi2.data_ptr(), st.data_ptr(), extinction=dext)
    engine.synchronize()
    return chi2.cpu().numpy(), st.cpu().numpy(), engine.last_launch_count()


def _pts(seed=0):
    t, nu, flux, err, ext = _point_data(seed)
    return fitting.consolidate_data(t, nu, flux, err), ext


@pytest.mark.gpu
@pytest.mark.parametrize("series_mode", [0, 1, 2])
@pytest.mark.parametrize("terms", ["points", "bands", "points+bands", "points+A_V", "points+bands+A_V"])
def test_chi2_dev_equals_chi2_ext(engine, terms, series_mode):
    P = _mixed_batch()
    pts, ext = _pts()
    bands = [fitting.band_obs(**_band())] if "bands" in terms else []
    A_V = np.random.default_rng(2).uniform(0, 2, P.size) if "A_V" in terms else None
    try:
        engine.set_series_mode(series_mode)
        (want, want_st, n_host), (got, st, n_dev) = _chi2_pair(engine, P, pts if "points" in terms else None, bands,
                                                               ext if A_V is not None else None, A_V)
    finally:
        engine.set_series_mode(0)
    assert np.isfinite(want).all()
    assert np.array_equal(got, want) and np.array_equal(st, want_st)
    assert n_dev == n_host + PLANNING_LAUNCHES


@pytest.mark.gpu
def test_chi2_dev_arguments_are_checked_before_any_work(engine):
    import torch

    P = configs.random_draw(4, seed=1)
    t = np.array([1e3, 1e4, 1e5])
    keep = [_dev(a) for a in (t, np.full(t.size, 1e9), np.zeros(t.size), np.ones(t.size), np.ones(t.size), np.zeros(t.size),
                              np.zeros(P.size))]
    d_t, d_nu, d_lnF, d_sig, d_w, d_ext, d_av = (a.data_ptr() for a in keep)
    rec = _records(P)
    xb = dict(t=d_t, lnF_obs=d_lnF, sigma_ln=d_sig, w=d_w, n=t.size, nu_min=7.25e16, nu_max=2.4e18, num_nu=5)

    def call(n_points=t.size, ext=None, A_V=None, **band):
        b = dict(xb, **band)
        arr = (abi.BandObs * 1)(abi.BandObs(b["t"], b["lnF_obs"], b["sigma_ln"], b["w"], b["n"], b["nu_min"], b["nu_max"],
                                            b["num_nu"]))
        chi2 = torch.full((P.size,), 7.0, dtype=torch.float64, device="cuda:0")
        st = torch.full((P.size,), 99, dtype=torch.int32, device="cuda:0")
        rc = engine._lib.vag_chi2_dev(engine._h, rec.data_ptr(), P.size, d_t, d_nu, d_lnF, d_sig, d_w, ext, n_points, A_V,
                                      C.cast(arr, C.c_void_p), 1, chi2.data_ptr(), st.data_ptr(), None)
        engine.synchronize()
        return rc, bool((chi2.cpu().numpy() == 7.0).all() and (st.cpu().numpy() == 99).all())

    assert call() == (abi.VAG_OK, False)
    # word in the message -> arguments
    cases = {
        "band 0: empty (n = 0)": dict(n=0),
        "band 0: data arrays must not be NULL": dict(sigma_ln=None),
        "band 0: time array must not be NULL": dict(t=None),
        "band 0: nu_max": dict(nu_max=1e16),
        "band 0: num_nu": dict(num_nu=1),
        "both": dict(ext=d_ext),
        "extinction needs point data": dict(n_points=0, ext=d_ext, A_V=d_av),
    }
    for word, kw in cases.items():
        rc, untouched = call(**kw)
        assert rc == abi.VAG_ERR_INVALID, word
        assert untouched, word
        msg = engine._lib.vag_last_error().decode()
        assert word in msg, (word, msg)


@pytest.mark.gpu
def test_chi2_dev_across_the_pass_boundary(engine):
    n = 32768 + 64
    P = configs.random_draw(n, seed=21)
    t = np.array([1e3, 1e4, 1e5, 1e6])
    nu = np.array([1e9, 4.84e14, 1e17, 1e18])
    pts = fitting.consolidate_data(t, nu, 1e-27 * (t / 1e4) ** -1.0, 0.2e-27 * (t / 1e4) ** -1.0)
    ext = np.array([0.0, 1.3, 0.4, 0.05])
    A_V = np.array([0.2, 0.9, 1.6])[(np.arange(n) // 16) % 3]
    (want, want_st, _), (got, st, _) = _chi2_pair(engine, P, pts, [], ext, A_V)
    assert np.array_equal(got, want) and np.array_equal(st, want_st)


@pytest.mark.gpu
def test_flux_band_dev_equals_flux_band(engine):
    import torch

    P = _mixed_batch()
    t = np.logspace(3, 6, 9)
    want, want_st = engine.flux_band(P, t, 7.25e16, 2.4e18, 7, return_status=True)
    n_host = engine.last_launch_count()
    out = torch.empty((P.size, abi.NCOMP, t.size), dtype=torch.float64, device="cuda:0")
    st = torch.empty(P.size, dtype=torch.int32, device="cuda:0")
    rec, dt = _records(P), _dev(t)
    engine.flux_band_dev(rec.data_ptr(), P.size, dt.data_ptr(), t.size, 7.25e16, 2.4e18, 7, out.data_ptr(), st.data_ptr())
    engine.synchronize()
    assert np.array_equal(out.cpu().numpy(), want) and np.array_equal(st.cpu().numpy(), want_st)
    assert engine.last_launch_count() == n_host + PLANNING_LAUNCHES


@pytest.mark.gpu
def test_device_validation_and_capacities_match_the_host(engine, host_caps):
    import torch

    P = fuzz_records(100_000, seed=3)
    ok = torch.empty(P.size, dtype=torch.int32, device="cuda:0")
    rec = _records(P)
    caps = engine.validate_dev(rec.data_ptr(), P.size, ok.data_ptr())
    assert engine.last_launch_count() == 1
    want = engine.valid_mask(P)
    assert np.array_equal(ok.cpu().numpy().astype(bool), want)
    assert 0.2 * P.size < want.sum() < 0.8 * P.size
    assert caps == host_caps(P[want])
    for seed in range(4):  # smaller accepted sets
        sub = P[want][np.random.default_rng(seed).choice(int(want.sum()), 64, replace=False)]
        rec = _records(sub)
        assert engine.validate_dev(rec.data_ptr(), sub.size, ok.data_ptr()) == host_caps(sub)


# Below 2368 (model x shock) CTAs (148 SMs) k_eats splits the rows of a model into partial sums whose number depends on the
# batch size (vag_b200.cu run_flux_pass), and a different split rounds differently.  A batch with its rejected records
# removed is smaller than the batch that runs them as stand-ins, so comparisons between the two use batches above that
# size, where neither is split.
EATS_UNSPLIT_MODELS = 1184  # FS + RS batches: 2 shocks per model


def _large_mixed_batch():
    P = np.concatenate([configs.random_draw(704, seed=31), configs.random_draw(704, seed=32, rvs=True),
                        configs.random_draw(192, seed=33, jet="gaussian", theta_obs_max=0.4)])
    return P[np.random.default_rng(6).permutation(P.size)]


def _with_rejected(P, every=5):
    Q = P.copy()
    bad = np.zeros(P.size, dtype=bool)
    bad[::every] = True
    faults = [("Gamma0", 1.0), ("theta_c", 0.0), ("E_iso", np.nan), ("n_ism", -1.0), ("theta_c", np.inf)]
    for k, i in enumerate(np.nonzero(bad)[0]):
        name, v = faults[k % len(faults)]
        Q[name][i] = v
    return Q, bad


@pytest.mark.gpu
@pytest.mark.parametrize("series_mode", [1, 2])
def test_rejected_walkers(engine, series_mode):
    import torch

    P, bad = _with_rejected(_large_mixed_batch())
    assert not engine.valid_mask(P)[bad].any() and engine.valid_mask(P)[~bad].all()
    assert (~bad).sum() >= EATS_UNSPLIT_MODELS
    pts, ext = _pts(1)
    bands = [fitting.band_obs(**_band())]
    A_V = np.random.default_rng(4).uniform(0, 2, P.size)
    try:
        engine.set_series_mode(series_mode)  # mode 0 chooses by the batch's longest lattice, stand-ins included
        got, st, _ = _chi2_dev(engine, P, pts, bands, ext, A_V)  # the host path raises on the rejected records
        want, want_st = engine.chi2(P[~bad], pts, bands, return_status=True, extinction=(ext, A_V[~bad]))
        t = np.logspace(3, 6, 5)
        fb = torch.empty((P.size, abi.NCOMP, t.size), dtype=torch.float64, device="cuda:0")
        rec, dt = _records(P), _dev(t)
        engine.flux_band_dev(rec.data_ptr(), P.size, dt.data_ptr(), t.size, 1e14, 1e15, 5, fb.data_ptr())
        engine.synchronize()
        fb = fb.cpu().numpy()
        want_fb = engine.flux_band(P[~bad], t, 1e14, 1e15, 5)
    finally:
        engine.set_series_mode(0)
    assert np.isposinf(got[bad]).all() and (st[bad] == abi.ST_INVALID).all()
    assert np.array_equal(got[~bad], want) and np.array_equal(st[~bad], want_st)
    assert np.isnan(fb[bad]).all() and np.array_equal(fb[~bad], want_fb)


@pytest.mark.gpu
def test_walker_beyond_the_default_capacity(engine, host_caps):
    import torch

    # 20 theta nodes per degree over the ~25 degrees where the Gaussian jet's Lorentz factor stays above the cut
    p = configs.make(jet="gaussian", theta_c=0.1, Gamma0=800.0, resolutions=(0.06, 20.0, 6.0))
    t = np.logspace(3, 6, 8)
    d = engine.details(p, t[0], t[-1])
    assert int(d["info"]["n_theta"]) > 384 and host_caps(p)[0] > 384
    pts = fitting.consolidate_data(t, np.full(t.size, 1e9), 1e-27 * (t / 1e4) ** -1.0, 0.2e-27 * (t / 1e4) ** -1.0)
    P = np.concatenate([p, configs.random_draw(3, seed=1)])
    dp, chi2, st = _records(P), torch.empty(P.size, dtype=torch.float64, device="cuda:0"), torch.empty(P.size, dtype=torch.int32, device="cuda:0")
    dpts = [_dev(a) for a in pts]
    engine.chi2_series_dev(dp.data_ptr(), P.size, *(a.data_ptr() for a in dpts), t.size, chi2.data_ptr(), st.data_ptr())
    engine.synchronize()
    assert st.cpu().numpy()[0] & abi.ST_CAPACITY
    (want, want_st, _), (got, gst, _) = _chi2_pair(engine, P, pts, [])
    assert not want_st[0] & abi.ST_CAPACITY and np.isfinite(want[0])
    assert np.array_equal(got, want) and np.array_equal(gst, want_st)


@pytest.mark.gpu
def test_device_likelihood_equals_batched_likelihood(engine):
    t, nu, flux, err, ext = _point_data(2)
    s = _samples(2048, 9)
    s[:, 8] = 0.0  # on axis
    lo, hi = np.min(s, axis=0), np.max(s, axis=0)
    hi[1] = np.quantile(s[:, 1], 0.9)  # out-of-bounds walkers
    assert (s[:, 4] > 0).any()  # eps_e = 10^s > 1: walkers the constructors reject, inside the bounds
    args = (_template(), _NAMES, _LOG, t, nu, flux, err)
    kw = dict(bands=[_band()], ext_kernel=ext, lower=lo, upper=hi, log_prior=lambda x: -0.5 * x[:, 2])
    try:
        engine.set_series_mode(1)  # the batches differ by the rejected walkers: fix the series evaluation
        want = fitting.BatchedLikelihood(engine, *args, **kw)(s)
        got = fitting.DeviceLikelihood(engine, *args, **kw)(s)
    finally:
        engine.set_series_mode(0)
    assert np.isneginf(want).sum() > 200 and np.isfinite(want).sum() >= EATS_UNSPLIT_MODELS
    assert np.array_equal(got, want)
