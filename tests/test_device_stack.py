"""Stacked fits on device buffers: vag_chi2_multi_bands_dev, Engine.chi2_multi_bands_dev and fitting.DeviceLikelihoodStack.

GPU tier, bit for bit: the planned ragged call against vag_chi2_multi_bands on the same valid batch (points, bands and
both, with and without A_V, SSC models, series modes 0 / 1 / 2); rejected records (+inf, VAG_ST_INVALID; the accepted
ones against the host call on the accepted subset, a fit with every record rejected, a batch with none accepted); the
32768-model pass boundary with rejected records on both sides; the launch formula of the header; argument checks before
any work; a call on a non-default torch stream; DeviceLikelihoodStack against BandLikelihoodStack and against each
DeviceLikelihood alone; an NCCL world-2 stack (two GPUs).
CPU tier: DeviceLikelihoodStack with a pointer engine on CPU tensors (one call, record bytes, sets / ext_k / A_V against
BandLikelihoodStack's, the split back per fit, the ValueError cases) and under gloo with two ranks.
"""
import ctypes as C
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from tests.test_device_likelihood import _previous_validate, _with_rejected
from tests.test_multi_band import XRAY, _band, _chi2_batch, _datasets
from tests.test_multi_dataset import _LOG, _NAMES, UNSPLIT_MODELS, _raw_points, _samples, _with_mode
from vegasafterglow_b200 import abi, configs, fitting
from vegasafterglow_b200.engine import Engine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLANNING_LAUNCHES = 2  # k_plan, k_reject
BAND_GATHER_LAUNCHES = 1  # k_gather_bands, when an accepted model has a band


# ---- fits shared by both tiers ------------------------------------------------------------------------------------------
def _raw_band(t, nu_min, nu_max, num, seed):
    b = _band(t, nu_min, nu_max, num, seed)
    return dict(t=b["t"], flux=np.exp(b["lnF_obs"]), err=np.exp(b["lnF_obs"]) * b["sigma_ln"], nu_min=nu_min, nu_max=nu_max,
                num_points=num)


def _fit_specs(gpu):
    """Four fits: tophat FS with points, an X-ray band and A_V; a Gaussian FS+RS fit with two bands only that names A_V
    (ignored without points); tophat FS with points and a radio band, no A_V; tophat FS with points only and A_V."""
    specs = [(configs.make(lumi_dist=1e28, z=0.3), True, _raw_points(1), [_raw_band(np.logspace(3, 5.5, 8), *XRAY, 5, 1)]),
             (configs.make(jet="gaussian", rvs=(0.1, 0.01, 2.3), lumi_dist=1e28, z=0.3, theta_obs=0.05), True, None,
              [_raw_band(np.logspace(3.5, 6, 6), *XRAY, 5, 2), _raw_band(np.logspace(3, 5, 5), 4e14, 7.5e14, 3, 3)]),
             (configs.make(lumi_dist=3e27, z=0.1), False, _raw_points(3, 12, (1e9, 5e9, 4.84e14, 1e17)),
              [_raw_band(np.logspace(4, 6, 4), 1e9, 5e9, 2, 4)]),
             (configs.make(lumi_dist=2e28, z=0.2), True, _raw_points(5, 6, (4.84e14, 1e18)), [])]
    for tmpl, *_ in specs:
        if gpu:
            tmpl["t_resol"] = 3.0
    return specs


def _fits(engine, n_walkers, cls, gpu=True, **kw):
    """The fits of _fit_specs as ``cls`` (BatchedLikelihood or DeviceLikelihood) and their samples: out-of-bounds walkers
    and walkers the constructors reject (eps_e = 10^s > 1) in every fit."""
    fits, samples = [], []
    for k, (tmpl, av, pts, bands) in enumerate(_fit_specs(gpu)):
        s = _samples(n_walkers, 80 + k, av)
        lo, hi = np.min(s, axis=0), np.max(s, axis=0)
        hi[1] = np.quantile(s[:, 1], 0.9)
        names, log = _NAMES + (["A_V"] if av else []), _LOG + ([False] if av else [])
        t, nu, flux, err, ext = pts if pts is not None else (np.zeros(0),) * 5
        fits.append(cls(engine, tmpl, names, log, t, nu, flux, err, lower=lo, upper=hi,
                        log_prior=lambda x, k=k: -0.5 * k * x[:, 2], bands=bands, ext_kernel=ext if av else None, **kw))
        samples.append(s)
    return fits, samples


# ---- CPU tier: a pointer engine on CPU tensors ------------------------------------------------------------------------
def _arr(ptr, n, ctype=C.c_double):
    return np.ctypeslib.as_array((ctype * n).from_address(ptr)).copy() if n else np.zeros(0)


def _stand_in(p, lnF, ext, av, band_lnF):
    """Not a likelihood: a value that depends on the model record, its points, its bands (in order) and A_V."""
    v = np.log10(p["E_iso"]) + p["Gamma0"] + p["theta_c"] + p["fwd"]["eps_e"] + lnF.sum() + av * (1.0 + ext.sum())
    for i, b in enumerate(band_lnF):
        v = v + (i + 1) * b.sum()
    return v if _previous_validate(p) is None else np.inf


class _PointerEngine:
    """Engine stand-in that reads every array behind the pointers of chi2_dev / chi2_multi_bands_dev and writes
    _stand_in's value per model; it records what the stack passes."""

    device = 0

    def __init__(self):
        self.calls = []

    @staticmethod
    def _records(d_params, n):
        return np.frombuffer((C.c_char * (n * abi.PARAMS_DTYPE.itemsize)).from_address(d_params), dtype=abi.PARAMS_DTYPE)

    def chi2_dev(self, d_params, n, points, bands, d_chi2, d_status=0, extinction=None, stream=0):
        P = self._records(d_params, n)
        n_pt = 0 if points is None else points[5]
        lnF = np.zeros(0) if points is None else _arr(points[2], n_pt)
        ext = np.zeros(n_pt) if extinction is None else _arr(extinction[0], n_pt)
        av = np.zeros(n) if extinction is None else _arr(extinction[1], n)
        blnF = [_arr(b["lnF_obs"], b["n"]) for b in bands]
        out = np.ctypeslib.as_array((C.c_double * n).from_address(d_chi2))
        out[:] = [_stand_in(P[m], lnF, ext, av[m], blnF) for m in range(n)]

    def chi2_multi_bands_dev(self, d_params, n, dataset_of, sets, points, bands, d_chi2, d_status=0, extinction=None,
                             stream=0):
        P = self._records(d_params, n)
        n_pt = 0 if points is None else points[5]
        lnF = np.zeros(n_pt) if points is None else _arr(points[2], n_pt)
        ext = None if extinction is None else _arr(extinction[0], n_pt)
        av = np.zeros(n) if extinction is None else _arr(extinction[1], n)
        blnF = [_arr(b["lnF_obs"], b["n"]) for b in bands]
        sets = [(s.offset, s.n, s.band0, s.n_bands) for s in sets]
        self.calls.append(dict(rec=P.tobytes(), dataset_of=np.array(dataset_of), sets=sets, ext=ext, A_V=av, stream=stream,
                               band_t=[_arr(b["t"], b["n"]) for b in bands], points=[_arr(p, n_pt) for p in points[:5]]
                               if points is not None else None))
        out = np.ctypeslib.as_array((C.c_double * n).from_address(d_chi2))
        for m in range(n):
            o, k, b0, nb = sets[dataset_of[m]]
            e = np.zeros(k) if ext is None else ext[o:o + k]
            out[m] = _stand_in(P[m], lnF[o:o + k], e, av[m] if k else 0.0, blnF[b0:b0 + nb])


class _RecordingEngine:
    """What BandLikelihoodStack passes to chi2_multi_bands (host arrays)."""

    device = 0

    def __init__(self):
        self.calls = []

    def chi2_multi_bands(self, P, datasets, bands, dataset_of, extinction=None):
        self.calls.append(dict(P=P.copy(), datasets=datasets, bands=bands, dataset_of=np.array(dataset_of),
                               extinction=extinction))
        return np.zeros(P.size)


def _in_bounds(fits, samples):
    return [s[lk._in_bounds(s)] for lk, s in zip(fits, samples)]


def test_device_stack_is_one_call_with_the_records_and_data_of_each_fit():
    eng = _PointerEngine()
    fits, samples = _fits(eng, 40, fitting.DeviceLikelihood, gpu=False, device="cpu")
    stack = fitting.DeviceLikelihoodStack(fits)
    got = stack(samples)
    assert len(eng.calls) == 1
    call = eng.calls[0]
    inb = _in_bounds(fits, samples)
    counts = [s.shape[0] for s in inb]
    assert np.array_equal(call["dataset_of"], np.repeat(np.arange(len(fits)), counts))
    assert call["rec"] == np.concatenate([lk.to_params(s) for lk, s in zip(fits, inb)]).tobytes()
    assert call["stream"] == 0  # CPU tensors: no CUDA stream
    # what BandLikelihoodStack passes for the same fits, restricted to the walkers it keeps (the valid ones)
    rec = _RecordingEngine()
    host_fits, _ = _fits(rec, 40, fitting.BatchedLikelihood, gpu=False)
    fitting.BandLikelihoodStack(host_fits)(samples)
    want = rec.calls[0]
    valid = np.concatenate([Engine.valid_mask(lk.to_params(s)) for lk, s in zip(fits, inb)])
    assert np.array_equal(call["dataset_of"][valid], want["dataset_of"])
    off = b0 = 0
    for k, (d, bl) in enumerate(zip(want["datasets"], want["bands"])):
        n = 0 if d is None else d[0].size
        assert call["sets"][k] == (off, n, b0, len(bl))
        if d is not None:
            for a, b in zip(call["points"], d):
                assert np.array_equal(a[off:off + n], b)
        for j, b in enumerate(bl):
            assert np.array_equal(call["band_t"][b0 + j], b["t"])
        off, b0 = off + n, b0 + len(bl)
    ext, A_V = want["extinction"]
    assert np.array_equal(call["ext"], np.concatenate([e for e in ext if e is not None]))
    assert not call["ext"][call["sets"][2][0]:call["sets"][2][0] + call["sets"][2][1]].any()  # fit 2: no A_V -> zeros
    assert np.array_equal(call["A_V"][valid], A_V)
    assert not call["A_V"][np.isin(call["dataset_of"], [1, 2])].any()  # bands only / no A_V: 0
    # the split back per fit and the -inf rules: each fit alone
    want_alone = [lk(s) for lk, s in zip(fits, samples)]
    for g, w in zip(got, want_alone):
        assert np.array_equal(g, w)
        assert np.isneginf(w).any() and np.isfinite(w).any()
    assert (~valid).any()  # rejected walkers were present


def test_device_stack_rejects_what_it_cannot_stack():
    eng = _PointerEngine()
    t, nu, flux, err, _ = _raw_points(1)
    args = (configs.make(), _NAMES, _LOG, t, nu, flux, err)
    dev = fitting.DeviceLikelihood(eng, *args, device="cpu")
    with pytest.raises(ValueError, match="likelihood 1: DeviceLikelihoodStack stacks DeviceLikelihood"):
        fitting.DeviceLikelihoodStack([dev, fitting.BatchedLikelihood(eng, *args)])
    with pytest.raises(ValueError, match="engine and device"):
        fitting.DeviceLikelihoodStack([dev, fitting.DeviceLikelihood(_PointerEngine(), *args, device="cpu")])
    with pytest.raises(ValueError, match="engine and device"):
        fitting.DeviceLikelihoodStack([dev, fitting.DeviceLikelihood(eng, *args, device="meta")])
    with pytest.raises(ValueError, match="distributed=True"):
        fitting.DeviceLikelihoodStack([dev, fitting.DeviceLikelihood(eng, *args, device="cpu", distributed=True)])
    with pytest.raises(ValueError, match="at least one"):
        fitting.DeviceLikelihoodStack([])


_GLOO_WORKER = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, {root!r})
    import numpy as np, torch.distributed as dist
    from tests.test_device_stack import _PointerEngine, _fits
    from vegasafterglow_b200 import fitting
    rank = int(sys.argv[1])
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2)
    eng = _PointerEngine()
    fits, samples = _fits(eng, 23, fitting.DeviceLikelihood, gpu=False, device="cpu")
    single = fitting.DeviceLikelihoodStack(fits)(samples)
    split = fitting.DeviceLikelihoodStack(fits, distributed=True)(samples)
    for a, b in zip(split, single):
        assert np.array_equal(a, b), (a, b)
    n = sum(int(lk._in_bounds(s).size) for lk, s in zip(fits, samples))
    mine = eng.calls[1]["dataset_of"].size
    assert 0 < mine < n, (mine, n)
    print("ok", rank, mine, n)
    dist.destroy_process_group()
""")


def _run_world2(script_text, tmp_path, env=None):
    script = tmp_path / "worker.py"
    script.write_text(script_text)
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                              env=env) for r in range(2)]
    outs = []
    for p in procs:
        out, err = p.communicate(timeout=600)
        assert p.returncode == 0, err[-3000:]
        assert "ok" in out
        outs.append(out)
    return outs


def test_device_stack_distributed_gloo_world2(tmp_path):
    outs = _run_world2(_GLOO_WORKER.format(root=ROOT, port=29417 + os.getpid() % 1000), tmp_path)
    shares = [int(o.split()[2]) for o in outs]
    n = int(outs[0].split()[3])
    assert sum(shares) == n


# ---- GPU tier -----------------------------------------------------------------------------------------------------------
def _dev(a):
    import torch

    return torch.as_tensor(np.ascontiguousarray(a), device="cuda:0")


def _layout(pts, bands):
    """The host call's concatenation (Engine.chi2_multi_bands): concatenated point columns, sets, flat bands."""
    cols, n_pts = [[] for _ in range(5)], []
    for p in pts:
        n_pts.append(0 if p is None else p[0].size)
        for c, a in zip(cols, p or ()):
            c.append(np.asarray(a, dtype=np.float64))
    cat = [np.concatenate(c) if c else np.zeros(0) for c in cols]
    off = np.concatenate([[0], np.cumsum(n_pts)]).astype(np.int64)
    b0 = np.concatenate([[0], np.cumsum([len(bl) for bl in bands])]).astype(np.int64)
    sets = [(int(off[d]), int(n_pts[d]), int(b0[d]), len(bands[d])) for d in range(len(pts))]
    return cat, sets, [b for bl in bands for b in bl]


def _dev_call(engine, P, pts, bands, ds, ext=None, A_V=None, stream=None, rec=None):
    """(chi2, status, launches) of vag_chi2_multi_bands_dev on device copies of the host call's arrays"""
    import torch

    cat, sets, flat = _layout(pts, bands)
    keep = [_dev(a) for a in cat]
    points = (*(a.data_ptr() for a in keep), cat[0].size) if cat[0].size else None
    dbands = []
    for b in flat:
        arrs = {k: _dev(b[k]) for k in ("t", "lnF_obs", "sigma_ln", "w")}
        keep.append(arrs)
        dbands.append(dict(b, n=b["t"].size, **{k: v.data_ptr() for k, v in arrs.items()}))
    extinction = None
    if ext is not None:
        e = np.concatenate([np.zeros(0) if x is None else x for x in ext])
        de, da = _dev(e), _dev(np.asarray(A_V, dtype=np.float64))
        keep += [de, da]
        extinction = (de.data_ptr(), da.data_ptr())
    if rec is None:
        rec = _dev(np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE).view(np.uint8))
    chi2 = torch.full((P.size,), 7.0, dtype=torch.float64, device="cuda:0")
    st = torch.full((P.size,), 99, dtype=torch.int32, device="cuda:0")
    engine.chi2_multi_bands_dev(rec.data_ptr(), P.size, ds, sets, points, dbands, chi2.data_ptr(), st.data_ptr(),
                                extinction=extinction, stream=stream or 0)
    engine.synchronize()
    torch.cuda.synchronize()
    return chi2.cpu().numpy(), st.cpu().numpy(), engine.last_launch_count()


def _ext_av(P, pts, seed=3):
    rng = np.random.default_rng(seed)
    return [None if p is None else rng.uniform(0.0, 1.7, p[0].size) for p in pts], rng.uniform(0.0, 2.0, P.size)


@pytest.mark.gpu
@pytest.mark.parametrize("series_mode", [0, 1, 2])
@pytest.mark.parametrize("extinction", [False, True])
def test_dev_equals_host_call_on_a_valid_batch(engine, series_mode, extinction):
    P, ds = _chi2_batch(10)  # sets 0 points + bands, 1 bands only, 2 and 3 points only; SSC+KN models among them
    assert P["fwd"]["ssc"].any()
    pts, bands = _datasets(0)
    ext, A_V = _ext_av(P, pts) if extinction else (None, None)
    kw = dict(extinction=(ext, A_V)) if extinction else {}

    def both():
        want = engine.chi2_multi_bands(P, pts, bands, ds, return_status=True, **kw)
        n_host = engine.last_launch_count()
        return want, n_host, _dev_call(engine, P, pts, bands, ds, ext, A_V)

    (want, want_st), n_host, (got, st, n_dev) = _with_mode(engine, series_mode, both)
    assert np.isfinite(want).all()
    assert np.array_equal(got, want) and np.array_equal(st, want_st)
    assert n_dev == n_host + PLANNING_LAUNCHES + BAND_GATHER_LAUNCHES


@pytest.mark.gpu
@pytest.mark.parametrize("series_mode", [0, 1, 2])
def test_rejected_records_are_left_out(engine, series_mode):
    P, ds = _chi2_batch(12)
    P, bad = _with_rejected(P)
    bad |= ds == 3  # every record of the fit on set 3 rejected as well
    P["Gamma0"][ds == 3] = 0.5
    assert not Engine.valid_mask(P)[bad].any() and Engine.valid_mask(P)[~bad].all()
    pts, bands = _datasets(1)
    ext, A_V = _ext_av(P, pts, 4)

    def both():
        got = _dev_call(engine, P, pts, bands, ds, ext, A_V)
        want = engine.chi2_multi_bands(P[~bad], pts, bands, ds[~bad], extinction=(ext, A_V[~bad]), return_status=True)
        return got, want, engine.last_launch_count()

    (got, st, n_dev), (want, want_st), n_host = _with_mode(engine, series_mode, both)
    assert np.isposinf(got[bad]).all() and (st[bad] == abi.ST_INVALID).all()
    assert np.array_equal(got[~bad], want) and np.array_equal(st[~bad], want_st)
    assert n_dev == n_host + PLANNING_LAUNCHES + BAND_GATHER_LAUNCHES
    # the rejected records' contents do not matter
    Q = P.copy()
    Q["E_iso"][bad] = 1e49
    Q["theta_c"][bad] = np.nan
    got2, st2, _ = _with_mode(engine, series_mode, lambda: _dev_call(engine, Q, pts, bands, ds, ext, A_V))
    assert np.array_equal(got2, got) and np.array_equal(st2, st)
    # none accepted: k_plan and k_reject only
    Z = P.copy()
    Z["Gamma0"] = 1.0
    got, st, n = _dev_call(engine, Z, pts, bands, ds, ext, A_V)
    assert np.isposinf(got).all() and (st == abi.ST_INVALID).all() and n == PLANNING_LAUNCHES


@pytest.mark.gpu
def test_pass_boundary_with_rejected_records(engine):
    n = 42000
    P, bad = _with_rejected(configs.random_draw(n, seed=23))  # every 5th rejected: 33600 accepted
    acc = np.nonzero(~bad)[0]
    assert acc.size > 32768 and bad[acc[32768] - 5:acc[32768]].any() and bad[acc[32768]:acc[32768] + 5].any()
    pts = [fitting.consolidate_data(np.array([1e3, 1e4, 1e5, 1e6]), np.array([1e9, 4.84e14, 1e17, 1e18]),
                                    1e-27 * np.array([10.0, 1.0, 0.1, 0.01]), 2e-28 * np.array([10.0, 1.0, 0.1, 0.01]))]
    ds = np.zeros(n, dtype=np.int32)
    ext = [np.array([0.0, 1.3, 0.4, 0.05])]
    A_V = np.array([0.2, 0.9, 1.6])[(np.arange(n) // 16) % 3]
    got, st, _ = _dev_call(engine, P, pts, [[]], ds, ext, A_V)
    want, want_st = engine.chi2_multi_bands(P[~bad], pts, [[]], ds[~bad], extinction=(ext, A_V[~bad]), return_status=True)
    assert np.isposinf(got[bad]).all() and (st[bad] == abi.ST_INVALID).all()
    assert np.array_equal(got[~bad], want) and np.array_equal(st[~bad], want_st)


@pytest.mark.gpu
def test_launch_count_follows_the_header(engine):
    P = configs.random_draw(96, seed=41, rvs=True)

    def count(n_fits, n_bands, with_points=True):
        pts = [_datasets(k)[0][0] if with_points else None for k in range(n_fits)]
        bands = [[_band(np.logspace(3 + 0.1 * j, 5.5, 6), *XRAY, 5, 10 * k + j) for j in range(n_bands)]
                 for k in range(n_fits)]
        ds = (np.arange(P.size) % n_fits).astype(np.int32)
        engine.chi2_multi_bands(P, pts, bands, ds)
        n_host = engine.last_launch_count()
        _, _, n_dev = _dev_call(engine, P, pts, bands, ds)
        assert n_dev == n_host + PLANNING_LAUNCHES + (BAND_GATHER_LAUNCHES if n_bands else 0), (n_fits, n_bands)
        return n_dev

    assert count(2, 1) == count(6, 1) == count(2, 4) == count(6, 4)
    assert count(2, 0) == count(6, 0)
    assert count(2, 1, with_points=False) == count(6, 4, with_points=False)


def _raw_dev(engine, P, ds, sets, t, n_points=None, bands=None, ext=None, A_V=None, null_points=False, null_band_t=False):
    """vag_chi2_multi_bands_dev on device arrays with sentinel outputs -> (return code, outputs untouched)"""
    import torch

    ds = np.ascontiguousarray(ds, dtype=np.int32)
    arr = (abi.MultiSet * max(len(sets), 1))(*[abi.MultiSet(*s) for s in sets])
    n = t.size if n_points is None else n_points
    keep = [_dev(a) for a in (t, np.full(t.size, 1e9), np.zeros(t.size), np.ones(t.size), np.ones(t.size))]
    rec = _dev(np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE).view(np.uint8))
    bands = bands or []
    barr = (abi.BandObs * max(len(bands), 1))()
    for i, b in enumerate(bands):
        bt = np.asarray(b["t"], dtype=np.float64)
        a = [_dev(bt if bt.size else np.zeros(1)), _dev(np.zeros(max(bt.size, 1))), _dev(np.ones(max(bt.size, 1))),
             _dev(np.ones(max(bt.size, 1)))]
        keep += a
        ptrs = [x.data_ptr() for x in a]
        if null_band_t and i == 1:
            ptrs[0] = None
        barr[i] = abi.BandObs(*ptrs, bt.size, b["nu_min"], b["nu_max"], b["num_nu"])
    de = da = None
    if ext is not None:
        keep.append(_dev(ext))
        de = keep[-1].data_ptr()
    if A_V is not None:
        keep.append(_dev(A_V))
        da = keep[-1].data_ptr()
    chi2 = torch.full((P.size,), 7.0, dtype=torch.float64, device="cuda:0")
    st = torch.full((P.size,), 99, dtype=torch.int32, device="cuda:0")
    ptrs = [None] * 5 if null_points else [a.data_ptr() for a in keep[:5]]
    rc = engine._lib.vag_chi2_multi_bands_dev(engine._h, rec.data_ptr(), P.size, ds.ctypes.data,
                                              C.cast(arr, C.c_void_p) if sets else None, len(sets), *ptrs, de, n, da,
                                              C.cast(barr, C.c_void_p) if bands else None, len(bands), chi2.data_ptr(),
                                              st.data_ptr(), None)
    engine.synchronize()
    return rc, bool((chi2.cpu().numpy() == 7.0).all() and (st.cpu().numpy() == 99).all())


@pytest.mark.gpu
def test_arguments_are_checked_before_any_work(engine):
    P = configs.random_draw(4, seed=1)
    t = np.array([1e3, 1e4, 1e5, 2e3, 2e4, 2e5])
    xb = dict(t=[1e3, 1e4], nu_min=XRAY[0], nu_max=XRAY[1], num_nu=5)
    ok_bands = [xb, dict(xb, num_nu=3)]
    ok_sets = [(0, 3, 0, 1), (3, 3, 0, 0), (0, 0, 1, 1)]
    ds = np.array([0, 1, 2, 0])
    assert _raw_dev(engine, P, ds, ok_sets, t, bands=ok_bands) == (abi.VAG_OK, False)
    ext = np.zeros(t.size)
    cases = {
        "data set 2: no data": dict(sets=[(0, 3, 0, 1), (3, 3, 0, 0), (0, 0, 1, 0)]),
        "data set 1: points [": dict(sets=[(0, 3, 0, 1), (4, 3, 0, 0), (0, 0, 1, 1)]),
        "data set 2: bands [": dict(sets=[(0, 3, 0, 1), (3, 3, 0, 0), (0, 0, 1, 2)]),
        "band 1: empty (n = 0)": dict(bands=[xb, dict(xb, t=[])]),
        "band 1: time array must not be NULL": dict(null_band_t=True),
        "band 1: num_nu": dict(bands=[xb, dict(xb, num_nu=1)]),
        "band 1: nu_max": dict(bands=[xb, dict(xb, nu_max=1e16)]),
        "model 2: dataset_of": dict(ds=np.array([0, 1, 3, 0])),
        "both": dict(ext=ext),
        "extinction needs point data": dict(sets=[(0, 0, 0, 1)], ds=np.zeros(4), n_points=0, ext=ext, A_V=np.zeros(4)),
        "point data arrays": dict(null_points=True),
        "no data sets": dict(sets=[]),
    }
    for word, kw in cases.items():
        args = dict(P=P, ds=ds, sets=ok_sets, t=t, bands=ok_bands)
        args.update(kw)
        rc, untouched = _raw_dev(engine, args.pop("P"), args.pop("ds"), args.pop("sets"), args.pop("t"), **args)
        assert rc == abi.VAG_ERR_INVALID, word
        assert untouched, word
        msg = engine._lib.vag_last_error().decode()
        assert word in msg, (word, msg)
    # no models: nothing to do
    assert _raw_dev(engine, P[:0], ds[:0], ok_sets, t, bands=ok_bands) == (abi.VAG_OK, True)
    # a failed call leaves the engine usable
    pts, bands = _datasets(2)
    Q, dq = _chi2_batch(30)
    Q, dq = Q[:200], dq[:200]
    want = engine.chi2_multi_bands(Q, pts, bands, dq)
    got, _, _ = _dev_call(engine, Q, pts, bands, dq)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_call_on_a_non_default_stream(engine):
    import torch

    P, ds = _chi2_batch(40)
    pts, bands = _datasets(3)
    ext, A_V = _ext_av(P, pts, 5)
    want = engine.chi2_multi_bands(P, pts, bands, ds, extinction=(ext, A_V))
    src = _dev(np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE).view(np.uint8))
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device="cuda:0")
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)  # keeps the stream busy, so a call not ordered after the copy below would see zeros
        rec = torch.zeros_like(src)
        rec.copy_(src)
        got, _, _ = _dev_call(engine, P, pts, bands, ds, ext, A_V, stream=s.cuda_stream, rec=rec)
    assert np.array_equal(got, want)


def _stack_fits(engine, n_walkers):
    dev, samples = _fits(engine, n_walkers, fitting.DeviceLikelihood)
    host, _ = _fits(engine, n_walkers, fitting.BatchedLikelihood)
    return dev, host, samples


@pytest.mark.gpu
@pytest.mark.parametrize("series_mode", [0, 1, 2])
def test_device_stack_equals_band_likelihood_stack(engine, series_mode):
    dev, host, samples = _stack_fits(engine, 300)
    got, want = _with_mode(engine, series_mode, lambda: (fitting.DeviceLikelihoodStack(dev)(samples),
                                                         fitting.BandLikelihoodStack(host)(samples)))
    for k, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), k
        assert np.isneginf(w).sum() > 10 and np.isfinite(w).sum() > 100
    # rejected walkers among the in-bounds ones
    assert any((~Engine.valid_mask(lk.to_params(s[lk._in_bounds(s)]))).any() for lk, s in zip(dev, samples))


@pytest.mark.gpu
def test_device_stack_equals_each_device_likelihood_alone(engine):
    dev, _, samples = _stack_fits(engine, 2 * UNSPLIT_MODELS)
    want = _with_mode(engine, 1, lambda: [lk(s) for lk, s in zip(dev, samples)])
    got = _with_mode(engine, 1, lambda: fitting.DeviceLikelihoodStack(dev)(samples))
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
        assert np.isneginf(w).sum() > 100 and np.isfinite(w).sum() >= UNSPLIT_MODELS


_NCCL_WORKER = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, {root!r})
    import numpy as np, torch, torch.distributed as dist
    rank = int(sys.argv[1])
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=2)
    from tests.test_device_stack import _fits, _with_mode
    from vegasafterglow_b200 import fitting
    from vegasafterglow_b200.engine import Engine
    eng = Engine(rank)
    fits, samples = _fits(eng, {n}, fitting.DeviceLikelihood)
    split = _with_mode(eng, 1, lambda: fitting.DeviceLikelihoodStack(fits, distributed=True)(samples))
    if rank == 0:
        single = _with_mode(eng, 1, lambda: fitting.DeviceLikelihoodStack(fits)(samples))
        for a, b in zip(split, single):
            assert np.array_equal(a, b)
    dist.barrier()
    dist.destroy_process_group()
    print("ok", rank)
""")


@pytest.mark.gpu
def test_device_stack_nccl_world2(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    # each rank's share stays above 2368 (model x shock) CTAs, where k_eats does not split a model's rows
    _run_world2(_NCCL_WORKER.format(root=ROOT, port=29517 + os.getpid() % 1000, n=2 * UNSPLIT_MODELS), tmp_path)
