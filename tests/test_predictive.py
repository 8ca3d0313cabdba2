"""Posterior-predictive light curves of many fits in one call: a (t x nu) grid per model and exact quantiles across each
set's models on the GPU (vag_flux_density_grid_multi, vag_flux_quantiles_multi, Engine.flux_density_grid_multi /
flux_quantiles_multi, LikelihoodStack.flux_quantiles, BatchedLikelihood.flux_quantiles).

GPU tier: the per-model grid call equals each set's models on that set alone on a shuffled mixed batch, bit for bit, and
to rounding across the 32768-model pass boundary; its launches are one vag_flux_density_grid call's; every argument check
fails before any work; the quantiles equal numpy.quantile of that call's total plane bit for bit (sets of 1, 2, odd and
even size, one selected from global memory, one without models, models excluded by VAG_ST_ODE_FAIL500); the likelihood
stack's bands equal numpy on each fit's own flux_density_grid.
CPU tier: the selection and interpolation body of csrc/vag_quantile.cuh, compiled for the host, against numpy.quantile;
the vag_grid_set layout against the header; LikelihoodStack.flux_quantiles with a recording engine.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from vegasafterglow_b200 import abi, configs, fitting
from tests.test_multi_dataset import UNSPLIT_MODELS, _fits, _models, _padded

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "vegasafterglow_b200", "csrc")
BANDS = (0.16, 0.5, 0.84)
FAIL = abi.ST_ODE_FAIL500 | abi.ST_CAPACITY  # statuses whose models are not members of their set's quantiles


# ---- data ------------------------------------------------------------------------------------------------------------
UNUSED = 4


def _grids():
    """Six grids: one epoch; nine frequencies (two tiles of k_eats: across its 8-wide tile); an early window with one
    frequency; a late window disjoint from it with three; one no model uses; a radio-only one."""
    return [
        (np.array([3e4]), np.array([1e9, 4.84e14, 1e18])),
        (np.logspace(3, 6, 20), np.logspace(9, 18, 9)),
        (np.logspace(2, 4, 15), np.array([4.84e14])),
        (np.logspace(5, 7, 12), np.array([5e9, 1e14, 1e17])),
        (np.logspace(3, 5, 6), np.array([1e9, 1e18])),
        (np.logspace(3, 6, 10), np.array([1e9, 5e9])),
    ]


def _batch(seed=0):
    """(params, grids, dataset_of) of the mixed batch of test_multi_dataset; every grid but UNUSED has models, the SSC
    models on the radio-only grid and the nine-frequency one"""
    P, is_ssc = _models(seed=seed)
    # time lattices of <= ~25 nodes: the nine-frequency grid widens the batch's k_eats tile to 8, and a lattice over ~33
    # nodes would then stage 7 rows per pass where a narrower set's call alone stages 8 (vag.h, DESIGN.md 5)
    P["t_resol"] = 2.0
    grids = _grids()
    used = [d for d in range(len(grids)) if d != UNUSED]
    ds = np.asarray(used, dtype=np.int32)[np.random.default_rng(seed + 7).integers(0, len(used), P.size)]
    ssc_idx = np.nonzero(is_ssc)[0]
    ds[ssc_idx[::2]] = 5
    ds[ssc_idx[1::2]] = 1
    return P, grids, ds


def _numpy_bands(flux, st, ds, n_sets, q):
    """numpy.quantile over each set's members of the total planes of a flux_density_grid_multi result"""
    out, n_used = [], []
    for d in range(n_sets):
        members = [m for m in np.nonzero(ds == d)[0] if not st[m] & FAIL]
        n_used.append(len(members))
        if members:
            out.append(np.quantile(np.stack([flux[m][0] for m in members]), q, axis=0, method="linear"))
        else:
            out.append(None)
    return out, np.array(n_used)


# ---- GPU tier -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_grid_multi_equals_each_set_alone(engine):
    P, grids, ds = _batch()
    assert 2 * P.size >= UNSPLIT_MODELS  # FS+RS models in the batch: 2 shocks per model, no row split
    got, st = engine.flux_density_grid_multi(P, grids, ds, return_status=True)
    assert len(got) == P.size
    for d in np.unique(ds):
        idx = np.nonzero(ds == d)[0]
        f, q = engine.flux_density_grid(_padded(P[idx]), *grids[d], return_status=True)
        assert np.array_equal(st[idx], q[:idx.size]), d
        for j, m in enumerate(idx):
            assert got[m].shape == (abi.NCOMP, grids[d][1].size, grids[d][0].size)
            assert np.array_equal(got[m], f[j], equal_nan=True), (d, m)
    assert UNUSED not in ds


@pytest.mark.gpu
def test_grid_multi_pass_boundary(engine):
    n = 32768 + 64
    P = configs.random_draw(n, seed=21)
    grids = [(np.logspace(3, 6, 4), np.array([1e9, 1e17])), (np.logspace(4, 7, 3), np.array([4.84e14]))]
    ds = ((np.arange(n) // 16) % 2).astype(np.int32)
    assert ds[32767] != ds[32768]
    got = engine.flux_density_grid_multi(P, grids, ds)
    for d in (0, 1):
        idx = np.nonzero(ds == d)[0]
        want = engine.flux_density_grid(P[idx], *grids[d])
        f = np.stack([got[m] for m in idx])
        first = idx < 32768
        assert np.array_equal(f[first], want[first])
        # the second pass is a batch of 64 models, whose rows k_eats splits into partial sums: to rounding
        np.testing.assert_allclose(f[~first], want[~first], rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_grid_multi_launches_are_one_grid_calls(engine):
    P = configs.random_draw(64, seed=41, rvs=True)
    grids = _grids()
    engine.flux_density_grid(P, *grids[1])
    single = engine.last_launch_count()
    engine.flux_density_grid_multi(P, [grids[1]], np.zeros(P.size, dtype=np.int32))
    one = engine.last_launch_count()
    engine.flux_density_grid_multi(P, grids, (np.arange(P.size) % len(grids)).astype(np.int32))
    many = engine.last_launch_count()
    assert one == many == single
    engine.flux_quantiles_multi(P, grids, (np.arange(P.size) % len(grids)).astype(np.int32), BANDS)
    assert engine.last_launch_count() == many + 2


def _raw(engine, P, ds, sets, t, nu, q=None):
    """vag_flux_density_grid_multi (q None) or vag_flux_quantiles_multi on the given arrays with sentinel outputs ->
    (return code, outputs untouched)"""
    P = np.ascontiguousarray(P, dtype=abi.PARAMS_DTYPE)
    ds = np.ascontiguousarray(ds, dtype=np.int32)
    arr = (abi.GridSet * max(len(sets), 1))(*[abi.GridSet(*s) for s in sets])
    out = np.full(4096, 7.0)
    st = np.full(P.size, 99, dtype=np.int32)
    used = np.full(max(len(sets), 1), 99, dtype=np.int64)
    args = [engine._h, P.ctypes.data, P.size, ds.ctypes.data, C.cast(arr, C.c_void_p) if sets else None, len(sets),
            t.ctypes.data, t.size, nu.ctypes.data, nu.size]
    if q is None:
        rc = engine._lib.vag_flux_density_grid_multi(*args, out.ctypes.data, st.ctypes.data)
    else:
        q = np.ascontiguousarray(q, dtype=np.float64)
        rc = engine._lib.vag_flux_quantiles_multi(*args, q.ctypes.data if q.size else None, q.size, out.ctypes.data,
                                                  used.ctypes.data, st.ctypes.data)
    return rc, bool((out == 7.0).all() and (st == 99).all() and (used == 99).all())


@pytest.mark.gpu
def test_arguments_are_validated_before_any_work(engine):
    P = configs.random_draw(4, seed=1)
    t = np.array([1e3, 1e4, 1e5, 2e3, 2e4, 2e5])
    nu = np.array([1e9, 1e14, 1e17])
    ok_sets = [(0, 3, 0, 2), (3, 3, 2, 1)]
    ds = np.array([0, 1, 1, 0])
    assert _raw(engine, P, ds, ok_sets, t, nu)[0] == abi.VAG_OK
    assert _raw(engine, P, ds, ok_sets, t, nu, BANDS)[0] == abi.VAG_OK
    bad_t = t.copy()
    bad_t[5] = np.inf  # last of set 1: still ascending
    neg_t = t.copy()
    neg_t[3] = -1.0
    bad_nu = nu.copy()
    bad_nu[2] = 0.0
    bad_P = P.copy()
    bad_P["Gamma0"][2] = 1.0
    cases = {
        "dataset_of": dict(ds=np.array([0, 1, 2, 0])),
        "dataset_of ": dict(ds=np.array([0, -1, 1, 0])),
        "times": dict(sets=[(0, 3, 0, 2), (4, 3, 2, 1)]),
        "frequencies [": dict(sets=[(0, 3, 0, 2), (3, 3, 2, 2)]),
        "n_t = 0": dict(sets=[(0, 3, 0, 2), (3, 0, 2, 1)]),
        "n_nu = 0": dict(sets=[(0, 3, 0, 0), (3, 3, 2, 1)]),
        "ascending": dict(sets=[(0, 4, 0, 2), (4, 2, 2, 1)]),
        "finite": dict(t=bad_t),
        "> 0": dict(t=neg_t),
        "frequencies must": dict(nu=bad_nu),
        "Gamma0": dict(P=bad_P),
        "no grid sets": dict(sets=[]),
    }
    for word, kw in cases.items():
        for q in (None, BANDS):
            args = dict(P=P, ds=ds, sets=ok_sets, t=t, nu=nu)
            args.update(kw)
            rc, untouched = _raw(engine, args["P"], args["ds"], args["sets"], args["t"], args["nu"], q)
            assert rc == abi.VAG_ERR_INVALID, (word, q)
            assert untouched, (word, q)
            msg = engine._lib.vag_last_error().decode()
            assert word.strip() in msg, (word, msg)
    for q, word in (([], "no quantiles"), ([0.5, 1.5], "q[1]"), ([np.nan], "q[0]"), ([-0.1], "[0, 1]")):
        rc, untouched = _raw(engine, P, ds, ok_sets, t, nu, q)
        assert rc == abi.VAG_ERR_INVALID and untouched, q
        assert word in engine._lib.vag_last_error().decode(), q
    # messages name the set / the model
    _raw(engine, P, ds, [(0, 3, 0, 2), (3, 0, 2, 1)], t, nu)
    assert "set 1" in engine._lib.vag_last_error().decode()
    _raw(engine, P, np.array([0, 1, 5, 0]), ok_sets, t, nu)
    assert "model 2" in engine._lib.vag_last_error().decode()
    _raw(engine, bad_P, ds, ok_sets, t, nu)
    assert "model 2" in engine._lib.vag_last_error().decode()
    # the context stays usable
    assert _raw(engine, P, ds, ok_sets, t, nu, BANDS)[0] == abi.VAG_OK


# q: 0, 1, the median, the 68 % band, and 0.25, whose (n - 1) q is an integer for the sets of 5 and 9 members
Q_ALL = (0.0, 1.0, 0.5, 0.16, 0.84, 0.25)


def _assert_bands_equal(bands, n_used, want, want_used, shapes):
    assert np.array_equal(n_used, want_used)
    for d, (b, w) in enumerate(zip(bands, want)):
        assert b.shape == (len(Q_ALL),) + shapes[d], d
        if w is None:
            assert np.isnan(b).all(), d
        else:
            np.testing.assert_array_equal(b, w, err_msg=f"set {d}")  # -0 == +0: the sign of a zero is not compared


@pytest.mark.gpu
@pytest.mark.parametrize("ode_fail", [False, True])
def test_quantiles_equal_numpy_of_the_grid_flux(engine, ode_fail):
    # sets of 1, 2, 5 (odd) and 6 (even) models, one of 5200 (more than the 5120 members k_quantiles stages in shared
    # memory: selected from global memory), one with none, and a set of 9 with a nine-frequency grid
    sizes = [1, 2, 5, 6, 5200, 0, 9]
    grids = [(np.logspace(3, 5, 7), np.array([1e9, 4.84e14])), (np.array([1e4]), np.array([1e9])),
             (np.logspace(2, 4, 5), np.array([5e9, 1e14, 1e17])), (np.logspace(5, 7, 6), np.array([4.84e14])),
             (np.logspace(3, 6, 3), np.array([1e9, 1e17])), (np.logspace(3, 5, 2), np.array([1e9])),
             (np.logspace(3, 6, 11), np.logspace(9, 18, 9))]
    n = sum(sizes)
    P = configs.random_draw(n, seed=61)
    P[::3] = configs.random_draw(len(P[::3]), seed=62, rvs=True)
    P["t_resol"] = 3.0
    ds = np.repeat(np.arange(len(sizes), dtype=np.int32), sizes)
    perm = np.random.default_rng(63).permutation(n)
    P, ds = P[perm], ds[perm]
    try:
        if ode_fail:  # Boost's 500-rejection limit lowered to 1: VAG_ST_ODE_FAIL500 for some of the models
            engine.debug_set_ode_limits(0, 1)
        flux, st = engine.flux_density_grid_multi(P, grids, ds, return_status=True)
        bands, n_used, st_q = engine.flux_quantiles_multi(P, grids, ds, Q_ALL, return_status=True)
    finally:
        engine.debug_set_ode_limits(0, 0)
    assert np.array_equal(st, st_q)
    fail = (st & abi.ST_ODE_FAIL500) != 0
    assert fail.any() == ode_fail
    if ode_fail:
        assert (~fail[ds == 4]).any()
    want, want_used = _numpy_bands(flux, st, ds, len(grids), Q_ALL)
    assert want_used[4] > 5120 or ode_fail
    _assert_bands_equal(bands, n_used, want, want_used, [(g[1].size, g[0].size) for g in grids])


@pytest.mark.gpu
def test_likelihood_stack_bands_equal_numpy_of_each_fit(engine):
    fits, samples = _fits(engine, 2 * UNSPLIT_MODELS)
    # three frequencies per grid: every fit's k_eats tile is the batch's, so each stages the rows it stages alone
    grids = [(np.logspace(3, 6, 40), np.array([1e9, 4.84e14, 1e18])), (np.logspace(4, 7, 30), np.array([5e9, 1e14, 1e17])),
             (np.logspace(3.5, 6.5, 25), np.array([1e9, 5e9, 4.84e14]))]
    bands, n_used = fitting.LikelihoodStack(fits).flux_quantiles(samples, grids, BANDS)
    for k, (lk, s, (t, nu)) in enumerate(zip(fits, samples, grids)):
        P = lk.to_params(s)
        P = P[engine.valid_mask(P)]
        assert P.size >= UNSPLIT_MODELS and P.size < s.shape[0]  # rejected draws are dropped
        f, st = engine.flux_density_grid(P, t, nu, return_status=True)
        keep = (st & FAIL) == 0
        want = np.quantile(f[keep, 0], BANDS, axis=0)
        assert n_used[k] == keep.sum()
        np.testing.assert_array_equal(bands[k], want)
        one, used = lk.flux_quantiles(s, t, nu, BANDS)  # the single-fit form: the same batch as the reference
        np.testing.assert_array_equal(one, want)
        assert used == keep.sum()


# ---- CPU tier ---------------------------------------------------------------------------------------------------------
_SHIM = r"""
#include "vag_quantile.cuh"
// columns x[n_cols][n] -> out[n_q][n_cols]: the body k_quantiles runs per warp, here with one host thread as the group
extern "C" void quant_columns(const double* x, int n_cols, int n, const double* q, int n_q, double* out) {
    unsigned hist[vag::QUANT_BINS];
    for (int c = 0; c < n_cols; ++c) {
        const double* col = x + (size_t)c * n;
        vag::quant_column(vag::QuantSeq{}, [col](int i) { return vag::quant_key(col[i]); }, n, q, n_q, out + c,
                          (size_t)n_cols, hist);
    }
}
"""


@pytest.fixture(scope="module")
def quant_host(tmp_path_factory):
    d = tmp_path_factory.mktemp("quant")
    src, so = d / "quant.cpp", d / "libquant.so"
    src.write_text(_SHIM)
    # the host emulation's flags (oracle/hostemu/emu.py), contraction included: the body must not depend on it
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-march=x86-64-v3", "-ffp-contract=fast", "-fPIC", "-shared",
                           "-I", CSRC, str(src), "-o", str(so)])
    lib = C.CDLL(str(so))
    lib.quant_columns.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]

    def run(cols, q):
        x = np.ascontiguousarray(cols, dtype=np.float64)  # [n_cols, n]
        q = np.ascontiguousarray(q, dtype=np.float64)
        out = np.full((q.size, x.shape[0]), 7.0)
        lib.quant_columns(x.ctypes.data, x.shape[0], x.shape[1], q.ctypes.data, q.size, out.ctypes.data)
        return out

    return run


def _columns(rng, n, n_cols):
    """seeded columns: log-normal fluxes, heavy ties, zeros of both signs, negatives, a wide dynamic range"""
    cols = [rng.lognormal(-60, 3, n) for _ in range(n_cols)]
    cols.append(rng.integers(0, 3, n).astype(np.float64))  # ties
    cols.append(rng.choice([0.0, -0.0, 1e-300, 5e-324], n))  # zeros, a subnormal
    cols.append(rng.standard_normal(n) * 10.0 ** rng.integers(-300, 300, n))
    cols.append(np.full(n, 3.25))
    return np.stack(cols)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 6, 10, 257, 1000])
def test_host_selection_equals_numpy_quantile(quant_host, n):
    rng = np.random.default_rng(100 + n)
    q = np.concatenate([Q_ALL, [0.9, 0.1, 0.75, 1 / 3, 0.999], rng.uniform(0, 1, 8)])
    if n > 2:
        q = np.append(q, [1 / (n - 1), (n - 2) / (n - 1)])  # (n - 1) q an integer, or within rounding of one
    cols = _columns(rng, n, 6)
    got = quant_host(cols, q)
    assert got.shape == (q.size, cols.shape[0])
    np.testing.assert_array_equal(got, np.quantile(cols, q, axis=1, method="linear"))  # -0 == +0: the sign of a zero is not compared


def test_host_selection_nan_and_empty(quant_host):
    rng = np.random.default_rng(7)
    cols = rng.lognormal(0, 1, (4, 9))
    cols[1, 3] = np.nan
    cols[2, 0] = -np.nan
    got = quant_host(cols, BANDS)
    assert np.isnan(got[:, 1:3]).all()
    np.testing.assert_array_equal(got, np.quantile(cols, BANDS, axis=1))
    empty = quant_host(np.zeros((3, 0)), BANDS)
    assert np.isnan(empty).all()


def test_grid_set_layout_matches_header(tmp_path):
    src = tmp_path / "grid_set.c"
    fields = [f[0] for f in abi.GridSet._fields_]
    body = "".join(f'printf("%zu ", offsetof(vag_grid_set, {k}));' for k in fields)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){%s printf("%%zu\\n", '
                   'sizeof(vag_grid_set)); return 0;}' % (os.path.join(ROOT, "include", "vag.h"), body))
    exe = tmp_path / "grid_set"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    vals = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert vals == [getattr(abi.GridSet, k).offset for k in fields] + [C.sizeof(abi.GridSet)]
    assert fields == ["t0", "n_t", "nu0", "n_nu"]


class _RecordingEngine:
    device = 0

    def __init__(self):
        self.calls = []

    def flux_quantiles_multi(self, P, grids, dataset_of, q):
        ds = np.array(dataset_of)
        self.calls.append(dict(P=P.copy(), grids=grids, dataset_of=ds, q=q))
        return [np.zeros((len(q), len(nu), len(t))) for t, nu in grids], np.bincount(ds, minlength=len(grids))


def test_likelihood_stack_bands_are_one_call_without_rejected_draws():
    eng = _RecordingEngine()
    fits, samples = _fits(eng, 40, gpu=False)
    grids = [(np.logspace(3, 6, 5), np.array([1e9, 1e17])), (np.logspace(4, 7, 4), np.array([5e9])),
             (np.logspace(3, 5, 3), np.array([1e9, 5e9, 1e18]))]
    bands, n_used = fitting.LikelihoodStack(fits).flux_quantiles(samples, grids)
    assert len(eng.calls) == 1
    call = eng.calls[0]
    from vegasafterglow_b200.engine import Engine

    valid = [Engine.valid_mask(lk.to_params(s)) for lk, s in zip(fits, samples)]
    assert all(0 < v.sum() < v.size for v in valid)  # some draws of every fit are rejected (eps_e > 1)
    # every valid draw, in bounds or not, of fit 0, then fit 1, then fit 2, through each fit's own to_params
    assert np.array_equal(call["dataset_of"], np.repeat(np.arange(3), [v.sum() for v in valid]))
    want_P = np.concatenate([lk.to_params(s)[v] for lk, s, v in zip(fits, samples, valid)])
    assert call["P"].tobytes() == want_P.tobytes()
    assert call["grids"] is grids and tuple(call["q"]) == BANDS
    assert np.array_equal(n_used, [v.sum() for v in valid])
    assert [b.shape for b in bands] == [(3, nu.size, t.size) for t, nu in grids]
    # one definition, inherited by the band and device stacks
    assert fitting.BandLikelihoodStack.flux_quantiles is fitting.LikelihoodStack.flux_quantiles
    assert fitting.DeviceLikelihoodStack.flux_quantiles is fitting.LikelihoodStack.flux_quantiles


def test_single_fit_bands_make_the_same_call_with_one_grid():
    eng = _RecordingEngine()
    fits, samples = _fits(eng, 30, gpu=False)
    t, nu = np.logspace(3, 6, 5), np.array([1e9, 1e17])
    band, used = fits[2].flux_quantiles(samples[2], t, nu, q=(0.5,))
    call = eng.calls[0]
    from vegasafterglow_b200.engine import Engine

    P = fits[2].to_params(samples[2])
    P = P[Engine.valid_mask(P)]
    assert call["P"].tobytes() == P.tobytes() and not call["dataset_of"].any() and len(call["grids"]) == 1
    assert band.shape == (1, 2, 5) and used == P.size
