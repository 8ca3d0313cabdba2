"""The grid builder gives the same grid bit for bit at every group width (lanes per model, vag_set_grid_lanes): the
width only decides which lane computes which element, every order-dependent reduction runs in uniform code."""
import numpy as np
import pytest

from tests.helpers import golden_names, load_golden

LANES = (4, 8, 16, 32)
# tophat, Gaussian (off-axis), power-law, two-component, reverse-shock and spreading models, and the edge fixtures
SOURCES = ("batch_fs_tophat_ism", "batch_fs_gauss_offaxis", "batch_fs_powerlaw_wind", "batch_fs_two_component",
           "batch_fs_spreading_gauss", "batch_fs_spreading_nonaxisym", "batch_rs_tophat_ism", "batch_rs_spreading_tophat",
           "batch_mixed_powerlaw_wing") + tuple(golden_names("edge_"))


def mixed_models():
    """(params, t_min, t_max) of every model of the sources, interleaved so that neighbouring groups of a warp build
    different kinds of grid."""
    models = []
    for name in SOURCES:
        g = load_golden(name)
        t = np.asarray(g["t"], dtype=np.float64)
        models += [(p, float(t.min()), float(t.max())) for p in g["params"][:8]]
    order = np.random.default_rng(7).permutation(len(models))
    return [models[i] for i in order]


@pytest.fixture
def lanes_reset(engine):
    yield engine
    engine.set_grid_lanes(0)


@pytest.mark.gpu
def test_grid_nodes_equal_host_build_at_every_width(lanes_reset):
    from oracle.hostemu import emu

    engine = lanes_reset
    models = mixed_models()
    host = [emu.details(p, t0, t1) for p, t0, t1 in models]
    for lanes in LANES:
        engine.set_grid_lanes(lanes)
        for (p, t0, t1), h in zip(models, host):
            d = engine.details(p, t0, t1)
            assert tuple(d["info"]) == tuple(h["info"]), lanes  # n_phi, n_theta, n_t, n_reps, symmetry, ..., status
            np.testing.assert_array_equal(d["theta"], h["theta"])
            np.testing.assert_array_equal(d["phi"], h["phi"])
            np.testing.assert_array_equal(d["reps"], h["reps"])


@pytest.mark.gpu
def test_mixed_batch_identical_at_every_width(lanes_reset):
    engine = lanes_reset
    p = np.concatenate([m[0][None] for m in mixed_models()])
    t, nu = np.logspace(1, 8, 40), np.array([1e9, 1e14, 1e18])
    ref = None
    for lanes in LANES:
        engine.set_grid_lanes(lanes)
        engine.set_profiling(True)
        try:
            out, st = engine.flux_density_grid(p, t, nu, return_status=True)
            work = engine.last_work()  # batch sums of theta nodes, quadrature attempts and rows: grid-derived
        finally:
            engine.set_profiling(False)
        if ref is None:
            ref = (out, st, work)
            continue
        np.testing.assert_array_equal(st, ref[1])
        np.testing.assert_array_equal(out, ref[0])  # NaN of a capacity-failed model compares equal to NaN
        assert work == ref[2], lanes


@pytest.mark.gpu
def test_grid_lanes_rejects_unsupported_widths(lanes_reset):
    for bad in (-1, 1, 2, 3, 64):
        with pytest.raises(ValueError, match="grid lanes"):
            lanes_reset.set_grid_lanes(bad)
