"""Posterior-predictive bands of K fits: K grid calls + numpy.quantile, one per-model grid call + numpy.quantile, or one
call that reduces on the GPU.

    python scripts/predictive_ab.py [--k 8 64] [--draws 500 2000] [--reps 3] [--q 0.16 0.5 0.84]

Workload: K seeded fits, fit k forward-shock tophat draws (configs.random_draw, seed 7000 + k) with a reverse shock for
every odd k, each on its own plotting grid: 100 to 200 log-spaced epochs over a window of its own (10^(2..3.5) s to
10^(5.5..7) s) x 3 to 6 frequencies between 1 GHz and 1 keV.  Three arms, alternated within one process (the order
rotates every repeat), wall time of host-buffer calls (each returns after a stream synchronisation), medians over
--reps after one warm-up of every arm:
  per_fit     K Engine.flux_density_grid calls, then numpy.quantile of each fit's total plane on the host
  grid_multi  one Engine.flux_density_grid_multi call, then numpy.quantile per fit on the host
  quantiles   one Engine.flux_quantiles_multi call: flux and quantiles on the GPU, only the bands come back
Each arm reports ms per call, the device-to-host bytes its calls move (flux or bands, status, n_used) and its kernel
launches (vag_last_launch_count summed over its calls).  Models whose ODE failed or whose grid exceeded the capacity are
left out of the quantiles in every arm.  Checks: quantiles equals numpy.quantile of grid_multi's flux bit for bit (the
same batch), and per_fit to rounding (a fit's batch of its own draws splits its rows into partial sums differently from
the batch of all fits: vag.h).  Prints the card's name and power limit, then one JSON line per (K, draws, arm) and per
check.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from vegasafterglow_b200 import abi, configs
from vegasafterglow_b200.engine import Engine

ap = argparse.ArgumentParser()
ap.add_argument("--k", type=int, nargs="+", default=[8, 64])
ap.add_argument("--draws", type=int, nargs="+", default=[500, 2000])
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--q", type=float, nargs="+", default=[0.16, 0.5, 0.84])
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("needs a CUDA device")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card or torch.cuda.get_device_name(0)}", flush=True)

FAIL = abi.ST_ODE_FAIL500 | abi.ST_CAPACITY
Q = np.asarray(args.q)
eng = Engine(0)


def grid_of(k):
    rng = np.random.default_rng(8000 + k)
    lo, hi = rng.uniform(2.0, 3.5), rng.uniform(5.5, 7.0)
    nu = np.sort(rng.choice([1e9, 5e9, 1.5e10, 1e14, 4.84e14, 1e15, 1e17, 2.4e17], int(rng.integers(3, 7)), replace=False))
    return np.logspace(lo, hi, int(rng.integers(100, 201))), nu


def fits(K, n):
    return [(configs.random_draw(n, seed=7000 + k, rvs=bool(k % 2)), *grid_of(k)) for k in range(K)]


def host_bands(F, st):
    """numpy.quantile of the total planes F[n, n_nu, n_t] of the members (status without FAIL bits)"""
    keep = (st & FAIL) == 0
    return np.quantile(F[keep], Q, axis=0, method="linear") if keep.any() else np.full((Q.size,) + F.shape[1:], np.nan)


def per_fit(fs):
    bands, d2h, launches = [], 0, 0
    for P, t, nu in fs:
        f, st = eng.flux_density_grid(P, t, nu, return_status=True)
        launches += eng.last_launch_count()
        d2h += f.nbytes + st.nbytes
        bands.append(host_bands(f[:, 0], st))
    return bands, d2h, launches


def batch(fs):
    P = np.concatenate([P for P, _, _ in fs])
    ds = np.repeat(np.arange(len(fs), dtype=np.int32), [P.size for P, _, _ in fs])
    return P, [(t, nu) for _, t, nu in fs], ds


def grid_multi(fs):
    P, grids, ds = batch(fs)
    flux, st = eng.flux_density_grid_multi(P, grids, ds, return_status=True)
    d2h = abi.NCOMP * 8 * sum(f[0].size for f in flux) + st.nbytes
    bands = [host_bands(np.stack([flux[m][0] for m in np.nonzero(ds == d)[0]]), st[ds == d]) for d in range(len(fs))]
    return bands, d2h, eng.last_launch_count()


def quantiles(fs):
    P, grids, ds = batch(fs)
    bands, n_used, st = eng.flux_quantiles_multi(P, grids, ds, Q, return_status=True)
    return bands, sum(b.nbytes for b in bands) + n_used.nbytes + st.nbytes, eng.last_launch_count()


ARMS = {"per_fit": per_fit, "grid_multi": grid_multi, "quantiles": quantiles}
for K in args.k:
    for n in args.draws:
        fs = fits(K, n)
        last = {a: fn(fs) for a, fn in ARMS.items()}  # warm-up: workspaces grown, modules loaded
        names, times = list(ARMS), {a: [] for a in ARMS}
        for r in range(args.reps):
            for a in names[r % len(names):] + names[:r % len(names)]:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                last[a] = ARMS[a](fs)
                times[a].append((time.perf_counter() - t0) * 1e3)
        cols = sum(t.size * nu.size for _, t, nu in fs)
        for a in names:
            print(json.dumps({"arm": a, "K": K, "draws_per_fit": n, "models": K * n, "columns": cols, "q": args.q,
                              "ms_median": round(float(np.median(times[a])), 3),
                              "ms_all": [round(x, 3) for x in times[a]], "d2h_bytes": int(last[a][1]),
                              "launches": int(last[a][2])}), flush=True)
        same = all(np.array_equal(g, w, equal_nan=True) for g, w in zip(last["quantiles"][0], last["grid_multi"][0]))
        rel = max(float(np.nanmax(np.abs(g - w) / np.abs(w))) for g, w in zip(last["quantiles"][0], last["per_fit"][0]))
        print(json.dumps({"check": "quantiles vs numpy.quantile", "K": K, "draws_per_fit": n,
                          "bit_identical_to_grid_multi_numpy": same, "max_rel_diff_to_per_fit_numpy": rel}), flush=True)
        assert same, "quantiles differ from numpy.quantile of the same flux"
        assert rel <= 1e-10, rel
