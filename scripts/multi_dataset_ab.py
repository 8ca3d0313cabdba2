"""K small fits on one GPU: K sequential calls, K calls over 4 engines in host threads, or one ragged call.

    python scripts/multi_dataset_ab.py [--walkers 64] [--reps 10] [--k 1 8 32 64]

Workload: K config-5-like fits (FS+RS tophat walkers, configs.random_draw with a different seed per fit), each with its
own synthetic light curve: 20 to 100 points, 3 to 5 bands, epochs over its own window.  Three arms, alternated within
one process (the order rotates every repeat), CUDA-synchronised wall time (the host-buffer calls return after a stream
synchronisation) after a warm-up of each arm:
  sequential  K Engine.chi2_series calls, one per fit, on one engine
  threads     the same K calls spread over 4 engines (one CUDA stream each), one host thread per engine
  multi       one Engine.chi2_multi call on the K data sets
Series mode 0 (the default) in every arm.  A second batch times one chi2_multi call on 8 of these fits whose odd
fits are SSC+KN forward-shock draws instead (configs.random_draw(..., ssc=True, kn=True)), in series modes 0 and 2: the
FS+RS fits never run the SSC kernels (k_ic_spectrum, k_eats MODE 2), and mode 0 never runs them banded.  Check: the multi result against per-fit chi2_series calls padded to 2368
models (37 copies of the 64 walkers, so that neither call splits rows) in series mode 1 -- bit for bit where both calls
stage the same rows per pass (include/vag.h) -- and the largest relative difference to the unpadded sequential arm.
Prints the card's name and power limit, then one JSON line per arm and K and one for the check.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from vegasafterglow_b200 import configs, fitting
from vegasafterglow_b200.engine import Engine

ap = argparse.ArgumentParser()
ap.add_argument("--walkers", type=int, default=64)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--k", type=int, nargs="+", default=[1, 8, 32, 64])
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("needs a CUDA device")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card or torch.cuda.get_device_name(0)}", flush=True)

N_THREADS = 4
UNSPLIT_MODELS = 2368


def light_curve(k):
    rng = np.random.default_rng(5000 + k)
    n_bands = int(rng.integers(3, 6))
    bands = np.sort(rng.choice([1e9, 5e9, 1.5e10, 1e14, 4.84e14, 1e15, 1e17, 1e18], n_bands, replace=False))
    n_epochs = int(rng.integers(-(-20 // n_bands), 100 // n_bands + 1))
    lo = rng.uniform(2.0, 4.0)
    t = np.repeat(np.logspace(lo, lo + rng.uniform(2.0, 4.0), n_epochs), n_bands)
    nu = np.tile(bands, n_epochs)
    flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
    return fitting.consolidate_data(t, nu, flux, 0.2 * flux, rng.uniform(0.5, 2.0, t.size))


K_MAX = max(args.k)
FITS = [(configs.random_draw(args.walkers, seed=2000 + k, rvs=True), light_curve(k)) for k in range(K_MAX)]
engines = [Engine(0) for _ in range(N_THREADS)]
pool = ThreadPoolExecutor(N_THREADS)


def sequential(K):
    return np.concatenate([engines[0].chi2_series(P, *data) for P, data in FITS[:K]])


def threads(K):
    def share(e):
        return [(k, engines[e].chi2_series(FITS[k][0], *FITS[k][1])) for k in range(e, K, N_THREADS)]

    parts = dict(kv for part in pool.map(share, range(N_THREADS)) for kv in part)
    return np.concatenate([parts[k] for k in range(K)])


def multi(K):
    P = np.concatenate([P for P, _ in FITS[:K]])
    ds = np.repeat(np.arange(K, dtype=np.int32), args.walkers)
    return engines[0].chi2_multi(P, [data for _, data in FITS[:K]], ds)


ARMS = {"sequential": sequential, "threads": threads, "multi": multi}
results = {}
for K in args.k:
    for fn in ARMS.values():
        fn(K)  # warm-up: workspaces grown, modules loaded
    times = {a: [] for a in ARMS}
    names = list(ARMS)
    for r in range(args.reps):
        for a in names[r % 3:] + names[:r % 3]:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            results[(a, K)] = ARMS[a](K)
            times[a].append((time.perf_counter() - t0) * 1e3)
    for a in names:
        ms = np.array(times[a])
        print(json.dumps({"arm": a, "K": K, "walkers_per_fit": args.walkers, "ms_median": round(float(np.median(ms)), 3),
                          "ms_min": round(float(ms.min()), 3), "ms_per_fit": round(float(np.median(ms)) / K, 3),
                          "reps": args.reps}), flush=True)

# ---- mixed batch with SSC+KN fits ---------------------------------------------------------------------------------------
K_SSC = 8
SSC_FITS = [(configs.random_draw(args.walkers, seed=3000 + k, ssc=True, kn=True) if k % 2 else
             configs.random_draw(args.walkers, seed=2000 + k, rvs=True), light_curve(k)) for k in range(K_SSC)]
P_SSC = np.concatenate([P for P, _ in SSC_FITS])
DS_SSC = np.repeat(np.arange(K_SSC, dtype=np.int32), args.walkers)
for mode in (0, 2):  # 0 picks per-point EATS on these light curves, 2 forces the banded one
    engines[0].set_series_mode(mode)
    engines[0].chi2_multi(P_SSC, [data for _, data in SSC_FITS], DS_SSC)  # warm-up
    ms = []
    for r in range(args.reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        engines[0].chi2_multi(P_SSC, [data for _, data in SSC_FITS], DS_SSC)
        ms.append((time.perf_counter() - t0) * 1e3)
    print(json.dumps({"arm": "multi_ssc_kn_mixed", "K": K_SSC, "walkers_per_fit": args.walkers, "series_mode": mode,
                      "ms_median": round(float(np.median(ms)), 3), "ms_min": round(float(np.min(ms)), 3),
                      "reps": args.reps}), flush=True)
engines[0].set_series_mode(0)

# ---- check ---------------------------------------------------------------------------------------------------------------
K = K_MAX
rel = lambda a, b: float(np.max(np.abs(a - b) / np.abs(b)))  # noqa: E731
vs_sequential = rel(results[("multi", K)], results[("sequential", K)])
try:
    engines[0].set_series_mode(1)
    got = multi(K)
    reps = -(-UNSPLIT_MODELS // args.walkers)
    want = np.concatenate([engines[0].chi2_series(np.tile(P, reps), *data)[:args.walkers] for P, data in FITS[:K]])
finally:
    engines[0].set_series_mode(0)
print(json.dumps({"check": "multi vs per-fit chi2_series", "K": K, "series_mode": 1, "padded_to": reps * args.walkers,
                  "bit_identical": bool(np.array_equal(got, want)), "max_rel_diff": rel(got, want),
                  "max_rel_diff_vs_unpadded_sequential": vs_sequential,
                  "threads_equal_sequential": bool(np.array_equal(results[("threads", K)], results[("sequential", K)])), "all_finite": bool(np.isfinite(got).all())}),
      flush=True)
pool.shutdown()
