"""K small fits with band-integrated data on one GPU: K sequential calls, K calls over 4 engines in host threads, or one
ragged call.

    python scripts/multi_band_ab.py [--walkers 64] [--reps 10] [--runs 3] [--k 1 8 32 64]

Workload: K fits of FS+RS tophat walkers (configs.random_draw with a different seed per fit), each with its own synthetic
data: 20 to 100 points in 3 to 5 bands (as scripts/multi_dataset_ab.py), an X-ray band of 0.3-10 keV (5 frequency nodes,
10 to 30 epochs) and, for every other fit, an optical band (3 nodes, 5 to 15 epochs).  Three arms, alternated within one
process (the order rotates every repeat), CUDA-synchronised wall time (the host-buffer calls return after a stream
synchronisation) after a warm-up of each arm:
  sequential  K Engine.chi2 calls, one per fit, on one engine: 1 + (its bands) pipeline runs each
  threads     the same K calls spread over 4 engines (one CUDA stream each), one host thread per engine
  multi       one Engine.chi2_multi_bands call on the K data sets: one point pass and one band pass
Series mode 0 (the default) in every arm.  Every arm is timed `--runs` times (each time `--reps` calls); the script prints
each run's median and the range of the medians.  A second batch times 8 of these fits whose odd fits are SSC+KN
forward-shock draws (configs.random_draw(..., ssc=True, kn=True)), so that the grid-kind ragged k_eats of MODE 1 and 2
run, in the sequential and the multi arm.  Check: the multi result against per-fit Engine.chi2 calls padded to 2368
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
ap.add_argument("--runs", type=int, default=3)
ap.add_argument("--k", type=int, nargs="+", default=[1, 8, 32, 64])
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("needs a CUDA device")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card or torch.cuda.get_device_name(0)}", flush=True)

N_THREADS = 4
UNSPLIT_MODELS = 2368


def fit_data(k):
    """(points, bands) of fit k"""
    rng = np.random.default_rng(5000 + k)
    n_bands = int(rng.integers(3, 6))
    freqs = np.sort(rng.choice([1e9, 5e9, 1.5e10, 1e14, 4.84e14, 1e15, 1e17, 1e18], n_bands, replace=False))
    n_epochs = int(rng.integers(-(-20 // n_bands), 100 // n_bands + 1))
    lo = rng.uniform(2.0, 4.0)
    hi = lo + rng.uniform(2.0, 4.0)
    t = np.repeat(np.logspace(lo, hi, n_epochs), n_bands)
    nu = np.tile(freqs, n_epochs)
    flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
    pts = fitting.consolidate_data(t, nu, flux, 0.2 * flux, rng.uniform(0.5, 2.0, t.size))

    def band(n, nu_min, nu_max, num):
        tb = np.logspace(lo + 0.5, hi, n)
        fb = 1e-12 * (tb / 1e4) ** -1.2 * np.exp(0.1 * rng.standard_normal(n))
        return fitting.band_obs(tb, fb, 0.2 * fb, nu_min, nu_max, num)

    bands = [band(int(rng.integers(10, 31)), 7.25e16, 2.4e18, 5)]
    if k % 2:
        bands.append(band(int(rng.integers(5, 16)), 4e14, 7.5e14, 3))
    return pts, bands


K_MAX = max(args.k)
FITS = [(configs.random_draw(args.walkers, seed=2000 + k, rvs=True), *fit_data(k)) for k in range(K_MAX)]
engines = [Engine(0) for _ in range(N_THREADS)]
pool = ThreadPoolExecutor(N_THREADS)


def sequential(fits, eng=None):
    eng = eng or engines[0]
    return np.concatenate([eng.chi2(P, pts, bands) for P, pts, bands in fits])


def threads(fits):
    def share(e):
        return [(k, engines[e].chi2(*fits[k])) for k in range(e, len(fits), N_THREADS)]

    parts = dict(kv for part in pool.map(share, range(N_THREADS)) for kv in part)
    return np.concatenate([parts[k] for k in range(len(fits))])


def multi(fits):
    P = np.concatenate([P for P, _, _ in fits])
    ds = np.repeat(np.arange(len(fits), dtype=np.int32), [P.size for P, _, _ in fits])
    return engines[0].chi2_multi_bands(P, [pts for _, pts, _ in fits], [bands for _, _, bands in fits], ds)


def timed(arms, fits):
    """{arm: [median ms of each run]} and the last result of each arm"""
    for fn in arms.values():
        fn(fits)  # warm-up: workspaces grown, modules loaded
    med, last, names = {a: [] for a in arms}, {}, list(arms)
    for _ in range(args.runs):
        times = {a: [] for a in arms}
        for r in range(args.reps):
            for a in names[r % len(names):] + names[:r % len(names)]:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                last[a] = arms[a](fits)
                times[a].append((time.perf_counter() - t0) * 1e3)
        for a in names:
            med[a].append(float(np.median(times[a])))
    return med, last


def report(arm, K, meds, **extra):
    print(json.dumps({"arm": arm, "K": K, "walkers_per_fit": args.walkers, "ms_median_per_run": [round(m, 3) for m in meds],
                      "ms_range": [round(min(meds), 3), round(max(meds), 3)], "reps": args.reps, **extra}), flush=True)


results = {}
for K in args.k:
    meds, last = timed({"sequential": sequential, "threads": threads, "multi": multi}, FITS[:K])
    n_band_sets = sum(len(b) for _, _, b in FITS[:K])
    for a, m in meds.items():
        report(a, K, m, band_sets=n_band_sets)
    results[K] = last

# ---- mixed batch with SSC+KN fits ---------------------------------------------------------------------------------------
K_SSC = 8
SSC_FITS = [(configs.random_draw(args.walkers, seed=3000 + k, ssc=True, kn=True) if k % 2 else
             configs.random_draw(args.walkers, seed=2000 + k, rvs=True), *fit_data(k)) for k in range(K_SSC)]
meds, ssc_last = timed({"sequential": sequential, "multi": multi}, SSC_FITS)
for a, m in meds.items():
    report(a + "_ssc_kn_mixed", K_SSC, m)

# ---- check ---------------------------------------------------------------------------------------------------------------
K = K_MAX
rel = lambda a, b: float(np.max(np.abs(a - b) / np.abs(b)))  # noqa: E731
vs_sequential = rel(results[K]["multi"], results[K]["sequential"])
ssc_vs_sequential = rel(ssc_last["multi"], ssc_last["sequential"])
try:
    engines[0].set_series_mode(1)
    got = multi(FITS[:K])
    reps = -(-UNSPLIT_MODELS // args.walkers)
    want = np.concatenate([engines[0].chi2(np.tile(P, reps), pts, bands)[:args.walkers] for P, pts, bands in FITS[:K]])
finally:
    engines[0].set_series_mode(0)
print(json.dumps({"check": "multi vs per-fit chi2", "K": K, "series_mode": 1, "padded_to": reps * args.walkers,
                  "bit_identical": bool(np.array_equal(got, want)), "max_rel_diff": rel(got, want),
                  "max_rel_diff_vs_unpadded_sequential": vs_sequential, "ssc_max_rel_diff_vs_sequential": ssc_vs_sequential,
                  "threads_equal_sequential": bool(np.array_equal(results[K]["threads"], results[K]["sequential"])),
                  "all_finite": bool(np.isfinite(got).all())}), flush=True)
pool.shutdown()
