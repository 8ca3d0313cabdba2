"""Exposure averaging on the GPU against the host composition it replaces, and the cost of exposures in a stacked
likelihood.

    python scripts/exposures_ab.py [--models 4096] [--points 100] [--samples 10] [--fits 64] [--walkers 256] [--reps 5]

Two pairs of arms, each pair alternated within one process (the order flips every repeat), wall time of host-buffer calls
(each returns after a stream synchronisation), medians over --reps after one warm-up of every arm:
  flux pair, --models seeded tophat FS / FS+RS draws on --points points (log-spaced epochs 10^2..10^6 s in three bands,
  exposures 5 % to 50 % of t) with --samples samples each:
    host    the composition Engine.flux_density_exposures used before: flux_density_series on the sorted samples, the
            [n, 5, points x samples] result to the host, np.add.at and / samples there
    device  Engine.flux_density_exposures (vag_flux_density_exposures): averaged on the GPU, [n, 5, points] to the host
  likelihood pair, a BandLikelihoodStack of --fits fits x --walkers walkers (30 points in three bands and an X-ray band
  per fit, A_V on every other fit):
    expo    every point with an exposure of 20 % of t, --samples samples
    zero    the same fits with every exposure 0 (one sample per point: the call without exposures, plus one launch)
Each arm reports ms per call, its kernel launches and, for the flux pair, the device-to-host bytes of its flux.  Checks:
the two flux arms agree bit for bit.  Prints the card's name and power limit, then one JSON line per arm and check.
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

from vegasafterglow_b200 import abi, configs, fitting
from vegasafterglow_b200.engine import Engine

ap = argparse.ArgumentParser()
ap.add_argument("--models", type=int, default=4096)
ap.add_argument("--points", type=int, default=100)
ap.add_argument("--samples", type=int, default=10)
ap.add_argument("--fits", type=int, default=64)
ap.add_argument("--walkers", type=int, default=256)
ap.add_argument("--reps", type=int, default=5)
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("needs a CUDA device")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card or torch.cuda.get_device_name(0)}", flush=True)
eng = Engine(0)


def timed(arms, reps):
    """{arm: (median ms, all ms, last result)} of arms alternated, after one warm-up each"""
    last = {a: fn() for a, fn in arms.items()}
    names, times = list(arms), {a: [] for a in arms}
    for r in range(reps):
        for a in (names if r % 2 == 0 else names[::-1]):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            last[a] = arms[a]()
            times[a].append((time.perf_counter() - t0) * 1e3)
    return {a: (float(np.median(times[a])), times[a], last[a]) for a in names}


# ---- flux pair ------------------------------------------------------------------------------------------------------------
n_half = args.models // 2
P = np.concatenate([configs.random_draw(args.models - n_half, seed=1), configs.random_draw(n_half, seed=2, rvs=True)])
t = np.repeat(np.logspace(2, 6, -(-args.points // 3)), 3)[:args.points]
nu = np.tile([1e9, 4.84e14, 1e18], -(-args.points // 3))[:args.points]
e = t * np.random.default_rng(3).uniform(0.05, 0.5, t.size)
k = args.samples


def host():
    kk = np.arange(k, dtype=np.float64)
    ts = (t[:, None] + kk[None, :] * (e / (k - 1))[:, None]).reshape(-1)
    idx = np.repeat(np.arange(t.size), k)
    order = np.argsort(ts, kind="stable")
    f = eng.flux_density_series(P, ts[order], np.repeat(nu, k)[order])
    launches, d2h = eng.last_launch_count(), f.nbytes
    out = np.zeros((f.shape[0], abi.NCOMP, t.size))
    np.add.at(out, (slice(None), slice(None), idx[order]), f)
    out /= float(k)
    return out, launches, d2h


def device():
    out = eng.flux_density_exposures(P, t, nu, e, k)
    return out, eng.last_launch_count(), out.nbytes


res = timed({"host": host, "device": device}, args.reps)
for a, (med, all_ms, (_, launches, d2h)) in res.items():
    print(json.dumps({"pair": "flux", "arm": a, "models": P.size, "points": t.size, "samples": k,
                      "ms_median": round(med, 3), "ms_all": [round(x, 3) for x in all_ms], "d2h_flux_bytes": int(d2h),
                      "launches": int(launches)}), flush=True)
same = np.array_equal(res["host"][2][0], res["device"][2][0], equal_nan=True)
print(json.dumps({"check": "device average vs host composition", "bit_identical": bool(same)}), flush=True)
assert same

# ---- likelihood pair ------------------------------------------------------------------------------------------------------
NAMES = ["E_iso", "Gamma0", "theta_c", "n_ism", "eps_e", "eps_B", "p"]
LOG = [True, True, False, True, True, True, False]


def stack(expo_frac):
    fits, samples = [], []
    for f in range(args.fits):
        rng = np.random.default_rng(100 + f)
        tf = np.repeat(np.logspace(rng.uniform(2, 3), rng.uniform(5.5, 6.5), 10), 3)
        nuf = np.tile([1e9, 4.84e14, 1e18], 10)
        flux = 1e-27 * (tf / 1e4) ** -1.0 * (nuf / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(tf.size))
        tb = np.logspace(3, 5.5, 8)
        fb = 1e-12 * (tb / 1e4) ** -1.2
        av = f % 2 == 1
        fits.append(fitting.BatchedLikelihood(eng, configs.make(lumi_dist=1e28, z=0.3), NAMES + (["A_V"] if av else []),
                                              LOG + ([False] if av else []), tf, nuf, flux, 0.2 * flux,
                                              bands=[dict(t=tb, flux=fb, err=0.2 * fb, nu_min=7.25e16, nu_max=2.4e18)],
                                              ext_kernel=rng.uniform(0, 1.5, tf.size) if av else None,
                                              expo_time=expo_frac * tf, expo_points=k))
        cols = [rng.uniform(51, 54, args.walkers), rng.uniform(1.7, 3, args.walkers), rng.uniform(0.03, 0.4, args.walkers),
                rng.uniform(-3, 1, args.walkers), rng.uniform(-2, -0.5, args.walkers), rng.uniform(-4, -1, args.walkers),
                rng.uniform(2.1, 2.8, args.walkers)]
        samples.append(np.column_stack(cols + ([rng.uniform(0, 2, args.walkers)] if av else [])))
    return fitting.BandLikelihoodStack(fits), samples


stacks = {"expo": stack(0.2), "zero": stack(0.0)}


def run(a):
    def f():
        s, samples = stacks[a]
        return s(samples), eng.last_launch_count()
    return f


res = timed({a: run(a) for a in stacks}, args.reps)
for a, (med, all_ms, (logp, launches)) in res.items():
    print(json.dumps({"pair": "likelihood", "arm": a, "fits": args.fits, "walkers_per_fit": args.walkers, "samples": k,
                      "ms_median": round(med, 3), "ms_all": [round(x, 3) for x in all_ms], "launches": int(launches),
                      "finite_logp": int(sum(np.isfinite(x).sum() for x in logp))}), flush=True)
