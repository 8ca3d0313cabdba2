"""K small fits with points and an X-ray band, three ways on one GPU: K DeviceLikelihood calls, one BandLikelihoodStack
call (host buffers), one DeviceLikelihoodStack call (device buffers, planned on the device).

    python scripts/device_stack_ab.py [--k 16 128] [--walkers 64 512] [--steps 20] [--warmup 3] [--out FILE]

Workload: K fits with FS tophat templates (ISM, t_resol 3), each with its own synthetic light curve: 36 points (3
frequencies x 12 epochs) and one 0.3-10 keV band of 5 frequency nodes over 6 epochs; every fit samples E_iso, Gamma0,
theta_c, n_ism, eps_e, eps_B, p and A_V (its points carry an extinction law).  Every walker is inside the bounds and valid,
so the three arms evaluate the same models.  Arms, alternated within one process (the order rotates every step):
  separate     K DeviceLikelihood.__call__, one vag_chi2_dev each
  band_stack   BandLikelihoodStack.__call__: host validation, one vag_chi2_multi_bands
  device_stack DeviceLikelihoodStack.__call__: one vag_chi2_multi_bands_dev
Per arm and (K, walkers): the median and range of the ms per step over --steps steps after --warmup warm-up steps, each
step timed from a device synchronisation to the next; the C-ABI launches per step (vag_last_launch_count summed over the
step's calls); the kernels per step that torch.profiler sees (the library's and torch's own); the H2D bytes per step
computed from the shapes (256-byte slice padding left out).  Checks: band_stack and device_stack give identical arrays.
The card's name, power limit and max SM clock come from a read-only nvidia-smi query and go into the JSON output.
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
ap.add_argument("--k", type=int, nargs="+", default=[16, 128])
ap.add_argument("--walkers", type=int, nargs="+", default=[64, 512])
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("needs a CUDA device")
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                   capture_output=True, text=True).stdout.strip()
card = dict(zip(("name", "power_limit", "max_sm_clock"), [s.strip() for s in q.split(",")])) if q else \
    {"name": torch.cuda.get_device_name(0)}
lines = []


def emit(d):
    s = json.dumps(d)
    print(s, flush=True)
    lines.append(s)


emit({"card": card})

NAMES = ["E_iso", "Gamma0", "theta_c", "n_ism", "eps_e", "eps_B", "p", "A_V"]
LOG = [True, True, False, True, True, True, False, False]
N_POINTS, N_BAND_T, BAND_NODES = 36, 6, 5
eng = Engine(0)


def fit_args(k):
    rng = np.random.default_rng(7000 + k)
    lo = rng.uniform(2.5, 3.5)
    t = np.repeat(np.logspace(lo, lo + 3.5, 12), 3)
    nu = np.tile([1e9, 4.84e14, 1e18], 12)
    flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
    tb = np.logspace(lo + 0.5, lo + 3, N_BAND_T)
    fb = 1e-12 * (tb / 1e4) ** -1.2 * np.exp(0.1 * rng.standard_normal(tb.size))
    tmpl = configs.make(lumi_dist=1e28, z=0.3)
    tmpl["t_resol"] = 3.0
    band = dict(t=tb, flux=fb, err=0.2 * fb, nu_min=7.25e16, nu_max=2.4e18, num_points=BAND_NODES)
    lower = np.array([51, 1.7, 0.03, -3, -2, -4, 2.1, 0])
    upper = np.array([54, 3, 0.4, 1, -0.1, -1, 2.8, 2])
    return (tmpl, NAMES, LOG, t, nu, flux, 0.2 * flux), dict(bands=[band], ext_kernel=rng.uniform(0, 1.5, t.size),
                                                          lower=lower, upper=upper)


def samples_of(k, n):
    rng = np.random.default_rng(9000 + k)
    return np.column_stack([rng.uniform(51, 54, n), rng.uniform(1.7, 3, n), rng.uniform(0.03, 0.4, n), rng.uniform(-3, 1, n),
                            rng.uniform(-2, -0.1, n), rng.uniform(-4, -1, n), rng.uniform(2.1, 2.8, n), rng.uniform(0, 2, n)])


def h2d_bytes(arm, K, n):
    """H2D bytes of one step from the shapes (N = K n walkers, all valid; 256-byte slice padding left out)."""
    N, P, T = K * n, K * N_POINTS, K * N_BAND_T
    grids = 2 * BAND_NODES * 8  # a band's frequency nodes and weights
    if arm == "separate":  # per fit: the columns; per band run: the nodes and weights
        return K * (n * len(NAMES) * 8 + grids)
    lists = 2 * N * 4 + N * 4 + (N + 1) * 4 + K * 16 + N * 4 + (N + 1) * 8  # gather, pt_of, e0, sets, set_of, pt_off
    bands = K * grids + K * 16 + N * 4 + 2 * (N + 1) * 8  # nodes + weights, table, band_of, grid / reduction offsets
    if arm == "band_stack":  # records, t / nu, the lists, lnF / sig / w / ext, A_V, band t / lnF / sig / w
        return N * abi.PARAMS_DTYPE.itemsize + 2 * P * 8 + lists + 4 * P * 8 + N * 8 + bands + 4 * T * 8
    # the packed columns with A_V and the fit of each walker, the lists, the band pointer table
    return N * (len(NAMES) + 1) * 8 + N * 8 + lists + bands + K * 4 * 8


def profiled_kernels(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type.name == "CUDA" and not e.name.startswith(("Memcpy", "Memset")))


for K in args.k:
    dev = [fitting.DeviceLikelihood(eng, *a, **kw) for a, kw in map(fit_args, range(K))]
    host = [fitting.BatchedLikelihood(eng, *a, **kw) for a, kw in map(fit_args, range(K))]
    dstack, bstack = fitting.DeviceLikelihoodStack(dev), fitting.BandLikelihoodStack(host)
    for n in args.walkers:
        S = [samples_of(k, n) for k in range(K)]
        launches = {}

        def separate():
            out, c = [], 0
            for lk, s in zip(dev, S):
                out.append(lk(s))
                c += eng.last_launch_count()
            launches["separate"] = c
            return out

        def band_stack():
            out = bstack(S)
            launches["band_stack"] = eng.last_launch_count()
            return out

        def device_stack():
            out = dstack(S)
            launches["device_stack"] = eng.last_launch_count()
            return out

        arms = {"separate": separate, "band_stack": band_stack, "device_stack": device_stack}
        names = list(arms)
        for _ in range(args.warmup):
            for fn in arms.values():
                fn()
        times, last = {a: [] for a in arms}, {}
        for step in range(args.steps):
            for a in names[step % 3:] + names[:step % 3]:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                last[a] = arms[a]()
                torch.cuda.synchronize()
                times[a].append((time.perf_counter() - t0) * 1e3)
        same = all(np.array_equal(x, y) for x, y in zip(last["band_stack"], last["device_stack"]))
        assert same, "band_stack and device_stack differ"
        assert all(np.isfinite(x).all() for x in last["device_stack"])
        for a in names:
            kernels = profiled_kernels(arms[a])
            emit({"arm": a, "K": K, "walkers_per_fit": n, "ms_median": round(float(np.median(times[a])), 3),
                  "ms_range": [round(float(np.min(times[a])), 3), round(float(np.max(times[a])), 3)], "steps": args.steps,
                  "warmup": args.warmup, "abi_launches_per_step": launches[a], "kernels_per_step_profiled": kernels,
                  "h2d_bytes_per_step": h2d_bytes(a, K, n), "card": card["name"], "power_limit": card.get("power_limit")})
        emit({"check": "band_stack == device_stack", "K": K, "walkers_per_fit": n, "identical": same})

if args.out:
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
