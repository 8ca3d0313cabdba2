"""Fitted extinction on a config-5-like ensemble: the grouped evaluation it replaces against one vag_chi2_ext call.

    python scripts/extinction_ab.py [--walkers 4096] [--reps 5] [--grouped-reps 2]

4096 FS+RS tophat walkers (configs.random_draw(..., rvs=True)), 5 bands x 20 epochs of point data and a per-walker
A_V ~ U(0, 2).  Three arms, CUDA-synchronised wall time after a warm-up of each:
  grouped  one Engine.chi2 per distinct A_V with the shift lnF_obs + A_V ext_k computed in numpy (a fitted A_V makes
           every group one walker): the evaluation GpuFitterEvaluator did before vag_chi2_ext
  ext      one Engine.chi2(..., extinction=(ext_k, A_V)): one vag_chi2_ext call
  plain    Engine.chi2_series (vag_chi2_series -> vag_chi2) without extinction, the control
Checks: `ext` equals the same-batch oracle (one whole-batch call per distinct A_V, that value's rows) bit for bit, and
`grouped` agrees with `ext` to 1e-9 relative (different batch sizes round differently).  Prints the card's name and
power limit, then one JSON line per arm and one for the checks.
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

from vegasafterglow_b200 import configs, fitting
from vegasafterglow_b200.engine import Engine

ap = argparse.ArgumentParser()
ap.add_argument("--walkers", type=int, default=4096)
ap.add_argument("--reps", type=int, default=5, help="timed repeats of the ext and plain arms")
ap.add_argument("--grouped-reps", type=int, default=2, help="timed repeats of the grouped arm (one call per walker)")
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("needs a CUDA device")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card or torch.cuda.get_device_name(0)}", flush=True)

rng = np.random.default_rng(7)
P = configs.random_draw(args.walkers, seed=2000, rvs=True)
t = np.sort(np.tile(np.logspace(2.5, 6.5, 20), 5))
nu = np.tile([1e9, 5e9, 4.84e14, 1e17, 1e18], 20)
flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
pts = fitting.consolidate_data(t, nu, flux, 0.2 * flux)
ext = rng.uniform(0.0, 1.5, t.size)  # finite coefficients at every point, so every point is shifted
A_V = rng.uniform(0.0, 2.0, P.size)
eng = Engine(0)


def shifted(av):
    return pts[0], pts[1], pts[2] + av * ext, pts[3], pts[4]


def grouped():
    out = np.empty(P.size)
    for av in np.unique(A_V):
        sel = A_V == av
        out[sel] = eng.chi2(P[sel], shifted(av), ())
    return out


arms = {"grouped": grouped, "ext": lambda: eng.chi2(P, pts, (), extinction=(ext, A_V)),
        "plain": lambda: eng.chi2_series(P, *pts)}


def timed(fn, reps):
    fn()  # warm-up: module loads, workspace growth
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ms.append(1e3 * (time.perf_counter() - t0))
    return out, ms


res = {}
for name, reps in (("plain", args.reps), ("ext", args.reps), ("grouped", args.grouped_reps)):
    out, ms = timed(arms[name], reps)
    res[name] = out
    print(json.dumps({"arm": name, "walkers": int(P.size), "distinct_A_V": int(np.unique(A_V).size),
                      "median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)),
                      "reps": reps}), flush=True)

oracle = np.empty(P.size)
for av in np.unique(A_V):
    sel = A_V == av
    oracle[sel] = eng.chi2(P, shifted(av), ())[sel]
assert np.array_equal(res["ext"], oracle), "vag_chi2_ext differs from the same-batch oracle"
fin = np.isfinite(res["ext"])  # +inf: an ODE that failed (VAG_ST_ODE_FAIL500), in both arms alike
assert np.array_equal(fin, np.isfinite(res["grouped"]))
rel = float(np.max(np.abs(res["grouped"][fin] - res["ext"][fin]) / np.abs(res["ext"][fin])))
assert rel <= 1e-9, rel
print(json.dumps({"check": "ext == same-batch oracle bit for bit", "ok": True, "grouped_vs_ext_max_rel": rel,
                  "walkers_inf": int((~fin).sum())}))
