"""The device-resident likelihood against the host-buffer one, and the cost of planning on the device.

    python scripts/device_likelihood_ab.py [--walkers 4096] [--reps 10]

Workload: config 5 (bench.py loglike_workload: FS+RS tophat walkers, 5 bands x 20 epochs of point data) plus one X-ray
band data set (6 epochs, 5 frequency nodes) and a fitted A_V ~ U(0, 2), sampled as a sampler would: 11 columns, the
log10 ones exponentiated by the likelihood.  Two pairs of arms, alternated within one process (the order flips every
repeat), CUDA-synchronised wall time after a warm-up of each:
  batched  fitting.BatchedLikelihood(samples): host validation, host records, one vag_chi2_ext call, D2H of chi2
  device   fitting.DeviceLikelihood(samples): the columns uploaded, records assembled in HBM, one vag_chi2_dev call
  series_dev  vag_chi2_series_dev on config-5 records and point data in HBM (fixed capacities, no validation)
  chi2_dev    vag_chi2_dev on the same buffers (device validation, planned capacities, one more stream sync)
Checks: batched == device and series_dev == chi2_dev, bit for bit.  Prints the card's name and power limit, then one
JSON line per arm and one for the checks.
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
ap.add_argument("--walkers", type=int, default=4096)
ap.add_argument("--reps", type=int, default=10)
args = ap.parse_args()

if not torch.cuda.is_available():
    sys.exit("needs a CUDA device")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"card: {card or torch.cuda.get_device_name(0)}", flush=True)

n = args.walkers
rng = np.random.default_rng(11)
eng = Engine(0)
stream = torch.cuda.current_stream().cuda_stream

# ---- likelihood classes ------------------------------------------------------------------------------------------
P5 = configs.random_draw(n, seed=2000, rvs=True)  # bench.py loglike_workload
t = np.sort(np.tile(np.logspace(2.5, 6.5, 20), 5))
nu = np.tile([1e9, 5e9, 4.84e14, 1e17, 1e18], 20)
flux = 1e-27 * (t / 1e4) ** -1.0 * (nu / 1e9) ** -0.6 * np.exp(0.1 * rng.standard_normal(t.size))
ext = rng.uniform(0.0, 1.5, t.size)
tb = np.logspace(3.2, 5.5, 6)
band = dict(t=tb, flux=1e-12 * (tb / 1e4) ** -1.2, err=2e-13 * (tb / 1e4) ** -1.2, nu_min=7.25e16, nu_max=2.4e18,
            num_points=5)
names = ["E_iso", "Gamma0", "theta_c", "n_ism", "eps_e", "eps_B", "p", "eps_e_r", "eps_B_r", "p_r", "A_V"]
log = [True, True, False, True, True, True, False, True, True, False, False]
samples = np.column_stack([np.log10(P5["E_iso"]), np.log10(P5["Gamma0"]), P5["theta_c"], np.log10(P5["n_ism"]),
                           np.log10(P5["fwd"]["eps_e"]), np.log10(P5["fwd"]["eps_B"]), P5["fwd"]["p"],
                           np.log10(P5["rvs"]["eps_e"]), np.log10(P5["rvs"]["eps_B"]), P5["rvs"]["p"],
                           rng.uniform(0.0, 2.0, n)])
lk_args = (P5[:1], names, log, t, nu, flux, 0.2 * flux)
lk_kw = dict(bands=[band], ext_kernel=ext)
batched = fitting.BatchedLikelihood(eng, *lk_args, **lk_kw)
device = fitting.DeviceLikelihood(eng, *lk_args, **lk_kw)

# ---- entry points on device buffers ------------------------------------------------------------------------------
pts = fitting.consolidate_data(t, nu, flux, 0.2 * flux)
d_pts = [torch.as_tensor(a, device="cuda:0") for a in pts]
d_P = torch.as_tensor(P5.view(np.uint8), device="cuda:0")
d_chi2 = {k: torch.empty(n, dtype=torch.float64, device="cuda:0") for k in ("series_dev", "chi2_dev")}


def series_dev():
    eng.chi2_series_dev(d_P.data_ptr(), n, *(a.data_ptr() for a in d_pts), t.size, d_chi2["series_dev"].data_ptr(),
                        stream=stream)
    return d_chi2["series_dev"]


def chi2_dev():
    eng.chi2_dev(d_P.data_ptr(), n, (*(a.data_ptr() for a in d_pts), t.size), (), d_chi2["chi2_dev"].data_ptr(),
                 stream=stream)
    return d_chi2["chi2_dev"]


pairs = [("batched", lambda: batched(samples), "device", lambda: device(samples)),
         ("series_dev", series_dev, "chi2_dev", chi2_dev)]
res = {}
for a_name, a_fn, b_name, b_fn in pairs:
    ms = {a_name: [], b_name: []}
    for fn in (a_fn, b_fn):  # warm-up: module loads, workspace growth
        fn()
    torch.cuda.synchronize()
    for rep in range(args.reps):
        order = ((a_name, a_fn), (b_name, b_fn)) if rep % 2 == 0 else ((b_name, b_fn), (a_name, a_fn))
        for name, fn in order:
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            ms[name].append(1e3 * (time.perf_counter() - t0))
            res[name] = out if isinstance(out, np.ndarray) else out.cpu().numpy()
    for name in (a_name, b_name):
        print(json.dumps({"arm": name, "walkers": n, "median_ms": float(np.median(ms[name])),
                          "min_ms": float(np.min(ms[name])), "max_ms": float(np.max(ms[name])), "reps": args.reps}),
              flush=True)

assert np.array_equal(res["batched"], res["device"]), "DeviceLikelihood differs from BatchedLikelihood"
assert np.array_equal(res["series_dev"], res["chi2_dev"]), "vag_chi2_dev differs from vag_chi2_series_dev"
print(json.dumps({"check": "batched == device and series_dev == chi2_dev bit for bit", "ok": True,
                  "finite_logp": int(np.isfinite(res["device"]).sum()), "walkers_inf_chi2": int(np.isinf(res["chi2_dev"]).sum()),
                  "st_invalid_bit": abi.ST_INVALID}))
