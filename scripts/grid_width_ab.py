"""Grid-builder (K0) stage time per group width G (lanes per model, vag_set_grid_lanes) on seeded batches, CUDA events.

    python scripts/grid_width_ab.py [--workload fs|ll] [--batch N ...] [--lanes G ...] [--reps R]

fs = bench.py's flux_density_grid batch (100 t x 3 nu), ll = its config-5 log-likelihood batch (FS+RS walkers, series).
Per (batch, G): the library's `grid` stage (CUDA events from the k_grid launch to the end of the row set-up, one batch
alone) and the whole call, L2 flushed before every call; the widths are interleaved within every repetition so that
drift on a shared machine hits all of them alike.  Prints one JSON line per (batch, G) with the median and the range,
and whether every width produced the same output bit for bit.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from vegasafterglow_b200 import abi
from vegasafterglow_b200.engine import Engine

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="fs", choices=["fs", "ll"])
ap.add_argument("--batch", type=int, nargs="+", default=[16384])
ap.add_argument("--lanes", type=int, nargs="+", default=[4, 8, 16, 32])
ap.add_argument("--reps", type=int, default=7)
args = ap.parse_args()

dev = torch.device("cuda:0")
torch.cuda.set_stream(torch.cuda.Stream(device=dev))  # a stream of its own: the library's calls and the events share it
eng = Engine(0)
eng.set_capacity(256, 128)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
print(json.dumps({"gpu": torch.cuda.get_device_name(0), "workload": args.workload}))

for batch in args.batch:
    if args.workload == "fs":
        P, t, nu = bench.workload(batch)
        series = False
    else:
        P, t, nu = bench.loglike_workload(batch)
        series = True
    d_p = torch.from_numpy(P.view(np.uint8).copy()).to(dev)
    d_t, d_nu = torch.from_numpy(np.ascontiguousarray(t)).to(dev), torch.from_numpy(np.ascontiguousarray(nu)).to(dev)
    d_out = torch.empty((P.size, abi.NCOMP, t.size) if series else (P.size, abi.NCOMP, nu.size, t.size),
                        dtype=torch.float64, device=dev)
    d_st = torch.zeros(P.size, dtype=torch.int32, device=dev)

    def call():  # on the stream the events are recorded on
        flush.zero_()
        s = torch.cuda.current_stream().cuda_stream
        if series:
            eng.flux_density_series_dev(d_p.data_ptr(), P.size, d_t.data_ptr(), d_nu.data_ptr(), t.size, d_out.data_ptr(),
                                        d_st.data_ptr(), s)
        else:
            eng.flux_density_grid_dev(d_p.data_ptr(), P.size, d_t.data_ptr(), t.size, d_nu.data_ptr(), nu.size,
                                      d_out.data_ptr(), d_st.data_ptr(), s)

    grid_ms = {g: [] for g in args.lanes}
    call_ms = {g: [] for g in args.lanes}
    same = {}
    ref = None
    for g in args.lanes:  # warm-up of every width, and its outputs against the first width's
        eng.set_grid_lanes(g)
        for _ in range(2):
            call()
        torch.cuda.synchronize()
        if ref is None:
            ref = (d_out.clone(), d_st.clone())
        same[g] = bool(torch.equal(d_out, ref[0]) and torch.equal(d_st, ref[1]))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.reps):
        for g in args.lanes:
            eng.set_grid_lanes(g)
            eng.set_profiling(True)
            call()
            torch.cuda.synchronize()
            grid_ms[g].append(eng.last_stage_ms()["grid"])
            eng.set_profiling(False)
            flush.zero_()
            a.record()
            call()
            b.record()
            torch.cuda.synchronize()
            call_ms[g].append(a.elapsed_time(b))
    eng.set_grid_lanes(0)
    for g in args.lanes:
        print(json.dumps({"batch": batch, "lanes": g,
                          "grid_ms": round(float(np.median(grid_ms[g])), 4),
                          "grid_ms_range": [round(min(grid_ms[g]), 4), round(max(grid_ms[g]), 4)],
                          "call_ms": round(float(np.median(call_ms[g])), 4),
                          "call_ms_range": [round(min(call_ms[g]), 4), round(max(call_ms[g]), 4)],
                          "same_output_as_first_width": same[g]}), flush=True)
