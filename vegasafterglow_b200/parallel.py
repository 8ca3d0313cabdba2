"""Walker partition across the GPUs of one box (SURVEY.md section 8e).

Every walker / parameter set is an independent model evaluation, so a batch is split into
contiguous blocks, one per rank (one process per GPU), with NO data-path collective; the only
inter-GPU traffic is the gather of the float64[n_walkers] chi-squared vector
(``torch.distributed`` all_gather over NCCL on GPUs -- NVLink/NVSwitch --, gloo in the CPU tests).
"""
from __future__ import annotations

import numpy as np


def partition(n: int, world: int, rank: int):
    """Contiguous block [lo, hi) of ``n`` walkers owned by ``rank``: ceil(n/world) per rank."""
    per = -(-n // world) if world > 0 else n
    lo = min(rank * per, n)
    return lo, min(lo + per, n)


def world_rank():
    """(world size, rank) of the initialised ``torch.distributed`` process group; (1, 0) without one."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def cost_proxy(params, t_min=1e2, t_max=1e7) -> np.ndarray:
    """Relative cost of one model evaluation from its parameters alone (SURVEY.md section 8e): unique ODE rows x
    lattice length for the dynamics, (phi rows) x (theta nodes) x (lattice length) for the EATS stage -- the node
    counts are the closed-form parts of ``auto_grid`` (src/core/grid-refinement.h:246-262,516-528,655,664-677), i.e. the
    same upper bounds the library sizes its workspaces with.  A tophat jet is one ODE row and, on axis, one phi row; a
    structured jet off axis is ~50 x ~15 of them: 10-30x the cost, which a contiguous split does not see."""
    from . import abi

    p = np.ascontiguousarray(params, dtype=abi.PARAMS_DTYPE).reshape(-1)
    rvs = p["has_rvs"] != 0
    th_res = np.where(p["theta_resol"] > 0, p["theta_resol"], np.where(rvs, 0.2, 0.15))
    ph_res = np.where(p["phi_resol"] > 0, p["phi_resol"], 0.06)
    t_res = np.where(p["t_resol"] > 0, p["t_resol"], np.where(rvs, 10.0, 6.0))
    lg = np.log10(np.maximum(1.0, np.maximum(p["Gamma0"], p["Gamma0_w"]) * 1.5708))
    n_theta = 36 + 90 * th_res + np.maximum(0.0, lg - 1) * th_res * 55 + np.where(p["theta_obs"] > 0, lg * th_res * 25, 0.0)
    phi_base = np.maximum(360 * ph_res, 1.0)
    n_phi = np.where((p["theta_obs"] == 0) & (p["axisymmetric"] != 0), 1.0,
                     np.where(p["axisymmetric"] != 0, 0.5 * (phi_base + 1) * 2.0, phi_base * 2.0))
    n_t = np.maximum(np.log10(t_max / t_min) + 6.0, 1.0) * t_res * np.where(rvs, 2.0, 1.0)
    uniform = (p["jet_type"] == abi.JET_TOPHAT) & (p["spreading"] == 0)
    few = p["jet_type"] == abi.JET_TWO_COMPONENT
    rows = np.where(uniform, 1.0, np.where(few & (p["spreading"] == 0), 3.0, n_theta))
    shocks = np.where(rvs, 2.0, 1.0)
    ode = rows * np.where(rvs, 6.0, 1.0) * 650.0 * 70.0                 # RHS calls x flops (SURVEY.md section 8d)
    ssc = np.where((p["fwd"]["ssc"] != 0) | (rvs & (p["rvs"]["ssc"] != 0)), 40.0, 1.0)
    eats = shocks * n_phi * n_theta * n_t * 5 * 120.0 * ssc
    return ode + eats + 3.0e5                                          # + the grid builder's fixed cost


def balanced_assignment(cost, world: int):
    """Index sets (one per rank) of near-equal total cost: walkers sorted by cost and dealt in serpentine order
    (rank 0..w-1, w-1..0, ...).  Deterministic, so every rank computes the same assignment from the same parameters."""
    cost = np.asarray(cost, dtype=np.float64)
    order = np.argsort(-cost, kind="stable")
    n = order.size
    pos = np.arange(n)
    lap, k = pos // max(world, 1), pos % max(world, 1)
    rank_of = np.where(lap % 2 == 0, k, world - 1 - k)
    return [np.sort(order[rank_of == r]) for r in range(world)]


def gather_indexed(local: np.ndarray, sets, n: int, device=None) -> np.ndarray:
    """All-gather per-rank float64 vectors whose entries belong to the walkers ``sets[rank]`` into a length-``n``
    vector: ``gather_indexed_tensor`` on the collective's device (the current GPU under NCCL, else the CPU), as numpy."""
    import torch
    import torch.distributed as dist

    if device is None:
        nccl = dist.is_available() and dist.is_initialized() and dist.get_backend() == "nccl"
        device = torch.device("cuda", torch.cuda.current_device()) if nccl else torch.device("cpu")
    local = torch.as_tensor(np.asarray(local, dtype=np.float64), device=device)
    return gather_indexed_tensor(local, sets, n).cpu().numpy()


def partitioned_chi2(engine, params, t, nu, lnF, sig, w, evaluate=None, balance=True, valid=None,
                     per_walker=None) -> np.ndarray:
    """chi2 of the whole ensemble, each rank evaluating its share on its own GPU; ONE all-gather of float64[~n / world].

    * ``valid`` (bool[n], computed identically on every rank -- ``Engine.valid_mask`` is pure host code): walkers the
      model constructor rejects are masked to +inf BEFORE the split, so every rank issues exactly one collective of one
      shape whatever its own block contains (the reference maps that exception to logL = -inf, samplers.py:63-70);
    * ``balance``: split by the cost proxy (mixed tophat / structured ensembles) instead of contiguous blocks;
    * ``evaluate(params_block) -> chi2_block`` defaults to ``engine.chi2_series``; the CPU tests pass a host evaluator
      to exercise the partition / gather logic under gloo;
    * ``per_walker``: a tuple of length-n arrays (e.g. a fitted A_V), sliced with the rank's walkers like ``params``
      and passed to ``evaluate`` as extra arguments."""
    n = len(params)
    world, rank = world_rank()
    keep = np.arange(n) if valid is None else np.nonzero(np.asarray(valid, dtype=bool))[0]
    if balance:
        sets = [keep[s] for s in balanced_assignment(cost_proxy(params[keep], float(np.min(t)), float(np.max(t))), world)]
    else:
        sets = [keep[slice(*partition(len(keep), world, r))] for r in range(world)]
    if evaluate is None:
        evaluate = lambda P: engine.chi2_series(P, t, nu, lnF, sig, w)  # noqa: E731
    mine = sets[rank]
    extra = [np.asarray(a)[mine] for a in per_walker or ()]
    local = evaluate(params[mine], *extra) if len(mine) else np.zeros(0)
    return gather_indexed(local, sets, n)


def gather_indexed_tensor(local, sets, n: int):
    """All-gather per-rank float64 tensors whose entries belong to the walkers ``sets[rank]``: the gather stays on the
    rank's device (NCCL on GPUs, gloo on the CPU) and the result is a length-``n`` tensor there, +inf where no rank
    wrote."""
    import torch
    import torch.distributed as dist

    dev = local.device
    out = torch.full((n,), float("inf"), dtype=torch.float64, device=dev)
    if len(sets) == 1 or not (dist.is_available() and dist.is_initialized()):
        out[torch.as_tensor(sets[0], dtype=torch.long, device=dev)] = local
        return out
    per = max(max(len(s) for s in sets), 1)
    buf = torch.full((per,), float("inf"), dtype=torch.float64, device=dev)
    buf[: local.numel()] = local
    got = torch.empty(per * len(sets), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(got, buf)
    for r, idx in enumerate(sets):
        out[torch.as_tensor(idx, dtype=torch.long, device=dev)] = got[r * per: r * per + len(idx)]
    return out
