"""Independent restarts / bootstrap fits, one fit per GPU slot (BASELINE.json config 5; SURVEY.md 8e).

The path shards over FITS, not inside a fit: rank r of W runs fits r, r + W, r + 2W, ... on its own GPU with
no data-path collective; only the per-fit results (final log-evidence, parameters, iterations) are gathered
at the end (`torch.distributed.all_gather_object`, NCCL or gloo).  `fit_fn(fit_index) -> dict` does the work,
which keeps this scheduler testable on CPU with a stub.

`concurrency` fits of a rank's share run at the same time on its GPU (one host thread and one fit handle each; the C
ABI is safe across handles).  A fit of a few thousand points is bound by the serial panel chain of its Cholesky, so a
second fit's GEMMs fill the SMs the chain leaves idle -- measured on one B200 (`scripts/concurrent_fits.py`,
`profiles/r02/concurrent_fits.log`): n = 4096 (C2 shape) 198 -> 285 -> 311 iterations/s aggregate with 1 / 2 / 3
concurrent fits, n = 8192 (config 5) 49.0 -> 53.2 -> 54.1 with 1 / 2 / 4; nothing to gain at n = 16384.
"""
from __future__ import annotations

from typing import Callable, Dict, List


def assign_fits(n_fits: int, world: int) -> List[List[int]]:
    """Static round-robin: fit i goes to rank i % world (8 per GPU for 64 fits on 8 GPUs)."""
    if world < 1 or n_fits < 0:
        raise ValueError("need world >= 1 and n_fits >= 0")
    return [list(range(r, n_fits, world)) for r in range(world)]


def run_restarts(n_fits: int, fit_fn: Callable[[int], Dict], dist=None, concurrency: int = 1) -> List[Dict]:
    """Runs this rank's share (`concurrency` fits at a time) and returns ALL results ordered by fit index (on every
    rank)."""
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    share = assign_fits(n_fits, world)[rank]
    if concurrency <= 1 or len(share) <= 1:
        mine = [dict(fit_fn(i), fit=i, rank=rank) for i in share]
    else:
        from concurrent.futures import ThreadPoolExecutor

        with ThreadPoolExecutor(max_workers=int(concurrency)) as pool:  # ctypes calls release the GIL
            mine = [dict(r, fit=i, rank=rank) for i, r in zip(share, pool.map(fit_fn, share))]
    if dist is None:
        return mine
    gathered = [None] * world
    dist.all_gather_object(gathered, mine)
    out = [r for part in gathered for r in part]
    out.sort(key=lambda r: r["fit"])
    if [r["fit"] for r in out] != list(range(n_fits)):
        raise RuntimeError("restart results are incomplete")
    return out


def assign_contiguous(n_fits: int, world: int) -> List[List[int]]:
    """Contiguous shares whose sizes differ by at most one (rank r of 3 for 8 fits: [0, 1, 2], [3, 4, 5], [6, 7])."""
    if world < 1 or n_fits < 0:
        raise ValueError("need world >= 1 and n_fits >= 0")
    base, extra = divmod(n_fits, world)
    out, lo = [], 0
    for r in range(world):
        hi = lo + base + (1 if r < extra else 0)
        out.append(list(range(lo, hi)))
        lo = hi
    return out


def run_batched_restarts(n_fits: int, make_batch: Callable[[List[int]], List[Dict]], dist=None) -> List[Dict]:
    """Like run_restarts, but each rank runs its contiguous share as ONE batched fit: `make_batch(fit_indices)` fits
    them together (e.g. through `fit.AceFitBatch` or `kernel.ace_train_batch`) and returns one result dict per index,
    in order.  Returns ALL results ordered by fit index on every rank, shaped like run_restarts' (so best_restart
    applies)."""
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    share = assign_contiguous(n_fits, world)[rank]
    res = list(make_batch(share)) if share else []
    if len(res) != len(share):
        raise RuntimeError(f"make_batch returned {len(res)} results for {len(share)} fits")
    mine = [dict(r, fit=i, rank=rank) for i, r in zip(share, res)]
    if dist is None:
        return mine
    gathered = [None] * world
    dist.all_gather_object(gathered, mine)
    out = [r for part in gathered for r in part]
    out.sort(key=lambda r: r["fit"])
    if [r["fit"] for r in out] != list(range(n_fits)):
        raise RuntimeError("restart results are incomplete")
    return out


def best_restart(results: List[Dict]) -> Dict:
    """The fit with the largest final log-evidence (non-finite evidences lose)."""
    import math

    ok = [r for r in results if math.isfinite(r.get("evidence", float("nan")))]
    if not ok:
        raise RuntimeError("no restart produced a finite evidence")
    return max(ok, key=lambda r: r["evidence"])
