"""torchrun --nproc-per-node 2 scripts/shard_posterior_check.py : the marginal posterior of a fit sharded over 2 GPUs
(predict_marginal with ATE / ATT / ATU, predict_marginal_batch with S = 21).  Every rank must return the same result
bit for bit, equal bit for bit to the same fit played by one process (shard_emulate(2), rank 0), and within the
tolerances of tests/test_gpu_shard_posterior.py of the unsharded fit.  Prints one JSON line with "ok"."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"
import numpy as np
import torch, torch.distributed as dist
from additivecausalexpansion_b200.fit import AceFit

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))

n, p, Bz, kernel, iters = 2048, 8, 3, "SE", 3
MEAN_Y, STD_Y, STD_Z = 0.4, 1.3, 1.1
rng = np.random.default_rng(31)
X = np.asfortranarray(rng.uniform(-1, 1, (n, p)))
Z = rng.uniform(-1, 1, (n, Bz))
Z[:, 0] = (rng.random(n) < 0.5).astype(float)
Z = np.asfortranarray(Z)
y = rng.standard_normal(n)
par0 = np.concatenate([[np.log(0.3), 0.1], rng.normal(0, 0.3, Bz + 1), np.log(2.0) + rng.normal(-1.0, 0.5, (Bz + 1) * p)])


def test_points(nx, seed):
    r = np.random.default_rng(seed)
    X2 = np.asfortranarray(r.uniform(-1, 1, (nx, p)))
    z2 = (r.random(nx) < 0.4).astype(float)
    z2[0], z2[-1] = 1.0, 0.0
    Z2 = r.uniform(-1, 1, (nx, Bz))
    Z2[:, 0] = z2
    dZ2 = np.asfortranarray(r.uniform(0.5, 1.5, (nx, Bz)))
    sub = r.random((nx, 21)) < 0.5
    sub[0, :] = True
    sub[:, 0] = z2 != 0.0  # no untreated point: ATU is 0 / 0
    return X2, np.asfortranarray(Z2), dZ2, sub


def posterior(f):
    out = []
    for nx in (37, 128 * world, 2501):
        X2, Z2, dZ2, sub = test_points(nx, nx)
        out.append([f.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, False),
                    f.predict_marginal(X2, Z2, dZ2, MEAN_Y, STD_Y, STD_Z, True),
                    f.predict_marginal_batch(X2, Z2, dZ2, sub, MEAN_Y, STD_Y, STD_Z)])
    return out


def same(a, b):
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(same(a[k], b[k]) for k in a)
    if isinstance(a, list):
        return len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    return bool(np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True))


def worst(got, ref):
    """Largest error of each kind over all results, relative as in the tolerances; non-finite patterns must match."""
    w = {"points": 0.0, "avg_map": 0.0, "avg_var": 0.0, "nonfinite_match": True}

    def avg(g, r, scale):
        for k in ("ate", "att", "atu"):
            for a, b in ((g[k]["map"], r[k]["map"]), (g[k]["var"], r[k]["var"])):
                if np.isfinite(a) != np.isfinite(b) or (np.isnan(a) != np.isnan(b)):
                    w["nonfinite_match"] = False
            if np.isfinite(r[k]["map"]):
                w["avg_map"] = max(w["avg_map"], abs(g[k]["map"] - r[k]["map"]) / max(abs(r[k]["map"]), scale))
            if np.isfinite(r[k]["var"]):
                w["avg_var"] = max(w["avg_var"], abs(g[k]["var"] - r[k]["var"]) / abs(r[k]["var"]))

    for gs, rs in zip(got, ref):
        for g, r in zip(gs, rs):
            for k in ("map", "var", "ci"):
                w["points"] = max(w["points"], float(np.abs(g[k] - r[k]).max() / np.abs(r[k]).max()))
            scale = float(np.abs(r["map"]).max())
            if "ate" in r:
                avg(g, r, scale)
            for ds, dr in zip(g.get("subsets", []), r.get("subsets", [])):
                avg(ds, dr, scale)
    return w


f = AceFit(y, X, Z, par0, kernel=kernel, device=lr, use_graph=False)
f.shard(dist)
if rank == 0:
    s = AceFit(y, X, Z, par0, kernel=kernel, device=lr, use_graph=False)
    s.shard_emulate(world)
    g = AceFit(y, X, Z, par0, kernel=kernel, device=lr, use_graph=False)
for it in range(1, iters + 1):
    factored = f.parameters  # every fit factors K at these parameters (bit-identical on all ranks)
    f.para_update(it)
    if rank == 0:
        s.para_update(it)
        g.para_update(it)
        s.parameters = g.parameters = f.parameters
# predict at the parameters of the stored factor, so that C = K_m,xx - W W^T is a posterior covariance (as in
# tests/test_gpu_shard_posterior.py)
f.parameters = factored
if rank == 0:
    s.parameters = g.parameters = factored
res = posterior(f)  # collective
gathered = [None] * world
dist.all_gather_object(gathered, res)
if rank == 0:
    emu, ref = posterior(s), posterior(g)
    out = {"world": world, "n": n, "p": p, "Bz": Bz,
           "ranks_bit_identical": all(same(gathered[0], r) for r in gathered[1:]),
           "equals_emulated": same(gathered[0], emu),
           "vs_unsharded": worst(gathered[0], ref), "emulated_vs_unsharded": worst(emu, ref)}
    v = out["vs_unsharded"]
    out["ok"] = bool(out["ranks_bit_identical"] and out["equals_emulated"] and v["nonfinite_match"]
                     and v["points"] <= 1e-12 and v["avg_map"] <= 1e-12 and v["avg_var"] <= 1e-10)
    print(json.dumps(out))
    s.close()
    g.close()
f.close()
dist.barrier()
dist.destroy_process_group()
