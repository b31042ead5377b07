"""torchrun --nproc-per-node G scripts/shard_check.py [config] : one fit sharded over G GPUs vs the same fit
unsharded on rank 0's GPU -- parameters / gradients / stats must agree to rounding; prints timings."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"
import numpy as np
import torch, torch.distributed as dist
from additivecausalexpansion_b200 import synth
from additivecausalexpansion_b200.fit import AceFit

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
cfg = sys.argv[1] if len(sys.argv) > 1 else "C3"
n = int(sys.argv[2]) if len(sys.argv) > 2 else None
prob = synth.make_problem(cfg, n=n)
K = 4
with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y, device=lr, use_graph=False) as f:
    f.shard(dist)
    res = []
    for it in range(1, K + 1):
        st, gn = f.para_update(it)
        res.append((st.copy(), gn, f.parameters, f.gradients, f.last_timing_ms))
    dist.barrier(); torch.cuda.synchronize()
    f.timer_start()
    for it in range(K + 1, K + 4):
        f.para_update(it)
    ms_sh = f.timer_stop() / 3
    ph = f.last_timing_ms
    # posterior of the sharded fit (collective: the test points are blocked over the ranks)
    rng = np.random.default_rng(7)
    nx = 1000
    X2 = np.asfortranarray(rng.uniform(-1, 1, (nx, prob.p))); z2 = rng.uniform(-1, 1, nx)
    tb = prob.basis.testbasis(z2)
    torch.cuda.synchronize(); dist.barrier()
    import time as _t
    t0 = _t.time(); pred_sh = f.predict(X2, tb["B"], prob.mean_y, prob.std_y); t_pred_sh = _t.time() - t0
    # few, odd-numbered test points: some ranks receive an empty (or 8-byte-misaligned, before the fix) block
    nx_s = 37
    pred_sh_small = f.predict(X2[:nx_s].copy(order="F"), tb["B"][:nx_s].copy(order="F"), prob.mean_y, prob.std_y)
    if os.environ.get("ACE_SHARD_TRACE") and rank in (0, 1):
        from additivecausalexpansion_b200._lib import lib
        lib().ace_dbg_shard_trace_dump(rank)
# bit-identical parameters on all ranks?
par = torch.tensor(res[-1][2], device=f"cuda:{lr}")
gathered = [torch.empty_like(par) for _ in range(world)]
dist.all_gather(gathered, par)
same = all(torch.equal(gathered[0], g) for g in gathered)
if rank == 0:
    with AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y, device=lr, use_graph=False) as g:
        out = {"world": world, "config": cfg, "n": prob.n, "params_bit_identical_across_ranks": bool(same), "iters": []}
        for it in range(1, K + 1):
            st, gn = g.para_update(it)
            s2, gn2, p2, g2, _ = res[it - 1]
            out["iters"].append({"it": it, "evid_rel": abs(s2[1] - st[1]) / abs(st[1]), "rmse_rel": abs(s2[0] - st[0]) / abs(st[0]),
                                 "grad_rel": float(np.abs(g2 - g.gradients).max() / np.abs(g.gradients).max()),
                                 "par_abs": float(np.abs(p2 - g.parameters).max())})
            g.parameters = p2  # re-synchronise
        g.timer_start()
        for it in range(K + 1, K + 4):
            g.para_update(it)
        ms_1 = g.timer_stop() / 3
        t0 = _t.time(); pred_1 = g.predict(X2, tb["B"], prob.mean_y, prob.std_y); t_pred_1 = _t.time() - t0
        out["predict"] = {"nx": nx, "map_rel": float(np.abs(pred_sh["map"] - pred_1["map"]).max() / np.abs(pred_1["map"]).max()),
                          "var_rel": float(np.abs(pred_sh["var"] - pred_1["var"]).max() / np.abs(pred_1["var"]).max()),
                          "wall_s_sharded": t_pred_sh, "wall_s_single": t_pred_1}
        pred_1s = g.predict(X2[:nx_s].copy(order="F"), tb["B"][:nx_s].copy(order="F"), prob.mean_y, prob.std_y)
        out["predict_small_odd"] = {"nx": nx_s, "map_rel": float(np.abs(pred_sh_small["map"] - pred_1s["map"]).max() / np.abs(pred_1s["map"]).max()),
                                    "var_rel": float(np.abs(pred_sh_small["var"] - pred_1s["var"]).max() / np.abs(pred_1s["var"]).max())}
        out.update({"ms_per_iter_sharded": ms_sh, "ms_per_iter_single": ms_1, "speedup": ms_1 / ms_sh, "phases_sharded": ph, "phases_single": g.last_timing_ms})
    print(json.dumps(out, default=float))
dist.barrier()
dist.destroy_process_group()
