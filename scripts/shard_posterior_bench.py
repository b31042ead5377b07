"""torchrun --nproc-per-node G scripts/shard_posterior_bench.py [out.json] : time of the marginal posterior of a sharded
fit against the unsharded fit on the same GPUs.  predict_marginal(calculate_ate = 1) and predict_marginal_batch with
S = 21 subsets (robust_treatment's n.steps + 1 sets), nx = 4096 test points, at the C4 shape (n = 65536, p = 8, Bz = 3,
SE) and the C3 shape (n = 16384, the same p, Bz and kernel).

Per call, median of 3 after one warm-up call (for a sharded fit, the slowest rank):
  - device_ms: CUDA events recorded on the fit's stream before and after the call (AceFit.timer_start / timer_stop):
    everything the call enqueues, uploads, kernels and NCCL, plus any idle time while the host allocates or waits;
  - host_ms: host clock around the call, which ends in a stream synchronise, so also the host averages;
  - peak_bytes_sampled: in one further call, the largest drop of the device's free memory (cudaMemGetInfo, polled
    from a second host thread) below its value before the call;
  - peak_bytes_counted: the call's O(nx n) and O(nx^2) buffers, counted from their shapes.
The unsharded fit runs on rank 0's GPU after the sharded fit is released.  With G = 1 the script also plays world 2,
4 and 8 on the one GPU (shard_emulate): those times are every rank's work in sequence, and time / world is labelled
as an emulated per-rank time, not a multi-GPU measurement.  The card's name, power limit and max SM clock are read
in the same run."""
import json, os, subprocess, sys, threading, time
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
NX, S, REPS = 4096, 21, 3
SHAPES = [("C3", 16384), ("C4", 65536)]


def rup(v, m=128):
    return (v + m - 1) // m * m


def peak_bytes(n, nx, G):
    """Largest buffers alive at once in one call (8-byte doubles), per rank."""
    n_pad = rup(n)
    if G == 1:  # unsharded: Kx and T (nx_pad x n_pad), the marginal K_xx / C (nx_pad x nx_pad)
        nx_pad = rup(nx)
        return 8 * (2 * nx_pad * n_pad + nx_pad * nx_pad)
    chunk = rup(-(-nx // G))
    nx_all = chunk * G  # Kx and W_r (chunk x n_pad), gathered W (nx_all x n_pad), C row block (chunk x nx_all)
    return 8 * (2 * chunk * n_pad + nx_all * n_pad + chunk * nx_all)


def inputs(prob):
    rng = np.random.default_rng(5)
    X2 = np.asfortranarray(rng.uniform(-1, 1, (NX, prob.p)))
    tb = prob.basis.testbasis(rng.choice(prob.z, NX))
    B, dB = np.asfortranarray(tb["B"]), np.asfortranarray(tb["dB"])
    sub = rng.random((NX, S)) < 0.5
    return X2, B, dB, sub


def timed(f, fn):
    fn()  # warm-up
    dev, host = [], []
    for _ in range(REPS):
        torch.cuda.synchronize()
        f.timer_start()
        t0 = time.perf_counter()
        fn()
        host.append((time.perf_counter() - t0) * 1e3)
        dev.append(f.timer_stop())
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(lr)[0]
    low, done = [free0], threading.Event()

    def poll():
        while not done.is_set():
            low[0] = min(low[0], torch.cuda.mem_get_info(lr)[0])

    th = threading.Thread(target=poll)
    th.start()
    fn()
    done.set()
    th.join()
    return {"device_ms": float(np.median(dev)), "host_ms": float(np.median(host)), "peak_bytes_sampled": free0 - low[0]}


def measure(f, prob, collective, G):
    X2, B, dB, sub = inputs(prob)
    res = {}
    for name, fn in (("ate", lambda: f.predict_marginal(X2, B, dB, prob.mean_y, prob.std_y, 1.0, True)),
                     ("batch21", lambda: f.predict_marginal_batch(X2, B, dB, sub, prob.mean_y, prob.std_y, 1.0))):
        if collective:
            dist.barrier()
        res[name] = timed(f, fn)
        res[name]["peak_bytes_counted"] = peak_bytes(prob.n, NX, G)
    return res


def fit(prob, device, G_emulate=0, shard=False):
    f = AceFit(prob.y, prob.X, prob.Z, prob.parameters, kernel=prob.kernel, std_y=prob.std_y, device=device,
               use_graph=False)
    if shard:
        f.shard(dist)
    if G_emulate > 1:
        f.shard_emulate(G_emulate)
    f.para_update(1)  # the posterior of a sharded fit is split once the factor exists
    return f


out = {"world": world, "nx": NX, "S": S, "shapes": []}
if rank == 0:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    out["gpus"] = q.stdout.strip().splitlines()
for name, n in SHAPES:
    prob = synth.make_problem("C4", n=n)
    row = {"shape": name, "n": n, "p": prob.p, "Bz": prob.Z.shape[1], "kernel": prob.kernel}
    if world > 1:
        f = fit(prob, lr, shard=True)
        mine = measure(f, prob, True, world)
        f.close()
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        row["sharded"] = {c: {k: max(r[c][k] for r in allr) for k in mine[c]} for c in mine}
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        g = fit(prob, lr)
        row["unsharded"] = measure(g, prob, False, 1)
        g.close()
        if world > 1:
            row["speedup_device"] = {c: row["unsharded"][c]["device_ms"] / row["sharded"][c]["device_ms"]
                                     for c in ("ate", "batch21")}
        else:
            row["multi_gpu_speedup"] = "not measured"
            row["emulated"] = []
            for G in (2, 4, 8):
                e = fit(prob, lr, G_emulate=G)
                t = measure(e, prob, False, G)
                e.close()
                row["emulated"].append({"world": G, "all_ranks": t,
                                        "per_rank_device_ms_emulated": {c: t[c]["device_ms"] / G for c in t}})
    dist.barrier()
    out["shapes"].append(row)
if rank == 0:
    js = json.dumps(out)
    print(js)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as fh:
            fh.write(js + "\n")
dist.barrier()
dist.destroy_process_group()
