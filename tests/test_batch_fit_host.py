"""Host side of the batched fit, no GPU: argument checks of AceFitBatch and ace_train_batch (they fail before any
device call), the contiguous split of run_batched_restarts, and its gather with a stub batch under gloo, world 2."""
import os
import socket

import numpy as np
import pytest
import torch.multiprocessing as mp

from additivecausalexpansion_b200 import restarts
from additivecausalexpansion_b200.fit import AceFitBatch
from additivecausalexpansion_b200.kernel import ace_train_batch


def test_batch_argument_checks():
    y, X, Z = np.zeros((3, 10)), np.zeros((3, 10, 2)), np.zeros((3, 10, 1))
    with pytest.raises(ValueError, match="S x P"):
        AceFitBatch(y, X, Z, np.zeros(8))
    with pytest.raises(ValueError, match="columns"):
        AceFitBatch(y, X, Z, np.zeros((3, 7)))
    with pytest.raises(ValueError, match="members"):
        AceFitBatch(y[:2], X, Z, np.zeros((3, 8)))
    with pytest.raises(ValueError, match="observations"):
        AceFitBatch(y, X[:, :9], Z, np.zeros((3, 8)))
    with pytest.raises(ValueError, match="kernel"):
        AceFitBatch(y, X, Z, np.zeros((3, 8)), kernel="RBF")
    with pytest.raises(ValueError, match="std_y"):
        AceFitBatch(y, X, Z, np.zeros((3, 8)), std_y=np.ones(2))


def test_train_batch_argument_checks():
    rng = np.random.default_rng(0)
    with pytest.raises(ValueError, match="same number"):
        ace_train_batch([rng.standard_normal(20)], [], [])
    # different knot counts per member (a binary treatment gets the binary basis): refused before any device call
    n = 40
    ys = [rng.standard_normal(n), rng.standard_normal(n)]
    Xs = [rng.standard_normal((n, 2)), rng.standard_normal((n, 2))]
    Zs = [rng.standard_normal(n), (rng.random(n) < 0.5).astype(float)]
    with pytest.raises(ValueError, match="basis dimension"):
        ace_train_batch(ys, Xs, Zs, basis="cubic", n_knots=3)


def test_assign_contiguous():
    assert restarts.assign_contiguous(8, 3) == [[0, 1, 2], [3, 4, 5], [6, 7]]
    assert restarts.assign_contiguous(2, 4) == [[0], [1], [], []]
    assert sorted(i for part in restarts.assign_contiguous(65, 8) for i in part) == list(range(65))
    with pytest.raises(ValueError):
        restarts.assign_contiguous(3, 0)


def _stub_batch(idx):
    return [{"evidence": -100.0 + (i * 37 % 11), "iters": 10 + i} for i in idx]


def test_run_batched_restarts_single_process():
    res = restarts.run_batched_restarts(5, _stub_batch)
    assert [r["fit"] for r in res] == list(range(5)) and all(r["rank"] == 0 for r in res)
    assert restarts.best_restart(res)["fit"] == max(range(5), key=lambda i: -100.0 + (i * 37 % 11))
    with pytest.raises(RuntimeError):
        restarts.run_batched_restarts(3, lambda idx: [{}])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    res = restarts.run_batched_restarts(7, _stub_batch, dist)
    q.put((rank, [(r["fit"], r["rank"], r["evidence"]) for r in res], restarts.best_restart(res)["fit"]))
    dist.destroy_process_group()


def test_run_batched_restarts_gloo_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    ref = None
    for rank, res, best in got:
        assert [f for f, _, _ in res] == list(range(7))
        assert all(rk == (0 if f < 4 else 1) for f, rk, _ in res)  # contiguous shares [0..3], [4..6]
        assert best == max(range(7), key=lambda i: -100.0 + (i * 37 % 11))
        ref = ref or res
        assert res == ref
