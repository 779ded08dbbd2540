"""world_size-2 gloo test (CPU) of the multi-GPU batch path with second-order cones: rank 0's dims reach every
rank, and s and z (rows in dims order: 'l', then the cones) come back in problem order.  The per-rank solver is a
stand-in that records the dims it was given and returns rows that identify the problem and the cone of every row."""
import os
import socket

import numpy as np
import pytest

DIMS = {"l": 3, "q": [2, 4, 1], "s": []}


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _standin_solver(P, q, G, h, dims):
    """x = q, s = h, z[j] = index of the cone of row j (0 for 'l' rows) + 10 * h[j]"""
    B, n = q.shape
    cone = np.concatenate([np.zeros(dims["l"])] + [np.full(k, i + 1.0) for i, k in enumerate(dims["q"])])
    return {"x": q.copy(), "y": np.zeros((B, 0)), "s": h.copy(), "z": cone[None, :] + 10.0 * h,
            "status_code": np.ones(B, np.int32), "iterations": np.full(B, len(dims["q"]), np.int32),
            "primal objective": h.sum(axis=1), "dual objective": h.sum(axis=1)}


def _problems(nprob, n=5):
    m = DIMS["l"] + sum(DIMS["q"])
    rng = np.random.default_rng(5)
    P = np.broadcast_to(np.eye(n), (nprob, n, n)).copy()
    q = rng.standard_normal((nprob, n))
    G = rng.standard_normal((nprob, m, n))
    h = np.arange(nprob * m, dtype=np.float64).reshape(nprob, m)
    return P, q, G, h


def _worker(rank, world, port, nprob, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from cvxopt_b200.batch import qp_batch_distributed
    seen = []

    def solver(P, q, G, h, dims):
        seen.append(dims)
        return _standin_solver(P, q, G, h, dims)
    P, q, G, h = _problems(nprob)
    if rank == 0:
        res = qp_batch_distributed(P, q, G, h, solver=solver, dims=DIMS)
    else:
        res = qp_batch_distributed(None, None, None, None, solver=solver)
    mine = res["indices"]
    want = _standin_solver(P[mine], q[mine], G[mine], h[mine], DIMS)
    ret["dims%d" % rank] = [(d["l"], list(d["q"]), list(d["s"])) for d in seen]
    ret["shard%d" % rank] = bool(np.array_equal(res["z"], want["z"]) and np.array_equal(res["s"], want["s"]))
    if rank == 0:
        want = _standin_solver(P, q, G, h, DIMS)
        got = res["all"]
        ret["ok"] = bool(np.array_equal(got["s"], want["s"]) and np.array_equal(got["z"], want["z"])
                         and np.array_equal(got["x"], want["x"]) and list(got["iterations"]) == [3] * nprob)
    dist.destroy_process_group()


@pytest.mark.parametrize("nprob", [5, 2])
def test_scatter_solve_gather_with_cones_gloo(nprob):
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    port = _free_port()
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, 2, port, nprob, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert ret["ok"]
    assert ret["shard0"] and ret["shard1"]
    assert ret["dims0"] == ret["dims1"] == [(3, [2, 4, 1], [])]


def test_dims_validation():
    from cvxopt_b200.batch import _check_dims
    assert _check_dims(None, 7) == (7, [])
    assert _check_dims({"l": 3, "q": [2, 4, 1], "s": []}, 10) == (3, [2, 4, 1])
    assert _check_dims({"l": 0, "q": [np.int64(5)], "s": []}, 5) == (0, [5])
    for bad in ({"l": 3, "q": [2, 4, 1], "s": [2]},          # 's' cones
                {"l": 3, "q": [2, 0, 5], "s": []},           # q_k < 1
                {"l": 3, "q": [2, 4], "s": []},              # l + sum(q) != m
                {"l": -1, "q": [11], "s": []},
                {"l": 2.0, "q": [8], "s": []},
                [3, [7]]):
        with pytest.raises(TypeError):
            _check_dims(bad, 10)


def test_refinement_option_validation():
    from cvxopt_b200.batch import _refinement
    assert _refinement({}) == -1
    assert _refinement({"refinement": 0}) == 0
    assert _refinement({"refinement": 2}) == 2
    for bad in (-1, 1.0, "1", True):
        with pytest.raises(ValueError):
            _refinement({"refinement": bad})
