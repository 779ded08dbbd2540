"""world_size-2 gloo test (CPU) of the multi-GPU batch path with equality constraints A x = b: A and b are
scattered with the other operands, y is gathered with the iterates, and both come back in problem order.  The
per-rank solver is a stand-in that solves the equality-constrained QP with the inequalities ignored, in closed form:

    [ P  A' ] [ x ]   [ -q ]
    [ A  0  ] [ y ] = [  b ]."""
import os
import socket

import numpy as np
import pytest


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _standin_solver(P, q, G, h, A, b):
    B, n = q.shape
    p = b.shape[1]
    xs, ys = np.zeros((B, n)), np.zeros((B, p))
    for k in range(B):
        K = np.block([[P[k], A[k].T], [A[k], np.zeros((p, p))]])
        sol = np.linalg.solve(K, np.concatenate([-q[k], b[k]]))
        xs[k], ys[k] = sol[:n], sol[n:]
    s = h - np.einsum("bmn,bn->bm", G, xs)
    obj = 0.5 * np.einsum("bn,bnk,bk->b", xs, P, xs) + np.einsum("bn,bn->b", q, xs)
    return {"x": xs, "y": ys, "s": s, "z": np.zeros_like(s), "status_code": np.ones(B, np.int32),
            "iterations": np.arange(B, dtype=np.int32), "primal objective": obj, "dual objective": obj}


def _problems(nprob, n=6, m=9, p=2):
    rng = np.random.default_rng(11)
    F = rng.standard_normal((nprob, n, n))
    P = np.einsum("bij,bkj->bik", F, F) + np.eye(n)
    q = rng.standard_normal((nprob, n))
    G = rng.standard_normal((nprob, m, n))
    h = 100.0 + rng.standard_normal((nprob, m))
    A = rng.standard_normal((nprob, p, n))
    b = rng.standard_normal((nprob, p))
    return P, q, G, h, A, b


def _worker(rank, world, port, nprob, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from cvxopt_b200.batch import qp_batch_distributed
    P, q, G, h, A, b = _problems(nprob)
    if rank == 0:
        res = qp_batch_distributed(P, q, G, h, solver=_standin_solver, A=A, b=b)
    else:
        res = qp_batch_distributed(None, None, None, None, solver=_standin_solver)
    # this rank's shard: its own problems, in the order of res["indices"]
    mine = res["indices"]
    want = _standin_solver(*(a[mine] for a in (P, q, G, h, A, b)))
    ret["shard%d" % rank] = bool(np.allclose(res["x"], want["x"]) and np.allclose(res["y"], want["y"]))
    if rank == 0:
        want = _standin_solver(P, q, G, h, A, b)
        got = res["all"]
        ret["ok"] = bool(got["y"].shape == (nprob, 2) and np.allclose(got["x"], want["x"])
                         and np.allclose(got["y"], want["y"]) and np.allclose(got["s"], want["s"])
                         and np.allclose(got["primal objective"], want["primal objective"])
                         and len(got["status"]) == nprob)
    dist.destroy_process_group()


@pytest.mark.parametrize("nprob", [7, 2, 1])
def test_scatter_solve_gather_with_equality_constraints_gloo(nprob):
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


def test_standin_satisfies_the_kkt_system():
    """the stand-in itself: A x = b and P x + q + A'y = 0"""
    P, q, G, h, A, b = _problems(3)
    r = _standin_solver(P, q, G, h, A, b)
    np.testing.assert_allclose(np.einsum("bpn,bn->bp", A, r["x"]), b, atol=1e-10)
    np.testing.assert_allclose(np.einsum("bij,bj->bi", P, r["x"]) + q + np.einsum("bpn,bp->bn", A, r["y"]), 0,
                               atol=1e-10)


def test_equality_argument_validation():
    from cvxopt_b200.batch import _stack_eq
    with pytest.raises(TypeError):
        _stack_eq(np.zeros((2, 1, 3)), None, 2, 3)
    with pytest.raises(TypeError):
        _stack_eq(np.zeros((2, 1, 4)), np.zeros((2, 1)), 2, 3)
    with pytest.raises(TypeError):
        _stack_eq(np.zeros((2, 1, 3)), np.zeros((2, 2)), 2, 3)
    Acm, b, p = _stack_eq(np.arange(12.0).reshape(2, 2, 3), np.zeros((2, 2)), 2, 3)
    assert p == 2 and Acm.shape == (2, 3, 2) and Acm[1, 2, 1] == 11.0      # p x n column-major per problem
    assert _stack_eq(None, None, 2, 3)[2] == 0
