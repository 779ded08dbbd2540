"""Batch / device-resident IPM (BASELINE config 4) vs the reference: a Python loop over solvers.qp on the same
problems (its stored results, tests/reference_results.py) — same status, same iteration count per problem, objectives
to rtol 1e-8, x to 1e-6."""
import numpy as np
import pytest

from problems import dense_qp

pytestmark = pytest.mark.gpu


def make_batch(B, n, m, seed0=0):
    Ps, qs, Gs, hs = [], [], [], []
    for k in range(B):
        P, q, G, h = dense_qp(n, m, seed=seed0 + k)
        Ps.append(P); qs.append(q); Gs.append(G); hs.append(h)
    return np.stack(Ps), np.stack(qs), np.stack(Gs), np.stack(hs)


def ref_loop(P, q, G, h):
    from cvxopt import matrix, solvers
    out = {}
    for k in range(P.shape[0]):
        sol = solvers.qp(matrix(P[k]), matrix(q[k]), matrix(G[k]), matrix(h[k]), kktsolver="chol")
        out.update({"%d.%s" % (k, key): sol[key] for key in ("status", "iterations", "primal objective",
                                                               "dual objective", "x", "s", "z")})
    return out


@pytest.mark.parametrize("B,n,m", [(5, 30, 70), (3, 150, 321), (2, 257, 300), (1, 300, 640)])
def test_batch_matches_reference_loop(ref_golden, B, n, m):
    import cvxopt_b200
    P, q, G, h = make_batch(B, n, m, seed0=10 * B)
    ref = ref_golden("qp_loop", lambda: ref_loop(P, q, G, h))
    want = [{key.split(".", 1)[1]: v for key, v in ref.items() if key.split(".", 1)[0] == str(k)} for k in range(B)]
    got = cvxopt_b200.qp_batch(P, q, G, h)
    for k in range(B):
        assert got["status"][k] == want[k]["status"] == "optimal"
        assert got["iterations"][k] == want[k]["iterations"], (k, got["iterations"], want[k]["iterations"])
        np.testing.assert_allclose(got["primal objective"][k], want[k]["primal objective"], rtol=1e-8)
        np.testing.assert_allclose(got["dual objective"][k], want[k]["dual objective"], rtol=1e-8)
        np.testing.assert_allclose(got["x"][k], np.array(want[k]["x"]).ravel(), rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(got["s"][k], np.array(want[k]["s"]).ravel(), rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(got["z"][k], np.array(want[k]["z"]).ravel(), rtol=1e-5, atol=1e-7)


def test_batch_mixed_difficulty_masks():
    """problems converge at different iterations: early finishers must stay frozen"""
    import cvxopt_b200
    P, q, G, h = make_batch(4, 40, 90, seed0=3)
    h[1] *= 50.0          # different scaling -> different iteration counts
    q[2] *= 1e-3
    got = cvxopt_b200.qp_batch(P, q, G, h)
    assert all(s == "optimal" for s in got["status"])
    for k in range(4):
        single = cvxopt_b200.qp_batch(P[k:k + 1], q[k:k + 1], G[k:k + 1], h[k:k + 1])
        assert single["iterations"][0] == got["iterations"][k]
        np.testing.assert_allclose(single["x"][0], got["x"][k], rtol=1e-9, atol=1e-12)


def test_batch_rank_deficient_raises():
    import cvxopt_b200
    n, m = 20, 5
    P = np.zeros((1, n, n))
    q = np.ones((1, n))
    G = np.random.default_rng(0).standard_normal((1, m, n))
    h = np.ones((1, m))
    with pytest.raises(ValueError):
        cvxopt_b200.qp_batch(P, q, G, h)


def test_concurrent_subbatches_match_single_batch():
    """QPBatchGroup: interleaved sub-batches solved concurrently on their own streams give the same per-problem
    results as one lock-step batch"""
    import cvxopt_b200
    P, q, G, h = make_batch(7, 60, 130, seed0=40)
    one = cvxopt_b200.qp_batch(P, q, G, h, nsub=1)
    three = cvxopt_b200.qp_batch(P, q, G, h, nsub=3)
    assert three["nsub"] == 3 and one["nsub"] == 1
    assert list(one["iterations"]) == list(three["iterations"])
    assert all(s == "optimal" for s in three["status"])
    np.testing.assert_allclose(three["x"], one["x"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(three["primal objective"], one["primal objective"], rtol=1e-12)


def test_distributed_entry_single_process_matches_qp_batch():
    """qp_batch_distributed without a process group (the bench's N=1 leg): device-side slicing into concurrent
    sub-batches must give exactly qp_batch's per-problem results.  Sized so that the slices are ~100 MB each: the
    library's copies run on the sub-batches' own streams and once raced with the torch kernels that write the
    slices (stale blocks of the caching allocator held OTHER problems' data: every solve still 'optimal', wrong
    iteration counts)."""
    import torch
    import cvxopt_b200
    B, n, m = 96, 192, 384
    P, q, G, h = make_batch(B, n, m, seed0=300)
    want = cvxopt_b200.qp_batch(P, q, G, h, nsub=2)
    for rep in range(3):
        # churn the caching allocator so that freed blocks hold unrelated problem data
        junk = [torch.randn(B * m * n // 2, dtype=torch.float64, device="cuda") for _ in range(3)]
        del junk
        tm = {}
        got = cvxopt_b200.qp_batch_distributed(P, q, G, h, nsub=2, timings=tm)["all"]
        assert list(got["iterations"]) == list(want["iterations"])
        np.testing.assert_allclose(got["x"], want["x"], rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(got["primal objective"], want["primal objective"], rtol=1e-12)
        assert set(tm) >= {"setup_ms", "scatter_ms", "solve_ms", "gather_ms"}


def test_compaction_of_finished_problems(monkeypatch):
    """The lock-step loop swaps finished problems out of the active prefix (csrc/batch_ipm.cu): per-problem results
    are those of the uncompacted loop, come back in the caller's order, and a second solve on the same loaded batch
    (slots restored first) repeats them."""
    import cvxopt_b200
    from cvxopt_b200.batch import QPBatch
    B, n, m = 24, 40, 90
    P, q, G, h = make_batch(B, n, m, seed0=500)
    # mixed difficulty: scale some problems so that iteration counts differ
    for k in range(0, B, 3):
        q[k] *= 1e3
        h[k] *= 1e-2
    monkeypatch.setenv("CVXB_BATCH_COMPACT", "0")
    plain = cvxopt_b200.qp_batch(P, q, G, h, nsub=1)
    monkeypatch.setenv("CVXB_BATCH_COMPACT", "1")
    b = QPBatch(B, n, m, 0)
    try:
        b.load(P, q, G, h)
        b.solve()
        r1 = b.results()
        b.solve()
        r2 = b.results()
    finally:
        b.close()
    assert len(set(plain["iterations"])) > 1          # the test needs problems that finish at different iterations
    for r in (r1, r2):
        assert list(r["iterations"]) == list(plain["iterations"])
        assert list(r["status_code"]) == list(plain["status_code"])
        np.testing.assert_array_equal(r["x"], plain["x"])
        np.testing.assert_array_equal(r["z"], plain["z"])
        np.testing.assert_array_equal(r["primal objective"], plain["primal objective"])
