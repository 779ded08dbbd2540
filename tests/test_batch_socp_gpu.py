"""Batch QP solver with second-order cone constraints vs the reference: a Python loop over
solvers.coneqp(P, q, G, h, dims[, A, b]) with its default options (kktsolver='chol', one step of iterative
refinement) on the same problems (its stored results, tests/reference_results.py).  Same status and iteration count
per problem, objectives to rtol 1e-8, x and y to 1e-6, s and z to 1e-5."""
import numpy as np
import pytest

from problems import cone_point

pytestmark = pytest.mark.gpu


def socp_qp(n, dims, p, seed):
    """P = A0'A0/n + I, G random, h = G x0 + s0 with s0 strictly inside the cones; p rows of A x = b through x0"""
    rng = np.random.Generator(np.random.PCG64(seed))
    m = dims["l"] + sum(dims["q"])
    A0 = rng.standard_normal((n, n))
    P = A0.T @ A0 / n + np.eye(n)
    q = rng.standard_normal(n)
    G = rng.standard_normal((m, n))
    x0 = rng.standard_normal(n)
    h = G @ x0 + cone_point(dict(dims, s=[]), rng)
    A = rng.standard_normal((p, n))
    return P, q, G, h, A, A @ x0


def singular_S_socp(n, dims, k, seed):
    """P zero on the last k coordinates, G with zero columns there, p = k rows of A that are generic on them:
    P + G'W^-1 W^-T G is singular, [P; A; G] has rank n"""
    P, q, G, h, A, b = socp_qp(n, dims, k, seed)
    rng = np.random.Generator(np.random.PCG64(seed + 1000))
    x0 = rng.standard_normal(n)
    P[-k:, :] = 0.0
    P[:, -k:] = 0.0
    G[:, -k:] = 0.0
    h = G @ x0 + cone_point(dict(dims, s=[]), rng)
    return P, q, G, h, A, A @ x0


def make_batch(B, n, dims, p, seed0=0, singular=()):
    probs = [singular_S_socp(n, dims, p, seed0 + k) if k in singular else socp_qp(n, dims, p, seed0 + k)
             for k in range(B)]
    return tuple(np.stack([pr[i] for pr in probs]) for i in range(6))


def ref_loop(P, q, G, h, A, b, dims, options=None):
    from cvxopt import matrix, solvers
    out = {}
    kw = {} if options is None else {"options": dict(options, show_progress=False)}
    for k in range(P.shape[0]):
        eq = (matrix(A[k]), matrix(b[k])) if A.shape[1] else ()
        sol = solvers.coneqp(matrix(P[k]), matrix(q[k]), matrix(G[k]), matrix(h[k]),
                             {"l": dims["l"], "q": list(dims["q"]), "s": []}, *eq, **kw)
        out.update({"%d.%s" % (k, key): sol[key] for key in ("status", "iterations", "primal objective",
                                                               "dual objective", "x", "y", "s", "z")})
    return out


def per_problem(ref, B):
    return [{key.split(".", 1)[1]: v for key, v in ref.items() if key.split(".", 1)[0] == str(k)} for k in range(B)]


def assert_matches(got, want, B):
    for k in range(B):
        assert got["status"][k] == want[k]["status"] == "optimal", k
        assert got["iterations"][k] == want[k]["iterations"], (k, got["iterations"], want[k]["iterations"])
        np.testing.assert_allclose(got["primal objective"][k], want[k]["primal objective"], rtol=1e-8)
        np.testing.assert_allclose(got["dual objective"][k], want[k]["dual objective"], rtol=1e-8)
        np.testing.assert_allclose(got["x"][k], np.array(want[k]["x"]).ravel(), rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(got["y"][k], np.array(want[k]["y"]).ravel(), rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(got["s"][k], np.array(want[k]["s"]).ravel(), rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(got["z"][k], np.array(want[k]["z"]).ravel(), rtol=1e-5, atol=1e-7)


# (B, n, ml, q, p): tiny cones next to 'l' rows; a few mid-size cones alone; many cones with equality constraints;
# one cone of size n + 1; n not a multiple of the tile size; cones of size 1 and 2
SHAPES = [(4, 30, 20, [3] * 10, 0), (3, 40, 0, [17, 40, 5], 0), (3, 80, 100, [4] * 50, 12),
          (3, 60, 0, [61], 0), (2, 257, 300, [8] * 40, 40), (3, 8, 5, [1, 2, 3], 0)]


@pytest.mark.parametrize("B,n,ml,qd,p", SHAPES)
def test_batch_socp_matches_reference_loop(ref_golden, B, n, ml, qd, p):
    import cvxopt_b200
    dims = {"l": ml, "q": qd, "s": []}
    P, q, G, h, A, b = make_batch(B, n, dims, p, seed0=100 + 10 * B + p + ml)
    want = per_problem(ref_golden("coneqp_loop", lambda: ref_loop(P, q, G, h, A, b, dims)), B)
    got = cvxopt_b200.qp_batch(P, q, G, h, A if p else None, b if p else None, dims=dims)
    assert got["s"].shape == (B, ml + sum(qd)) and got["y"].shape == (B, p)
    assert_matches(got, want, B)


@pytest.mark.parametrize("B,n,ml,qd,p", [SHAPES[0], SHAPES[2], SHAPES[3]])
def test_batch_socp_without_refinement(ref_golden, B, n, ml, qd, p):
    import cvxopt_b200
    dims = {"l": ml, "q": qd, "s": []}
    P, q, G, h, A, b = make_batch(B, n, dims, p, seed0=300 + 10 * B + p + ml)
    want = per_problem(ref_golden("coneqp_loop_refinement0",
                                  lambda: ref_loop(P, q, G, h, A, b, dims, {"refinement": 0})), B)
    got = cvxopt_b200.qp_batch(P, q, G, h, A if p else None, b if p else None, dims=dims, refinement=0)
    assert_matches(got, want, B)


def test_l_only_dims_and_refinement(ref_golden):
    """explicit 'l'-only dims are the call without dims, bit for bit; refinement=1 follows the reference's"""
    import cvxopt_b200
    B, n, m, p = 4, 40, 90, 3
    dims = {"l": m, "q": [], "s": []}
    P, q, G, h, A, b = make_batch(B, n, dims, p, seed0=60)
    want = per_problem(ref_golden("coneqp_loop_refinement1",
                                  lambda: ref_loop(P, q, G, h, A, b, dims, {"refinement": 1})), B)
    old = cvxopt_b200.qp_batch(P, q, G, h, A, b)
    new = cvxopt_b200.qp_batch(P, q, G, h, A, b, dims=dims)
    assert list(new["iterations"]) == list(old["iterations"])
    for key in ("x", "y", "s", "z", "primal objective", "dual objective"):
        np.testing.assert_array_equal(new[key], old[key])
    got = cvxopt_b200.qp_batch(P, q, G, h, A, b, dims=dims, refinement=1)
    assert_matches(got, want, B)


def test_compaction_with_cones(monkeypatch):
    """problems of very different difficulty finish at different iterations: the finished ones leave the active
    prefix with v and beta of their cones; results are those of the uncompacted loop, in the caller's order, and
    a second solve repeats them.  Problems 4 and 13 take kkt_chol2's singular-S branch.  (p is even: with an odd p
    the GEMVs with A' pick their vectorised kernel by the batch count when a single problem is left active, which
    changes the last bits of that problem's iterates.)"""
    import cvxopt_b200
    from cvxopt_b200.batch import QPBatch
    B, n, p = 24, 40, 6
    dims = {"l": 30, "q": [3] * 8 + [12], "s": []}
    m = 30 + 36
    P, q, G, h, A, b = make_batch(B, n, dims, p, seed0=500, singular=(4, 13))
    for k in range(0, B, 3):
        q[k] *= 1e3
        h[k] *= 1e-2
        b[k] *= 1e-2
    monkeypatch.setenv("CVXB_BATCH_COMPACT", "0")
    plain = cvxopt_b200.qp_batch(P, q, G, h, A, b, nsub=1, dims=dims)
    monkeypatch.setenv("CVXB_BATCH_COMPACT", "1")
    bt = QPBatch(B, n, m, 0, p=p, dims=dims)
    try:
        bt.load(P, q, G, h, A, b)
        bt.solve()
        r1 = bt.results()
        f1 = bt.singular()
        bt.solve()
        r2 = bt.results()
        f2 = bt.singular()
    finally:
        bt.close()
    assert len(set(plain["iterations"])) > 1
    assert all(s == "optimal" for s in plain["status"])
    for r, f in ((r1, f1), (r2, f2)):
        assert list(f) == [k in (4, 13) for k in range(B)]
        assert list(r["iterations"]) == list(plain["iterations"])
        assert list(r["status_code"]) == list(plain["status_code"])
        for key in ("x", "y", "s", "z", "primal objective", "dual objective"):
            np.testing.assert_array_equal(r[key], plain[key])


def test_subbatches_and_distributed_entry_with_cones():
    import cvxopt_b200
    B, n, p = 7, 50, 4
    dims = {"l": 40, "q": [5] * 6 + [30], "s": []}
    P, q, G, h, A, b = make_batch(B, n, dims, p, seed0=40, singular=(3,))
    one = cvxopt_b200.qp_batch(P, q, G, h, A, b, nsub=1, dims=dims)
    three = cvxopt_b200.qp_batch(P, q, G, h, A, b, nsub=3, dims=dims)
    assert three["nsub"] == 3
    assert all(s == "optimal" for s in one["status"])
    assert list(one["iterations"]) == list(three["iterations"])
    for key in ("x", "y", "s", "z", "primal objective"):
        np.testing.assert_allclose(three[key], one[key], rtol=1e-12, atol=1e-12)
    dist = cvxopt_b200.qp_batch_distributed(P, q, G, h, A=A, b=b, nsub=1, dims=dims)["all"]
    assert list(dist["iterations"]) == list(one["iterations"])
    for key in ("x", "y", "s", "z", "primal objective", "dual objective"):
        np.testing.assert_allclose(dist[key], one[key], rtol=1e-12, atol=1e-12)


def test_int8_syrk_path_with_cones(ref_golden, monkeypatch):
    """B = 1 with the int8-slice SYRK forced: it serves the 'l' rows, the DMMA GEMM adds the cones' rows"""
    from cvxopt_b200.batch import QPBatch
    n, p = 200, 8
    dims = {"l": 300, "q": [6] * 20 + [50], "s": []}
    m = 300 + 170
    P, q, G, h, A, b = make_batch(1, n, dims, p, seed0=900)
    want = per_problem(ref_golden("coneqp_loop", lambda: ref_loop(P, q, G, h, A, b, dims)), 1)
    monkeypatch.setenv("CVXB_OZAKI", "2")
    bt = QPBatch(1, n, m, 0, p=p, dims=dims)
    try:
        bt.load(P, q, G, h, A, b)
        bt.solve()
        got = bt.results()
        assert bt.stats()["syrk_path"] == "int8"
    finally:
        bt.close()
    assert_matches(got, want, 1)


def test_rank_deficient_raises_with_cones():
    import cvxopt_b200
    dims = {"l": 10, "q": [4, 4], "s": []}
    P, q, G, h, A, b = make_batch(2, 20, dims, 3, seed0=90, singular=(0,))
    A[0, :, -1] = 0.0                      # the last coordinate is in no row of [P; A; G]
    with pytest.raises(ValueError, match="Rank"):
        cvxopt_b200.qp_batch(P, q, G, h, A, b, dims=dims)


@pytest.mark.parametrize("dims", [{"l": 10, "q": [4], "s": [2]}, {"l": 10, "q": [4, 0], "s": []},
                                  {"l": 10, "q": [5], "s": []}, {"l": -1, "q": [19], "s": []}])
def test_malformed_dims_raise_before_device_work(dims, monkeypatch):
    import cvxopt_b200
    from cvxopt_b200 import batch
    P, q, G, h, _, _ = make_batch(2, 12, {"l": 10, "q": [4, 4], "s": []}, 0, seed0=7)

    def no_device(*a, **k):
        raise AssertionError("device work started")
    monkeypatch.setattr(batch, "QPBatch", no_device)
    with pytest.raises(TypeError):
        cvxopt_b200.qp_batch(P, q, G, h, dims=dims)
