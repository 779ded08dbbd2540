"""Batch of independent dense QPs solved in lock-step on the device (BASELINE config 4).

    minimize 1/2 x'P x + q'x   subject to   G x + s = h,  s in C,  A x = b     (p rows of A)

C is one 'l' cone of m rows by default.  With dims = {'l': ml, 'q': [q_1 .. q_K], 's': []} it is ml linear rows
followed by K second-order cones, the same for every problem of the batch; each problem is then solved as
coneqp(P, q, G, h, dims[, A, b]) with the reference's default options (kktsolver='chol', one step of iterative
refinement), which the batch replaces by the equivalent kkt_chol2 elimination.

The per-problem algorithm is coneprog.coneqp restricted to dims={'l': m} (reference
src/python/coneprog.py:1998-2547) — same start, stopping rule, Mehrotra steps — so every
problem converges in the same number of iterations as `solvers.qp(P, q, G, h)` does, or, with
equality constraints, as `solvers.qp(P, q, G, h, A, b)` does (its default KKT solver for this
case, kktsolver='chol2', misc.py:1352-1567).  p = 0 (no A) is the default.
The reference has no batch API; its counterpart is a Python loop over `solvers.qp`.
"""
import ctypes as C

import numpy as np

from . import _lib

STATUS = {0: "running", 1: "optimal", 2: "unknown", 3: "unknown"}
DEFAULTS = dict(maxiters=100, abstol=1e-7, reltol=1e-6, feastol=1e-7)   # coneprog.py:436-456


def _stack(P, q, G, h):
    """-> contiguous (B,n,n), (B,n), (B,n,m) [= m x n column-major per problem], (B,m)"""
    P = np.ascontiguousarray(np.asarray(P, dtype=np.float64))
    q = np.ascontiguousarray(np.asarray(q, dtype=np.float64))
    G = np.asarray(G, dtype=np.float64)
    h = np.ascontiguousarray(np.asarray(h, dtype=np.float64))
    if P.ndim != 3 or P.shape[1] != P.shape[2]:
        raise TypeError("P must have shape (B, n, n)")
    B, n = P.shape[0], P.shape[1]
    if q.shape != (B, n):
        raise TypeError("q must have shape (B, n)")
    if G.ndim != 3 or G.shape[0] != B or G.shape[2] != n:
        raise TypeError("G must have shape (B, m, n)")
    m = G.shape[1]
    if h.shape != (B, m):
        raise TypeError("h must have shape (B, m)")
    # P is symmetric: its row-major image equals its column-major image as far as tril goes
    Pcm = np.ascontiguousarray(np.transpose(P, (0, 2, 1)))
    Gcm = np.ascontiguousarray(np.transpose(G, (0, 2, 1)))      # (B, n, m): column-major m x n
    return Pcm, q, Gcm, h, B, n, m


def _stack_eq(A, b, B, n):
    """-> contiguous (B,n,p) [= p x n column-major per problem], (B,p); (B,n,0), (B,0) without A"""
    if A is None and b is None:
        return np.zeros((B, n, 0)), np.zeros((B, 0)), 0
    if A is None or b is None:
        raise TypeError("A and b must be given together")
    A = np.asarray(A, dtype=np.float64)
    b = np.ascontiguousarray(np.asarray(b, dtype=np.float64))
    if A.ndim != 3 or A.shape[0] != B or A.shape[2] != n:
        raise TypeError("A must have shape (B, p, n)")
    p = A.shape[1]
    if b.shape != (B, p):
        raise TypeError("b must have shape (B, p)")
    return np.ascontiguousarray(np.transpose(A, (0, 2, 1))), b, p


def _check_dims(dims, m):
    """-> (ml, [q_1 .. q_K]) of a cone dimension dict for G with m rows; dims=None is {'l': m, 'q': [], 's': []}.
    Raises TypeError for malformed dims, 's' cones (not supported by the batch) or sizes that do not add up to m."""
    if dims is None:
        return int(m), []
    if not isinstance(dims, dict):
        raise TypeError("dims must be a dict with keys 'l', 'q', 's'")
    ml, ql, sl = dims.get("l", 0), list(dims.get("q", [])), list(dims.get("s", []))
    ints = (int, np.integer)
    if not isinstance(ml, ints) or isinstance(ml, bool) or ml < 0:
        raise TypeError("dims['l'] must be a nonnegative integer")
    if any(not isinstance(k, ints) or isinstance(k, bool) or k < 1 for k in ql):
        raise TypeError("dims['q'] must be a list of positive integers")
    if sl:
        raise TypeError("the batch solver has no 's' cones: dims['s'] must be empty")
    if int(ml) + sum(int(k) for k in ql) != m:
        raise TypeError("dims: l + sum(q) = %d, but G and h have %d rows" % (int(ml) + sum(int(k) for k in ql), m))
    return int(ml), [int(k) for k in ql]


def _refinement(options):
    """options['refinement'] as the library takes it: -1 for the reference's default rule"""
    r = options.get("refinement")
    if r is None:
        return -1
    if not isinstance(r, (int, np.integer)) or isinstance(r, bool) or r < 0:
        raise ValueError("options['refinement'] must be a nonnegative integer")
    return int(r)


class QPBatch:
    def __init__(self, nprob, n, m, device=0, p=0, dims=None):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        self.B, self.n, self.m, self.p = int(nprob), int(n), int(m), int(p)
        self.ml, self.qdims = _check_dims(dims, self.m)
        qarr = (C.c_int * max(1, len(self.qdims)))(*self.qdims)
        _lib.check(self._lib.cvxb_batch_create_cones(C.byref(self._h), self.B, self.n, self.ml, len(self.qdims),
                                                     qarr, self.p, device), "batch")

    def load(self, P, q, G, h, A=None, b=None):
        Pcm, q, Gcm, h, B, n, m = _stack(P, q, G, h)
        if (B, n, m) != (self.B, self.n, self.m):
            raise TypeError("problem shapes do not match the batch")
        Acm, b, p = _stack_eq(A, b, B, n)
        if p != self.p:
            raise TypeError("A has %d rows, the batch was created with p = %d" % (p, self.p))
        rc = self._lib.cvxb_batch_load(self._h, Pcm.ctypes.data, q.ctypes.data, Gcm.ctypes.data,
                                       h.ctypes.data, _lib.HOST)
        _lib.check(rc, "batch_load")
        _lib.check(self._lib.cvxb_batch_load_eq(self._h, Acm.ctypes.data, b.ctypes.data, _lib.HOST), "batch_load_eq")

    def load_ptr(self, P, q, G, h, space=_lib.DEVICE, A=None, b=None):
        """raw addresses of already laid-out buffers (device-resident callers); A (p x n column-major per
        problem) and b are required when p > 0"""
        _lib.check(self._lib.cvxb_batch_load(self._h, P, q, G, h, space), "batch_load")
        if self.p > 0 and (not A or not b):
            raise TypeError("A and b are required: the batch was created with p = %d" % self.p)
        _lib.check(self._lib.cvxb_batch_load_eq(self._h, A, b, space), "batch_load_eq")

    def solve(self, **options):
        """options as coneqp's: maxiters, abstol, reltol, feastol, refinement (default: 1 with 'q' cones, else 0)"""
        o = dict(DEFAULTS)
        o.update(options)
        rc = self._lib.cvxb_batch_solve_ref(self._h, int(o["maxiters"]), float(o["abstol"]),
                                            float(o["reltol"]), float(o["feastol"]), _refinement(o))
        if rc == _lib.E_ARG and "Rank(" in _lib.last_error():
            raise ValueError(_lib.last_error())       # coneprog.py:2065-2067
        _lib.check(rc, "batch_solve")

    def results(self):
        B, n, m = self.B, self.n, self.m
        x, s, z = np.zeros((B, n)), np.zeros((B, m)), np.zeros((B, m))
        y = np.zeros((B, self.p))
        status = np.zeros(B, dtype=np.int32)
        iters = np.zeros(B, dtype=np.int32)
        pobj, dobj = np.zeros(B), np.zeros(B)
        rc = self._lib.cvxb_batch_results(self._h, x.ctypes.data, s.ctypes.data, z.ctypes.data,
                                          status.ctypes.data, iters.ctypes.data, pobj.ctypes.data,
                                          dobj.ctypes.data, _lib.HOST)
        _lib.check(rc, "batch_results")
        _lib.check(self._lib.cvxb_batch_results_y(self._h, y.ctypes.data, _lib.HOST), "batch_results_y")
        return {"x": x, "y": y, "s": s, "z": z, "status": [STATUS[int(k)] for k in status],
                "status_code": status, "iterations": iters, "primal objective": pobj,
                "dual objective": dobj}

    def singular(self):
        """per problem: True where S = P + G'G was singular at the starting point, so that S + A'A is factored
        (the reference's kkt_chol2 'singular' branch)"""
        flags = np.zeros(self.B, dtype=np.int32)
        _lib.check(self._lib.cvxb_batch_singular(self._h, flags.ctypes.data), "batch_singular")
        return flags.astype(bool)

    def phase_ms(self):
        """factorisation time of the last solve by phase (batch created with CVXB_BATCH_PHASE_MS=1)"""
        ms = (C.c_double * 3)()
        _lib.check(self._lib.cvxb_batch_phase_ms(self._h, ms), "batch_phase_ms")
        out = {"S_syrk_potrf_ms": ms[0], "trsm_ms": ms[1], "Kp_syrk_potrf_ms": ms[2]}
        if self.qdims:
            mq = (C.c_double * 2)()
            _lib.check(self._lib.cvxb_batch_phase_ms_cones(self._h, mq), "batch_phase_ms_cones")
            out.update({"Gs_q_scale_ms": mq[0], "Gs_q_gemm_ms": mq[1]})       # both inside S_syrk_potrf_ms
        return out

    def stats(self):
        ms, it = C.c_double(), C.c_int()
        self._lib.cvxb_batch_stats(self._h, C.byref(ms), C.byref(it))
        return {"solve_ms": ms.value, "lockstep_iterations": it.value,
                "syrk_path": ("none", "dmma", "int8")[self._lib.cvxb_batch_syrk_path(self._h)]}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.cvxb_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _split(n, parts):
    base, extra = divmod(n, parts)
    out, lo = [], 0
    for r in range(parts):
        hi = lo + base + (1 if r < extra else 0)
        out.append((lo, hi))
        lo = hi
    return out


class QPBatchGroup:
    """`nsub` QPBatch objects over interleaved slices of one batch, solved CONCURRENTLY on their own CUDA streams
    (one host thread each; ctypes releases the GIL inside the library calls).  A lock-step batch alternates
    throughput-bound phases (batched SYRK / GEMV) with latency-bound ones (the chain of diagonal-block
    factorisations, the flag-chained triangular solves); with two or more sub-batches in flight the GPU runs one
    sub-batch's latency-bound phase under another's throughput-bound phase, and a sub-batch stops iterating as soon
    as ITS slowest problem is done.  Interleaved slices (problem i -> sub-batch i mod nsub) spread hard and easy
    problems evenly."""

    def __init__(self, nprob, n, m, device=0, nsub=None, p=0, dims=None):
        if nsub is None:
            # measured on B200 (profiles/r02h_batch_nsub.txt, n=512 m=1024): 512 problems 148 -> 142 ms with 2
            # sub-batches; 64 problems 25.0 -> 21.3 ms with 8
            nsub = int(__import__("os").environ.get("CVXB_BATCH_NSUB", "0")) or (
                2 if nprob >= 256 else (max(1, min(8, nprob // 8)) if nprob >= 16 else 1))
        self.nsub = max(1, min(int(nsub), nprob))
        self.B, self.n, self.m, self.p = int(nprob), int(n), int(m), int(p)
        self.idx = [np.arange(r, self.B, self.nsub) for r in range(self.nsub)]
        _check_dims(dims, self.m)
        self.parts = [QPBatch(len(ix), n, m, device, p, dims) for ix in self.idx]

    def load_ptr_sliced(self, loader):
        """loader(part_index, indices, QPBatch) loads one sub-batch (device-resident callers)"""
        for r, (ix, b) in enumerate(zip(self.idx, self.parts)):
            loader(r, ix, b)

    def load(self, P, q, G, h, A=None, b=None):
        P, q, G, h = (np.asarray(a) for a in (P, q, G, h))
        if A is not None:
            A = np.asarray(A)
        if b is not None:
            b = np.asarray(b)
        for ix, part in zip(self.idx, self.parts):
            part.load(P[ix], q[ix], G[ix], h[ix], None if A is None else A[ix], None if b is None else b[ix])

    def solve(self, **options):
        if self.nsub == 1:
            self.parts[0].solve(**options)
            return
        import threading
        errs = []

        def run(b):
            try:
                b.solve(**options)
            except BaseException as e:      # noqa: BLE001  re-raised on the calling thread
                errs.append(e)
        th = [threading.Thread(target=run, args=(b,)) for b in self.parts]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]

    def results(self):
        B, n, m = self.B, self.n, self.m
        out = {"x": np.zeros((B, n)), "y": np.zeros((B, self.p)), "s": np.zeros((B, m)), "z": np.zeros((B, m)),
               "status_code": np.zeros(B, dtype=np.int32), "iterations": np.zeros(B, dtype=np.int32),
               "primal objective": np.zeros(B), "dual objective": np.zeros(B)}
        for ix, b in zip(self.idx, self.parts):
            r = b.results()
            for key in out:
                out[key][ix] = r[key]
        out["status"] = [STATUS[int(k)] for k in out["status_code"]]
        return out

    def singular(self):
        out = np.zeros(self.B, dtype=bool)
        for ix, b in zip(self.idx, self.parts):
            out[ix] = b.singular()
        return out

    def stats(self):
        st = [b.stats() for b in self.parts]
        return {"solve_ms": max(s["solve_ms"] for s in st),
                "lockstep_iterations": max(s["lockstep_iterations"] for s in st),
                "lockstep_iterations_per_subbatch": [s["lockstep_iterations"] for s in st],
                "syrk_path": st[0]["syrk_path"], "nsub": self.nsub}

    def close(self):
        for b in self.parts:
            b.close()


def qp_batch(P, q, G, h, A=None, b=None, device=0, nsub=None, dims=None, **options):
    """Solve B independent dense QPs on one GPU.  P (B,n,n), q (B,n), G (B,m,n), h (B,m), and optionally
    equality constraints A (B,p,n), b (B,p) as in solvers.qp(P, q, G, h, A, b).
    dims: the cone of G x + s = h, {'l': ml, 'q': [q_1 .. q_K], 's': []}, shared by all problems (default: 'l' only);
    s and z are returned in its order, 'l' rows then the cones.  Options: maxiters, abstol, reltol, feastol and
    refinement, as coneqp's.
    nsub: number of concurrently solved sub-batches (QPBatchGroup); default 4 (1 for tiny batches)."""
    P = np.asarray(P)
    G = np.asarray(G)
    if G.ndim != 3:
        raise TypeError("G must have shape (B, m, n)")
    _check_dims(dims, G.shape[1])
    _refinement(options)
    p = 0 if A is None else np.asarray(A).shape[1]
    grp = QPBatchGroup(P.shape[0], P.shape[1], G.shape[1], device, nsub, p, dims)
    try:
        grp.load(P, q, G, h, A, b)
        import time
        t0 = time.perf_counter()
        grp.solve(**options)
        wall = (time.perf_counter() - t0) * 1e3
        out = grp.results()
        out.update(grp.stats())
        out["solve_wall_ms"] = wall
        return out
    finally:
        grp.close()


# ---------------------------------------------------------------------------------------
# multi-GPU: problems are independent -> shard them across ranks, no data-path collective.
# One scatter of (P, q, G, h[, A, b]) from rank 0, one gather of (x, s, z[, y], status, iters, objectives):
# point-to-point send/recv groups over the process group (NCCL over NVLink on GPUs: ncclSend/ncclRecv
# inside one group call; gloo in the CPU tests), exact shard sizes, nothing padded, and on GPUs nothing
# bounces through the host: shards land in device memory and QPBatch loads them from there.

def shard_bounds(nprob, world):
    """contiguous block partition: rank r owns [lo, hi)"""
    base, extra = divmod(nprob, world)
    bounds, lo = [], 0
    for r in range(world):
        hi = lo + base + (1 if r < extra else 0)
        bounds.append((lo, hi))
        lo = hi
    return bounds


def shard_indices(nprob, world, mode="interleaved"):
    """problem indices owned by each rank.  'interleaved': i -> rank i mod world (SURVEY.md §8e; spreads
    hard and easy problems evenly, which matters because a rank's lock-step loop runs until its slowest
    problem is done); 'contiguous': blocks (shard_bounds)."""
    if mode == "contiguous":
        return [np.arange(lo, hi) for lo, hi in shard_bounds(nprob, world)]
    return [np.arange(r, nprob, world) for r in range(world)]


def _p2p(ops):
    import torch.distributed as dist
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()


def qp_batch_distributed(P, q, G, h, solver=None, group=None, sharding="interleaved", timings=None,
                         nsub=None, A=None, b=None, dims=None, **options):
    """Rank 0 passes the full batch (other ranks pass None); every rank returns its shard's results and
    rank 0 additionally gets the gathered batch, in the original problem order, under key 'all'.
    Equality constraints A (B,p,n), b (B,p) are optional (rank 0 only); `solver` (a stand-in for the
    device solver) is then called as solver(P, q, G, h, A, b).  dims (rank 0's) is the cone of every problem, as
    in qp_batch; with 'q' cones the stand-in is called with dims= as well.

    `timings` (dict, optional) receives scatter_ms / solve_ms / gather_ms of this rank, measured with
    device events on the current stream (wall clock on CPU)."""
    import time
    import torch
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        on_gpu = dist.get_backend(group) == "nccl"
    else:                                   # no process group: a one-rank "world", same code path
        rank, world, on_gpu = 0, 1, torch.cuda.is_available()
    dev = torch.device("cuda", torch.cuda.current_device()) if on_gpu else torch.device("cpu")
    f64 = torch.float64

    class _Clock:
        def __init__(self):
            self.t = {}
            self._open = None

        def start(self, name):
            if on_gpu:
                e = torch.cuda.Event(enable_timing=True); e.record()
            else:
                e = time.perf_counter()
            self._open = (name, e)

        def stop(self):
            name, e0 = self._open
            if on_gpu:
                e1 = torch.cuda.Event(enable_timing=True); e1.record(); e1.synchronize()
                self.t[name] = e0.elapsed_time(e1)
            else:
                self.t[name] = (time.perf_counter() - e0) * 1e3
    clk = _Clock()

    meta = torch.zeros(6, dtype=torch.int64, device=dev)
    full = None
    qlist = []
    if rank == 0:
        # the batch in the layout QPBatch loads: column-major n x n / m x n / p x n per problem
        Pcm, qh, Gcm, hh, Btot, n, m = _stack(P, q, G, h)
        Acm, bh, p = _stack_eq(A, b, Btot, n)
        ml, qlist = _check_dims(dims, m)
        _refinement(options)
        meta = torch.tensor([Btot, n, m, p, ml, len(qlist)], dtype=torch.int64, device=dev)
        full = [torch.from_numpy(a).to(dev) for a in ((Pcm, qh, Gcm, hh) + ((Acm, bh) if p else ()))]  # one H2D
    if world > 1:
        dist.broadcast(meta, 0, group=group)
    Btot, n, m, p, ml, nq = (int(v) for v in meta.tolist())
    if nq and world > 1:                    # the cone sizes: one more broadcast, only with 'q' cones
        qt = torch.tensor(qlist, dtype=torch.int64, device=dev) if rank == 0 else \
            torch.zeros(nq, dtype=torch.int64, device=dev)
        dist.broadcast(qt, 0, group=group)
        qlist = [int(v) for v in qt.tolist()]
    dims = {"l": ml, "q": qlist, "s": []}
    owners = shard_indices(Btot, world, sharding)
    mine = owners[rank]
    k = len(mine)
    tails = [(n, n), (n,), (n, m), (m,)] + ([(n, p), (p,)] if p else [])

    # ---- setup (not data path): this rank's batch object = its device allocations ----
    local_dev = torch.cuda.current_device() if on_gpu else 0
    clk.start("setup_ms")
    bobj = QPBatchGroup(k, n, m, local_dev, nsub, p, dims) if (solver is None and k) else None
    clk.stop()

    # ---- scatter ----
    if on_gpu:
        torch.cuda.synchronize()
    clk.start("scatter_ms")
    if rank == 0:
        ops, keep = [], []
        shard = None
        for r in range(world):
            idx = torch.from_numpy(owners[r]).to(dev)
            parts = [t.index_select(0, idx) for t in full]            # contiguous copy of rank r's problems
            if r == 0:
                shard = parts
            elif len(owners[r]):
                keep.append(parts)
                ops += [dist.P2POp(dist.isend, t, r, group) for t in parts]
        _p2p(ops)
        del keep, full
    else:
        shard = [torch.empty((k,) + t, dtype=f64, device=dev) for t in tails]
        if k:
            _p2p([dist.P2POp(dist.irecv, t, 0, group) for t in shard])
    clk.stop()

    # ---- solve ----
    clk.start("solve_ms")
    if solver is not None:
        # stand-in (CPU tests): numpy in the public (B, m, n) / (B, p, n) layout
        sh = [t.cpu().numpy() for t in shard]
        args = [np.transpose(sh[0], (0, 2, 1)), sh[1], np.transpose(sh[2], (0, 2, 1)), sh[3]]
        if p:
            args += [np.transpose(sh[4], (0, 2, 1)), sh[5]]
        res = (solver(*args, dims=dims) if nq else solver(*args)) if k else None

        def rows(key, d):
            if not k or not d:
                return torch.empty((k, d), dtype=f64, device=dev)
            return torch.from_numpy(np.ascontiguousarray(res[key], dtype=np.float64)).to(dev)
        xs, ss, zs, ys = rows("x", n), rows("s", m), rows("z", m), rows("y", p)
        sc = torch.zeros((k, 4), dtype=f64, device=dev)
        if k:
            for j, key in enumerate(("status_code", "iterations", "primal objective", "dual objective")):
                sc[:, j] = torch.from_numpy(np.asarray(res[key], dtype=np.float64))
        stats = {}
    else:
        xs = torch.empty((k, n), dtype=f64, device=dev)
        ss = torch.empty((k, m), dtype=f64, device=dev)
        zs = torch.empty((k, m), dtype=f64, device=dev)
        ys = torch.empty((k, p), dtype=f64, device=dev)
        sc = torch.zeros((k, 4), dtype=f64, device=dev)
        stats = {}
        if k:
            grp = bobj
            try:
                # shards are already in device memory: straight into the sub-batches, no host bounce
                keepalive = []

                def loader(r, ix, part):
                    it = torch.from_numpy(ix).to(dev)
                    sl = [t.index_select(0, it) for t in shard] if grp.nsub > 1 else shard
                    keepalive.append(sl)
                    # the library copies on the sub-batch's own stream: the slices (written on torch's current
                    # stream) must be complete before it reads them
                    torch.cuda.current_stream().synchronize()
                    eq = dict(A=sl[4].data_ptr(), b=sl[5].data_ptr()) if p else {}
                    part.load_ptr(sl[0].data_ptr(), sl[1].data_ptr(), sl[2].data_ptr(), sl[3].data_ptr(), _lib.DEVICE,
                                  **eq)
                tw = time.perf_counter()
                grp.load_ptr_sliced(loader)
                del keepalive
                clk.t["solve_load_wall_ms"] = (time.perf_counter() - tw) * 1e3
                tw = time.perf_counter()
                grp.solve(**options)
                clk.t["solve_ipm_wall_ms"] = (time.perf_counter() - tw) * 1e3
                tw = time.perf_counter()
                for ix, part in zip(grp.idx, grp.parts):
                    kk = len(ix)
                    it = torch.from_numpy(ix).to(dev)
                    px = torch.empty((kk, n), dtype=f64, device=dev)
                    ps = torch.empty((kk, m), dtype=f64, device=dev)
                    pz = torch.empty((kk, m), dtype=f64, device=dev)
                    py = torch.empty((kk, p), dtype=f64, device=dev)
                    status = np.zeros(kk, dtype=np.int32); iters = np.zeros(kk, dtype=np.int32)
                    pobj, dobj = np.zeros(kk), np.zeros(kk)
                    lib = part._lib
                    torch.cuda.current_stream().synchronize()     # px/ps/pz may reuse blocks with work still queued
                    _lib.check(lib.cvxb_batch_results(part._h, px.data_ptr(), ps.data_ptr(), pz.data_ptr(), None, None,
                                                      None, None, _lib.DEVICE), "batch_results")
                    _lib.check(lib.cvxb_batch_results(part._h, None, None, None, status.ctypes.data, iters.ctypes.data,
                                                      pobj.ctypes.data, dobj.ctypes.data, _lib.HOST), "batch_results")
                    if p:
                        _lib.check(lib.cvxb_batch_results_y(part._h, py.data_ptr(), _lib.DEVICE), "batch_results_y")
                        ys.index_copy_(0, it, py)
                    xs.index_copy_(0, it, px); ss.index_copy_(0, it, ps); zs.index_copy_(0, it, pz)
                    sc.index_copy_(0, it, torch.from_numpy(np.stack(
                        [status.astype(np.float64), iters.astype(np.float64), pobj, dobj], axis=1)).to(dev))
                stats = grp.stats()
                torch.cuda.synchronize()
                clk.t["solve_collect_wall_ms"] = (time.perf_counter() - tw) * 1e3
            except BaseException:
                grp.close()
                raise
    del shard
    clk.stop()

    # ---- gather ----
    clk.start("gather_ms")
    local = [xs, ss, zs, sc] + ([ys] if p else [])
    widths = (n, m, m, 4) + ((p,) if p else ())
    gathered = None
    if rank == 0:
        outs = [torch.empty((Btot, d), dtype=f64, device=dev) for d in widths]
        ops, bufs = [], {}
        for r in range(1, world):
            kr = len(owners[r])
            if kr:
                bufs[r] = [torch.empty((kr, d), dtype=f64, device=dev) for d in widths]
                ops += [dist.P2POp(dist.irecv, t, r, group) for t in bufs[r]]
        _p2p(ops)
        bufs[0] = local
        for r, parts in bufs.items():
            idx = torch.from_numpy(owners[r]).to(dev)
            for o, t in zip(outs, parts):
                o.index_copy_(0, idx, t)
        gathered = [o.cpu().numpy() for o in outs]
    elif k:
        _p2p([dist.P2POp(dist.isend, t, 0, group) for t in local])
    clk.stop()
    if bobj is not None:
        bobj.close()          # device frees (tens of ms for GBs of buffers) stay outside the timed phases
    if timings is not None:
        timings.update(clk.t)

    scn = sc.cpu().numpy()
    res = {"x": xs.cpu().numpy(), "y": ys.cpu().numpy(), "s": ss.cpu().numpy(), "z": zs.cpu().numpy(),
           "status_code": scn[:, 0].astype(np.int32), "iterations": scn[:, 1].astype(np.int32),
           "primal objective": scn[:, 2].copy(), "dual objective": scn[:, 3].copy(), "indices": mine}
    res.update(stats)
    res["status"] = [STATUS[int(c)] for c in res["status_code"]]
    if rank == 0:
        g = gathered
        res["all"] = {"x": g[0], "y": g[4] if p else np.zeros((Btot, 0)), "s": g[1], "z": g[2],
                      "status_code": g[3][:, 0].astype(np.int64),
                      "iterations": g[3][:, 1].astype(np.int64), "primal objective": g[3][:, 2].copy(),
                      "dual objective": g[3][:, 3].copy(),
                      "status": [STATUS[int(c)] for c in g[3][:, 0]]}
    return res
