"""Cost of equality constraints in the batch QP solver: BASELINE config 4's shape (512 dense QPs, n = 512, m = 1024)
with p in {0, 1, 16, 64} rows of A x = b, through cvxopt_b200.qp_batch_distributed (as bench.py's `batch` leg).

    python tools/batch_eq_bench.py [--out FILE]                      # one GPU
    torchrun --nproc_per_node N tools/batch_eq_bench.py [--out FILE]  # N GPUs, NCCL

Per p: device-event solve ms (max over ranks), lock-step and total iterations, ms per lock-step iteration, and
scatter / gather ms.  On one GPU, also the factorisations' phases of a separate solve created with
CVXB_BATCH_PHASE_MS=1 (which synchronises after every phase, so its total is not a solve time): S (SYRK + Cholesky),
TRSM (Asct = L^{-1} A'), Kp (SYRK + Cholesky of Asct' Asct).

Problems: bench.py's make_qp(n, m, k) for problem k (the same P, q, G, h as its batch leg), and A = the next p x n
standard normal draws of the same generator, b = A x0 through its strictly feasible point x0.  Prints one JSON line and
writes it to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def make_eq_qp(n, m, pmax, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    A0 = rng.standard_normal((n, n))
    P = A0.T @ A0 / n + np.eye(n)
    q = rng.standard_normal(n)
    G = rng.standard_normal((m, n))
    x0 = rng.standard_normal(n)
    h = G @ x0 + rng.uniform(0.1, 1.1, m)
    A = rng.standard_normal((pmax, n))
    return P, q, G, h, A, A @ x0


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        return []


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--m", type=int, default=1024)
    ap.add_argument("--p", default="0,1,16,64")
    ap.add_argument("--reps", type=int, default=3, help="timed solves per p (the median is reported)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    import cvxopt_b200
    from cvxopt_b200.batch import QPBatch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl")
    rank = dist.get_rank() if world > 1 else 0
    dev = torch.device("cuda", torch.cuda.current_device())
    if cvxopt_b200.device_count() == 0:
        raise RuntimeError("no B200 visible")
    ps = [int(v) for v in args.p.split(",")]
    B, n, m, pmax = args.batch, args.n, args.m, max(ps)

    data = None
    if rank == 0:
        t0 = time.perf_counter()
        cols = [make_eq_qp(n, m, pmax, k) for k in range(B)]
        data = [np.stack([c[i] for c in cols]) for i in range(6)]
        del cols
        print("generated %d problems in %.1f s" % (B, time.perf_counter() - t0), file=sys.stderr)

    def run(p, sl=slice(None)):
        tm = {}
        if rank != 0:
            return cvxopt_b200.qp_batch_distributed(None, None, None, None, timings=tm), tm
        P, q, G, h, A, b = (a[sl] for a in data)
        eq = dict(A=A[:, :p], b=b[:, :p]) if p else {}
        return cvxopt_b200.qp_batch_distributed(P, q, G, h, timings=tm, **eq), tm

    out = {"tool": "tools/batch_eq_bench.py", "batch": B, "n": n, "m": m, "gpus": world, "gpu": gpu_info(),
           "timing": "device events per phase (max over ranks); solve_ms = the IPM on every rank's shard, ms = "
                     "scatter + solve + gather; median of %d solves" % args.reps, "results": []}
    for p in ps:
        # warm-up on a small slice (NCCL channels, first launches of this p's kernels)
        run(p, slice(0, 2 * world))
        reps = []
        for _ in range(args.reps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            res, tm = run(p)
            keys = ("scatter_ms", "solve_ms", "gather_ms")
            t = torch.tensor([tm.get(k, 0.0) for k in keys] + [float(res.get("lockstep_iterations", 0))],
                             dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            reps.append((t.tolist(), res))
        if rank != 0:
            continue
        reps.sort(key=lambda r: r[0][1])
        (sc, so, ga, lockstep), res = reps[len(reps) // 2]
        full = res["all"]
        row = {"p": p, "solve_ms": so, "scatter_ms": sc, "gather_ms": ga, "ms": sc + so + ga,
               "solve_ms_all_reps": sorted(r[0][1] for r in reps),
               "lockstep_iterations": int(lockstep), "iterations_total": int(full["iterations"].sum()),
               "ms_per_lockstep_iteration": so / max(lockstep, 1),
               "all_optimal": bool(all(s == "optimal" for s in full["status"]))}
        if p:
            P, q, G, h, A, b = data
            row["max_rel_residual_Ax_b"] = float(np.max(np.linalg.norm(
                np.einsum("bpn,bn->bp", A[:, :p], full["x"]) - b[:, :p], axis=1) /
                np.maximum(1.0, np.linalg.norm(b[:, :p], axis=1))))
        if world == 1:
            # the factorisations' phases, one sub-batch (nsub = 1), synchronising after each phase
            os.environ["CVXB_BATCH_PHASE_MS"] = "1"
            bt = QPBatch(B, n, m, 0, p=p)
            os.environ.pop("CVXB_BATCH_PHASE_MS")
            try:
                P, q, G, h, A, b = data
                bt.load(P, q, G, h, A[:, :p], b[:, :p])
                bt.solve()
                ph = bt.phase_ms()
                st = bt.stats()
            finally:
                bt.close()
            nf = st["lockstep_iterations"] + 1          # factorisations: the starting point + one per iteration
            row["factor_phases_nsub1"] = dict(ph, factorisations=nf, lockstep_iterations=st["lockstep_iterations"],
                                              per_factorisation_ms={k: v / nf for k, v in ph.items()})
        out["results"].append(row)
        print(json.dumps(row), file=sys.stderr)
    if rank == 0:
        base = out["results"][0] if out["results"] and out["results"][0]["p"] == 0 else None
        if base:
            for row in out["results"]:
                row["solve_ms_vs_p0"] = row["solve_ms"] / base["solve_ms"]
                row["ms_per_lockstep_iteration_vs_p0"] = (row["ms_per_lockstep_iteration"] /
                                                          base["ms_per_lockstep_iteration"])
        line = json.dumps(out)
        print(line)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
