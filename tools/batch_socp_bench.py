"""Cost of second-order cones in the batch QP solver: BASELINE config 4's shape (512 dense QPs, n = 512, m = 1024) with
the m rows of G split into cones in five ways, through cvxopt_b200.qp_batch_distributed (as bench.py's `batch` leg).

    python tools/batch_socp_bench.py [--out FILE]                      # one GPU
    torchrun --nproc_per_node N tools/batch_socp_bench.py [--out FILE]  # N GPUs, NCCL

Cases: 'l' only;  ml = 512 + 64 cones of 8;  256 cones of 4;  8 cones of 128;  one cone of 1024 (the cone kernels'
three group sizes: a thread, a warp and the whole CTA per cone).  Per case: device-event solve ms (max
over ranks), lock-step and total iterations, ms per lock-step iteration, scatter / gather ms.  On one GPU, also the
factorisations' phases of a separate solve created with CVXB_BATCH_PHASE_MS=1 (which synchronises after every phase,
so its total is not a solve time): S (all of it: SYRK of the 'l' rows, the cones' rows, Cholesky) and, inside it,
the scaling Gs_q = W^{-T} G_q and the GEMM K += Gs_q' Gs_q.

Problems: P = A0'A0/n + I, q, G standard normal, h = G x0 + s0 with s0 strictly inside the cones (tests/problems.py's
cone_point), from numpy's PCG64(k) for problem k.  Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for d in (ROOT, os.path.join(ROOT, "tests")):
    if d not in sys.path:
        sys.path.insert(0, d)

CASES = {"l_only": None,
         "l512_q8x64": {"l": 512, "q": [8] * 64, "s": []},
         "q4x256": {"l": 0, "q": [4] * 256, "s": []},
         "q128x8": {"l": 0, "q": [128] * 8, "s": []},
         "q1024x1": {"l": 0, "q": [1024], "s": []}}


def make_socp_qp(n, m, dims, seed):
    from problems import cone_point
    rng = np.random.Generator(np.random.PCG64(seed))
    A0 = rng.standard_normal((n, n))
    P = A0.T @ A0 / n + np.eye(n)
    q = rng.standard_normal(n)
    G = rng.standard_normal((m, n))
    x0 = rng.standard_normal(n)
    h = G @ x0 + cone_point(dims or {"l": m, "q": [], "s": []}, rng)
    return P, q, G, h


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
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--reps", type=int, default=3, help="timed solves per case (the median is reported)")
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
    B, n = args.batch, args.n
    cases = args.cases.split(",")
    m = 1024
    for c in cases:
        d = CASES[c]
        if d is not None and d["l"] + sum(d["q"]) != m:
            raise SystemExit("case %s does not have m = %d rows" % (c, m))

    out = {"tool": "tools/batch_socp_bench.py", "batch": B, "n": n, "m": m, "gpus": world, "gpu": gpu_info(),
           "timing": "device events per phase (max over ranks); solve_ms = the IPM on every rank's shard, ms = "
                     "scatter + solve + gather; median of %d solves" % args.reps, "results": []}
    for case in cases:
        dims = CASES[case]
        data = None
        if rank == 0:
            t0 = time.perf_counter()
            cols = [make_socp_qp(n, m, dims, k) for k in range(B)]
            data = [np.stack([c[i] for c in cols]) for i in range(4)]
            del cols
            print("%s: generated %d problems in %.1f s" % (case, B, time.perf_counter() - t0), file=sys.stderr)

        def run(sl=slice(None)):
            tm = {}
            if rank != 0:
                return cvxopt_b200.qp_batch_distributed(None, None, None, None, timings=tm), tm
            P, q, G, h = (a[sl] for a in data)
            return cvxopt_b200.qp_batch_distributed(P, q, G, h, timings=tm, dims=dims), tm

        run(slice(0, 2 * world))        # warm-up on a small slice (NCCL channels, first launches)
        reps = []
        for _ in range(args.reps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            res, tm = run()
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
        row = {"case": case, "dims": dims and {"l": dims["l"], "q": "%d x %d" % (len(dims["q"]), dims["q"][0])},
               "solve_ms": so, "scatter_ms": sc, "gather_ms": ga, "ms": sc + so + ga,
               "solve_ms_all_reps": sorted(r[0][1] for r in reps),
               "lockstep_iterations": int(lockstep), "iterations_total": int(full["iterations"].sum()),
               "ms_per_lockstep_iteration": so / max(lockstep, 1),
               "all_optimal": bool(all(s == "optimal" for s in full["status"]))}
        if world == 1:
            # the factorisations' phases, one sub-batch (nsub = 1), synchronising after each phase
            os.environ["CVXB_BATCH_PHASE_MS"] = "1"
            bt = QPBatch(B, n, m, 0, dims=dims)
            os.environ.pop("CVXB_BATCH_PHASE_MS")
            try:
                bt.load(*data)
                bt.solve()
                ph = bt.phase_ms()
                st = bt.stats()
            finally:
                bt.close()
            nf = st["lockstep_iterations"] + 1          # factorisations: the starting point + one per iteration
            ph.pop("trsm_ms", None)
            ph.pop("Kp_syrk_potrf_ms", None)
            row["factor_phases_nsub1"] = dict(ph, factorisations=nf, lockstep_iterations=st["lockstep_iterations"],
                                              per_factorisation_ms={k: v / nf for k, v in ph.items()})
        out["results"].append(row)
        print(json.dumps(row), file=sys.stderr)
        del data
    if rank == 0:
        base = out["results"][0] if out["results"] and out["results"][0]["case"] == "l_only" else None
        if base:
            for row in out["results"]:
                row["solve_ms_vs_l_only"] = row["solve_ms"] / base["solve_ms"]
                row["ms_per_lockstep_iteration_vs_l_only"] = (row["ms_per_lockstep_iteration"] /
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
