#!/usr/bin/env python
"""bench.py — KKT factor+solve throughput of the cone-program hot path on B200.

A "step" is one interior-point iteration's KKT work on the north-star workload
(dense QP n=8192, m=2n 'l' cone rows): 1 factor (NT scaling fused into the
normal-equations SYRK + Cholesky) and 2 solves (affine + combined direction;
coneqp with refinement 0, reference src/python/coneprog.py:2256, 2360-2401).

  value  : algorithmic GF/s (F_it / step time, SURVEY.md §8d) with every input resident
           in HBM, timed with CUDA events on the library's launch stream.
  e2e    : the same metric through the public plugin call a CVXOPT user makes
           (cvxopt_b200.kkt_chol -> factor(W) -> solve(x,y,z)) with pinned HOST buffers;
           H2D/D2H copies inside the timed region.
  --impl reference : the unmodified reference path (oracle/_ref: cvxopt's misc.kkt_chol +
           OpenBLAS) on the box's host cores, same workload and metric.

N > 1 GPUs: a single factorisation does not shard (DESIGN.md §multi-GPU) -> N independent
replicas, one per rank, weak scaling; value = total flops / max-over-ranks time.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "kkt_factor_solve_gflops_fp64"
INT8_TENSOR_NOMINAL_TOPS = 4500.0   # nominal dense int8 (B200): used only if no measured value is committed
FP64_DMMA_PEAK_TFLOPS = 37.2   # tools/fp64_peak.cu on this pool's B200 (profiles/r01_fp64_peak_dmma_dfma.txt)


def measured_constants():
    """numbers measured on this pool's B200s by committed tools (tools/int8_peak.cu, ncu captures), kept in
    profiles/measured_constants.json together with their sources"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "measured_constants.json")))
    except Exception:       # noqa: BLE001
        return {}


def workload(n, m):
    """the one workload string both arms print (config.workload)"""
    return "dense QP KKT step n=%d m=%d ('l' cone): 1 factor + 2 solves (kkt_chol)" % (n, m)


def flops(n, m, refinement=0):
    f_fac = float(n) * n * m + float(n) ** 3 / 3.0          # SYRK n^2 Kp + POTRF n^3/3
    f_sol = 4.0 * m * n + 2.0 * float(n) * n
    return f_fac, f_sol, f_fac + 2 * (1 + refinement) * f_sol


def make_problem(n, m, seed):
    """SURVEY.md §8(d) dense QP generator (numpy PCG64)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    A0 = rng.standard_normal((n, n))
    P = np.asfortranarray(A0.T @ A0 / n + np.eye(n))
    del A0
    G = np.asfortranarray(rng.standard_normal((n, m)).T)     # m x n, column-major
    # mid-IPM scaling: d spans ~4 decades
    d = 10.0 ** rng.uniform(-2.0, 2.0, m)
    return P, G, d, rng


def make_qp(n, m, seed):
    """full dense QP (SURVEY.md §8d): P, q, G, h with a strictly feasible point"""
    rng = np.random.Generator(np.random.PCG64(seed))
    A0 = rng.standard_normal((n, n))
    P = A0.T @ A0 / n + np.eye(n)
    del A0
    q = rng.standard_normal(n)
    G = rng.standard_normal((m, n))
    x0 = rng.standard_normal(n)
    h = G @ x0 + rng.uniform(0.1, 1.1, m)
    return P, q, G, h


def run_ipm(n, m, seed, device):
    """whole interior-point solve of one dense QP, device resident (cvxopt_b200.QPBatch, B=1)"""
    import cvxopt_b200
    P, q, G, h = make_qp(n, m, seed)
    b = cvxopt_b200.QPBatch(1, n, m, device)
    b.load(P[None], q[None], G[None], h[None])
    b.solve()                      # warm-up (first-launch overheads, clocks)
    t0 = time.perf_counter()
    b.solve()
    wall = (time.perf_counter() - t0) * 1e3
    r, st = b.results(), b.stats()
    b.close()
    it = int(r["iterations"][0])
    f_fac, f_sol, f_it = flops(n, m)
    return {"n": n, "m": m, "iterations": it, "status": r["status"][0], "ms_total": st["solve_ms"],
            "syrk_path": st["syrk_path"],
            "wall_ms": wall, "iters_per_s": (it + 1) / (st["solve_ms"] * 1e-3),
            "primal_objective": float(r["primal objective"][0]),
            "gflops": (it + 1) * f_it / (st["solve_ms"] * 1e-3) * 1e-9}


def run_batch_distributed(nprob, n, m, rank, world, dev):
    """BASELINE config 4 through cvxopt_b200.qp_batch_distributed: rank 0 holds every problem; timed region =
    scatter (NCCL send/recv groups from rank 0's device copy) + solve + gather (NCCL), max over ranks."""
    import torch
    import torch.distributed as dist
    import cvxopt_b200
    args = (None, None, None, None)
    if rank == 0:
        P, q, G, h = (np.empty((nprob, n, n)), np.empty((nprob, n)), np.empty((nprob, m, n)), np.empty((nprob, m)))
        for k in range(nprob):
            P[k], q[k], G[k], h[k] = make_qp(n, m, k)
        args = (P, q, G, h)
    # warm-up on a small slice: NCCL point-to-point channels, kernels' first launches
    warm = tuple(a[: 2 * world] for a in args) if rank == 0 else args
    cvxopt_b200.qp_batch_distributed(*warm)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    tm = {}
    t0 = time.perf_counter()
    res = cvxopt_b200.qp_batch_distributed(*args, timings=tm)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    keys = ("scatter_ms", "solve_ms", "gather_ms")
    sub = ("solve_load_wall_ms", "solve_ipm_wall_ms", "solve_collect_wall_ms")
    t = torch.tensor([tm[k] for k in keys] + [sum(tm[k] for k in keys), res.get("solve_ms", 0.0), wall] +
                     [tm.get(k, 0.0) for k in sub], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    full = res["all"]
    total = float(t[3].item())
    bf = flops(n, m)[2]
    its = int(full["iterations"].sum())
    return {"workload": "%d independent dense QPs n=%d m=%d held by rank 0: NCCL scatter -> device IPM on %d GPU(s) "
                        "(interleaved shards) -> NCCL gather" % (nprob, n, m, world),
            "scatter_ms": float(t[0].item()), "solve_ms": float(t[1].item()), "gather_ms": float(t[2].item()),
            "ms": total, "ipm_kernel_ms": float(t[4].item()), "wall_ms_incl_h2d_of_batch": float(t[5].item()),
            "solve_phase_wall_ms": {"load_shards_into_subbatches": float(t[6].item()), "ipm": float(t[7].item()),
                                    "collect_results": float(t[8].item())},
            "timing": "device events per phase, max over ranks; ms = scatter + solve + gather; the one-off H2D of "
                      "the 3.2 GB batch on rank 0 is outside (wall_ms includes it)",
            "scattered_bytes": int(8 * (nprob - len(res["indices"])) * (n * n + n + m * n + m)),
            "problems_per_s": nprob / (total * 1e-3), "ipm_iterations_total": its,
            "gflops": (its + nprob) * bf / (total * 1e-3) * 1e-9,
            "all_optimal": bool(all(x == "optimal" for x in full["status"])), "scaling": "strong"}


def run_e2e_driver(n, m, seed, device):
    """What a CVXOPT user sees: the UNMODIFIED reference driver solvers.qp (oracle/_ref acting as the host
    application) at BASELINE config 2, (a) with this library's kktsolver and matrix-valued P, G (residual GEMVs
    on the host), (b) with kktsolver + device-backed G/P operators.  Host Python glue included."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "cvxopt")):
        return {"unavailable": "oracle/_ref not built"}
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import cvxopt_b200
    from cvxopt import matrix, solvers
    solvers.options["show_progress"] = False
    P, q, G, h = make_qp(n, m, seed)
    Pm, qm, Gm, hm = matrix(P), matrix(q), matrix(G), matrix(h)
    dims = {"l": m, "q": [], "s": []}
    f = cvxopt_b200.kkt_chol(Gm, dims, None, H=Pm, device=device)
    out = {"workload": "solvers.coneqp dense QP n=%d m=%d through the unmodified reference driver" % (n, m)}

    def Gop(u, v, alpha=1.0, beta=0.0, trans="N"):
        f.G(u, v, alpha, beta, trans)

    def Pop(u, v, alpha=1.0, beta=0.0):
        f.P(u, v, alpha, beta)
    for name, (Pa, Ga) in (("plugin", (Pm, Gm)), ("plugin_and_operators", (Pop, Gop))):
        solvers.coneqp(Pa, qm, Ga, hm, dims, kktsolver=lambda W: f(W))         # warm-up
        t0 = time.perf_counter()
        sol = solvers.coneqp(Pa, qm, Ga, hm, dims, kktsolver=lambda W: f(W))
        dt = time.perf_counter() - t0
        out[name] = {"seconds": dt, "iterations": int(sol["iterations"]), "status": sol["status"],
                     "ms_per_iteration": dt / (sol["iterations"] + 1) * 1e3,
                     "iters_per_s": (sol["iterations"] + 1) / dt,
                     "primal_objective": float(sol["primal objective"])}
    f.close()
    return out


def run_e2e_cones(device):
    """BASELINE configs 3 and 5 as whole solves: (a) through the UNMODIFIED reference driver (solvers.conelp from
    oracle/_ref) with every device piece plugged in, (b) through the device-resident restatement cvxopt_b200.conelp.
    (a): kktsolver (Cholesky route), and misc.compute_scaling /
    misc.update_scaling swapped for the device versions (NT scaling of the 'q' / 's' cones, Jacobi SVD).
    Reference numbers beside it: tests/golden/config_runs.json (the reference's own kktsolver='chol' runs)."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "cvxopt")):
        return {"unavailable": "oracle/_ref not built"}
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cvxopt_b200
    from cvxopt import matrix, misc, solvers
    from problems import cone_lp
    solvers.options["show_progress"] = False
    try:
        gold = json.load(open(os.path.join(ROOT, "tests", "golden", "config_runs.json")))
    except Exception:       # noqa: BLE001
        gold = {}
    out = {}
    for name, n, dims in (("cfg3_socp", 2048, {"l": 0, "q": [64] * 64, "s": []}),
                          ("cfg5_sdp", 512, {"l": 0, "q": [], "s": [512]})):
        c, G, h = cone_lp(n, dims, seed=11)
        cm, Gm, hm = matrix(c), matrix(G), matrix(h)
        f = cvxopt_b200.kkt_chol(Gm, dims, device=device)
        res = {}
        for mode in ("kktsolver", "kktsolver_and_device_scaling"):
            saved = misc.compute_scaling, misc.update_scaling
            if mode != "kktsolver":
                misc.compute_scaling = lambda s, z, lmbda, dims, mnl=None: cvxopt_b200.scaling.compute_scaling(
                    s, z, lmbda, dims, mnl, new_matrix=lambda r, cc: matrix(0.0, (r, cc)))
                misc.update_scaling = cvxopt_b200.scaling.update_scaling
            try:
                f.reset()
                t0 = time.perf_counter()
                sol = solvers.conelp(cm, Gm, hm, dims, kktsolver=lambda W: f(W))
                dt = time.perf_counter() - t0
            finally:
                misc.compute_scaling, misc.update_scaling = saved
            res[mode] = {"seconds": dt, "iterations": int(sol["iterations"]), "status": sol["status"],
                         "iters_per_s": (sol["iterations"] + 1) / dt,
                         "primal_objective": float(sol["primal objective"])}
        f.close()
        # the device-resident driver (cvxopt_b200.conelp): all iterates in HBM, scalars only over PCIe; the time
        # includes uploading G (1.07 GB for config 5)
        cvxopt_b200.conelp(c, G, h, dims, maxiters=2)            # warm-up: first launches of its kernels
        t0 = time.perf_counter()
        sol = cvxopt_b200.conelp(c, G, h, dims)
        dt = time.perf_counter() - t0
        res["device_conelp"] = {"seconds": dt, "iterations": int(sol["iterations"]), "status": sol["status"],
                                "iters_per_s": (sol["iterations"] + 1) / dt,
                                "primal_objective": float(sol["primal objective"])}
        g = gold.get(name.split("_")[0])
        if g:
            res["reference_cpu_golden"] = {"seconds": g["seconds"], "iterations": g["iterations"],
                                           "primal_objective": g["primal objective"],
                                           "note": "reference kktsolver='chol' on the 8-core build container"}
        out[name] = res
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self._stop, self._th = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=6)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4)
                          if len(s) >= 7 and s[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons}


def run_reference(args, rank, world):
    """CPU arm: the reference's own kkt_chol (oracle/_ref) on host cores, same step."""
    if rank != 0:
        return
    n, m = args.n, args.m
    f_fac, f_sol, f_it = flops(n, m)
    base = {"metric": METRIC, "unit": "GF/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload(n, m)}}
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "cvxopt")):
        base["unavailable"] = "oracle/_ref not built (oracle/build_ref.sh needs /root/reference)"
        print(json.dumps(base))
        return
    cores = os.cpu_count() or 1
    os.environ.setdefault("OPENBLAS_NUM_THREADS", str(min(cores, 64)))
    sys.path.insert(0, ref_dir)
    from cvxopt import matrix, misc
    P, G, d, rng = make_problem(n, m, args.seed)
    Gm, Pm = matrix(G), matrix(P)
    dims = {"l": m, "q": [], "s": []}
    factor = misc.kkt_chol(Gm, dims, matrix(0.0, (0, n)))
    W = {"d": matrix(d), "di": matrix(1.0 / d), "v": [], "beta": [], "r": [], "rti": []}
    y = matrix(0.0, (0, 1))

    def step():
        f = factor(W, Pm)
        for _ in range(2):
            x, z = matrix(rng.standard_normal(n)), matrix(rng.standard_normal(m))
            f(x, y, z)
    # a full-size reference step takes 8-30 s on this pool's hosts (single-threaded glue in
    # misc.kkt_chol.factor around the OpenBLAS calls): the number of timed steps is derived from the timed
    # warm-up so that the whole arm ends within a few minutes, never fewer than 3
    warm_run = 0
    t0 = time.perf_counter()
    step()
    warm_run += 1
    t_step = time.perf_counter() - t0
    while warm_run < args.warmup and (warm_run + 1) * t_step < 20.0:
        t0 = time.perf_counter()
        step()
        t_step = min(t_step, time.perf_counter() - t0)
        warm_run += 1
    steps_run = max(3, min(args.steps, int(150.0 / max(t_step, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps_run):
        step()
    dt = time.perf_counter() - t0
    ms = dt / steps_run * 1e3
    val = f_it / (ms * 1e-3) * 1e-9
    base.update({"value": val, "ms_per_step": ms, "steps": steps_run, "warmup": warm_run,
                 "steps_requested": args.steps, "warmup_requested": args.warmup,
                 "cpu_baseline": {"value": val, "unit": "GF/s", "cores": min(cores, 64), "kind": "reference",
                                  "sample": "%d full-size steps after %d warm-up (misc.kkt_chol, scipy-openblas)"
                                            % (steps_run, warm_run)},
                 "steps_run": steps_run,
                 "e2e": {"value": val, "unit": "GF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    print(json.dumps(base))


def cpu_baseline_sample(args, P, G, d):
    """Bounded sample of the reference path on this box's host cores (rank 0, N=1)."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "cvxopt")):
        return {"value": None, "unit": "GF/s", "cores": 0, "kind": "reference",
                "sample": "oracle/_ref not built"}
    code = r"""
import os, sys, json, time
import numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import bench
from cvxopt import matrix, misc
n, m, seed = %d, %d, %d
P, G, d, rng = bench.make_problem(n, m, seed)
factor = misc.kkt_chol(matrix(G), {'l': m, 'q': [], 's': []}, matrix(0.0, (0, n)))
W = {'d': matrix(d), 'di': matrix(1.0 / d), 'v': [], 'beta': [], 'r': [], 'rti': []}
Pm, y = matrix(P), matrix(0.0, (0, 1))
def step():
    f = factor(W, Pm)
    for _ in range(2):
        f(matrix(rng.standard_normal(n)), y, matrix(rng.standard_normal(m)))
# warm-up (OpenBLAS thread start-up, first-touch) on a small instance of the same code path: a
# full-size reference step takes 30-70 s on this pool's hosts
Pw, Gw, dw, rw = bench.make_problem(512, 1024, seed)
fw = misc.kkt_chol(matrix(Gw), {'l': 1024, 'q': [], 's': []}, matrix(0.0, (0, 512)))
fw({'d': matrix(dw), 'di': matrix(1.0 / dw), 'v': [], 'beta': [], 'r': [], 'rti': []}, matrix(Pw))(
    matrix(rw.standard_normal(512)), y, matrix(rw.standard_normal(1024)))
t0 = time.perf_counter(); k = 0
while k < 1 or (time.perf_counter() - t0 < 10.0 and k < 20):
    step(); k += 1
print(json.dumps({'ms': (time.perf_counter() - t0) / k * 1e3, 'steps': k}))
""" % (ref_dir, ROOT, args.n, args.m, args.seed)
    cores = os.cpu_count() or 1
    env = dict(os.environ, OPENBLAS_NUM_THREADS=str(min(cores, 64)))
    try:
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env,
                             timeout=600)
        res = json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as e:   # noqa: BLE001
        return {"value": None, "unit": "GF/s", "cores": min(cores, 64), "kind": "reference",
                "sample": "failed: %s" % e}
    _, _, f_it = flops(args.n, args.m)
    return {"value": f_it / (res["ms"] * 1e-3) * 1e-9, "unit": "GF/s", "cores": min(cores, 64),
            "kind": "reference", "ms_per_step": res["ms"],
            "sample": "%d full-size step(s) (n=%d, m=%d) after a small warm-up, reference misc.kkt_chol "
                      "on scipy-openblas, %d threads" % (res["steps"], args.n, args.m, min(cores, 64))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nvars", "--n", dest="n", type=int, default=8192)
    ap.add_argument("--mrows", "--m", dest="m", type=int, default=0)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ipm", action="store_true", help="skip the full-IPM and batch extras")
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--no-driver", action="store_true", help="skip the e2e_driver extra (solvers.coneqp n=4096)")
    ap.add_argument("--no-i8", action="store_true", help="skip the extra leg on the experimental int8-slice SYRK")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the solutions of the last timed step (x and z of both solves, float64) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.m <= 0:
        args.m = 2 * args.n
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import cvxopt_b200
    from cvxopt_b200 import _lib
    if not torch.cuda.is_available() or cvxopt_b200.device_count() == 0:
        raise RuntimeError("bench.py needs a B200: no CUDA device visible (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n, m = args.n, args.m
    # csrc/kkt_api.cu: the 'l'-row SYRK of large problems runs on the int8 tensor path unless CVXB_OZAKI=0
    oz_env = os.environ.get("CVXB_OZAKI", "1")[:1]
    i8_default = (oz_env == "2") or (oz_env == "1" and n >= 4096 and m >= 8192)
    f_fac, f_sol, f_it = flops(n, m)
    P, G, d, rng = make_problem(n, m, args.seed + rank)
    dims = {"l": m, "q": [], "s": []}
    kkt = cvxopt_b200.kkt_chol(G, dims, None, H=P, device=local_rank)

    # ---------------- device-resident arm (value) ----------------
    dev = torch.device("cuda", local_rank)
    d_d = torch.from_numpy(d).to(dev)
    d_di = torch.from_numpy(1.0 / d).to(dev)
    xs = [torch.from_numpy(rng.standard_normal(n)).to(dev) for _ in range(2)]
    zs = [torch.from_numpy(rng.standard_normal(m)).to(dev) for _ in range(2)]
    xw, zw = torch.empty_like(xs[0]), torch.empty_like(zs[0])

    def step_dev(keep=None):
        kkt.factor_ptr(d=d_d.data_ptr(), di=d_di.data_ptr(), space=_lib.DEVICE)
        for i in range(2):
            xw.copy_(xs[i]); zw.copy_(zs[i])
            torch.cuda.current_stream().synchronize()
            kkt.solve_ptr(xw.data_ptr(), zw.data_ptr(), space=_lib.DEVICE)
            if keep is not None:
                # the library solves on its own stream and returns once the solution is in xw / zw
                keep["x_rhs%d" % i] = xw.clone()
                keep["z_rhs%d" % i] = zw.clone()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_dev()
    syrk_ms, potrf_ms, fac_ms, sol_ms, mma_ms = [], [], [], [], []
    outputs = {}
    barrier()
    launches0 = cvxopt_b200.launch_count()
    with ClockSampler(local_rank) as clk:
        kkt.timer_start()
        for k in range(args.steps):
            step_dev(outputs if k == args.steps - 1 and args.dump_outputs else None)
            b = kkt.last_breakdown()
            syrk_ms.append(b["syrk_ms"]); potrf_ms.append(b["potrf_ms"])
            if "syrk_mma_ms" in b:
                mma_ms.append(b["syrk_mma_ms"])
            f, s = kkt.last_ms()
            fac_ms.append(f); sol_ms.append(s)
        total_ms = kkt.timer_stop()
    launches = cvxopt_b200.launch_count() - launches0
    barrier()
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = world * f_it / (ms_step * 1e-3) * 1e-9
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives: the directions x, z of the step's two solves (n + m values each)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, v in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), v.cpu().numpy().astype(np.float64))

    # ---------------- end-to-end arm (host buffers through the plugin API) ----------------
    def pinned(a):
        tt = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return tt, tt.numpy()
    keep = []
    h_d = pinned(d); h_di = pinned(1.0 / d)
    keep += [h_d, h_di]
    W = {"d": h_d[1], "di": h_di[1], "v": [], "beta": [], "r": [], "rti": []}
    hx = [pinned(rng.standard_normal(n)) for _ in range(2)]
    hz = [pinned(rng.standard_normal(m)) for _ in range(2)]
    hxw, hzw = pinned(np.zeros(n)), pinned(np.zeros(m))

    def step_e2e():
        solve = kkt(W)                       # f = kktsolver(W)
        for i in range(2):
            hxw[1][:] = hx[i][1]; hzw[1][:] = hz[i][1]
            solve(hxw[1], None, hzw[1])      # f(x, y, z), in place on host buffers
    for _ in range(args.warmup):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_val = world * f_it / (e2e_ms * 1e-3) * 1e-9
    h2d = 2 * m * 8 + 2 * (n + m) * 8
    d2h = 2 * (n + m) * 8

    if rank == 0:
        syrk = float(np.mean(syrk_ms))
        f_syrk = float(n) * n * m
        achieved = f_syrk / (syrk * 1e-3) * 1e-12
        if i8_default:
            # the 'l'-row SYRK ran as 45 exact int8 products (nine radix-2^7 slices per entry) on
            # tcgen05.mma kind::i8: the bounding pipe is the int8 tensor pipe.  `achieved` divides the int8 operations
            # by the CUDA-event time of the MMA launches alone (oz_mma_kernel main + split-K tail launch + tail
            # reduce; cvxb_kkt_syrk_mma_ms), measured live in this run; syrk_ms also covers the two slicing kernels
            # (~1 ms) and gives `frac_incl_slicing_kernels`.
            tiles = ((n + 127) // 128) * ((n + 127) // 128 + 1) // 2
            i8_ops = 45.0 * 2.0 * tiles * 128.0 * 128.0 * m
            a8_all = i8_ops / (syrk * 1e-3) * 1e-12
            mma = float(np.mean(mma_ms)) if mma_ms else syrk
            a8 = i8_ops / (mma * 1e-3) * 1e-12
            mc = measured_constants()
            pk = mc.get("int8_tensor_peak_tops")
            peak8 = float(pk) if pk else INT8_TENSOR_NOMINAL_TOPS
            tr = mc.get("oz_mma_dram_bytes_n8192_m16384") if (n == 8192 and m == 16384) else None
            roofline = {"kernel": "oz_mma_kernel (int8-slice SYRK: tcgen05.mma.kind::i8, int32 accumulators in TMEM)",
                        "bound": "tensor", "achieved": a8, "peak": peak8, "unit": "TFLOP/s",
                        "frac": a8 / peak8,
                        "kernel_ms": mma, "frac_incl_slicing_kernels": a8_all / peak8,
                        "peak_source": (mc.get("int8_tensor_peak_source") if pk else
                                        "nominal dense int8 rate of B200 (4.5 POP/s): no measured value committed")
                                       + "; `achieved` counts int8 multiply-add ops of the 45 slice products over the "
                                         "CUDA-event time of the MMA launches (kernel_ms)",
                        "nominal_int8_tops": INT8_TENSOR_NOMINAL_TOPS,
                        "fp64_equivalent_tflops": achieved, "fp64_dmma_peak_tflops": FP64_DMMA_PEAK_TFLOPS,
                        "fp64_equivalent_note": "above the fp64 DMMA peak only because it is a different pipe (int8 tensor)",
                        # dram__bytes_read.sum + dram__bytes_write.sum of one oz_mma_kernel launch: from the committed
                        # ncu capture named in profiles/measured_constants.json (not re-measured in this run)
                        "traffic": float(tr) if tr else None,
                        "traffic_source": mc.get("oz_mma_dram_source") if tr else None,
                        "algorithmic_bytes": 8.0 * m * n + 9.0 * m * n * 2 + 8.0 * n * n}
        else:
            roofline = {"kernel": "dmma_gemm_kernel<XK,YK,VEC> (fused NT-scaled SYRK)", "bound": "tensor",
                        "achieved": achieved, "peak": FP64_DMMA_PEAK_TFLOPS, "unit": "TFLOP/s",
                        "frac": achieved / FP64_DMMA_PEAK_TFLOPS,
                        "peak_source": "measured DMMA.8x8x4 pipe rate on this pool (tools/fp64_peak.cu; "
                                       "MEASURED_PEAKS.json has no fp64 entry; cuBLAS DGEMM 8192^3 = 35.4)",
                        # dram__bytes_read.sum + dram__bytes_write.sum of this kernel, one launch, from the
                        # committed capture profiles/r01j_syrk_band_order_dram.md (n=8192 only)
                        "traffic": measured_constants().get("dmma_syrk_dram_bytes_n8192_m16384")
                        if (n == 8192 and m == 16384) else None,
                        "algorithmic_bytes": 8.0 * m * n + 8.0 * n * n}
        out = {
            "metric": METRIC, "value": value, "unit": "GF/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload(n, m),
                       "parallelism": "replicas x%d" % world if world > 1 else "single GPU",
                       "l2": "inputs larger than L2 (G = %.2f GB, K = %.2f GB)" % (8.0 * n * m / 1e9, 8.0 * n * n / 1e9),
                       "flops_per_step": f_it,
                       "syrk_path": ("9 int8 slices per entry on tcgen05.mma kind::i8 (exact int32 products, fp64 recombination)"
                                     if i8_default else "fp64 DMMA"),
                       "precision": ("fp64 results: the slice products are exact integers and 9 slices keep 62 bits below each "
                                     "column maximum; error vs an 80-bit evaluation 4e-16 * sum|terms|, the fp64 dot-product level "
                                     "(tests/test_i8_syrk_gpu.py, profiles/r01k); the all-fp64 path is timed as other_syrk_path")
                                    if i8_default else "fp64 throughout"},
            "e2e": {"value": e2e_val, "unit": "GF/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "clocks": clk.summary(),
            "breakdown_ms": {"factor": float(np.mean(fac_ms)), "syrk": syrk, "potrf": float(np.mean(potrf_ms)),
                             "solve_each": float(np.mean(sol_ms))},
            "ipm_iters_per_s_kkt_bound": 1e3 / ms_step,
            "roofline": roofline,
        }
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_sample(args, P, G, d)
    extras = {}
    if rank == 0 and world == 1 and not args.no_i8:
        # extra leg (not the headline): the same KKT step with the 'l'-row SYRK on the other tensor path
        # (fp64 DMMA kernel when the int8-slice kernel is the default, and vice versa), timed the same way,
        # and its direction against the default path's
        saved = os.environ.get("CVXB_OZAKI")
        os.environ["CVXB_OZAKI"] = "0" if i8_default else "2"
        kkt8 = cvxopt_b200.kkt_chol(G, dims, None, H=P, device=local_rank)
        if saved is None:
            os.environ.pop("CVXB_OZAKI")
        else:
            os.environ["CVXB_OZAKI"] = saved

        def step8():
            kkt8.factor_ptr(d=d_d.data_ptr(), di=d_di.data_ptr(), space=_lib.DEVICE)
            for i in range(2):
                xw.copy_(xs[i]); zw.copy_(zs[i])
                torch.cuda.current_stream().synchronize()
                kkt8.solve_ptr(xw.data_ptr(), zw.data_ptr(), space=_lib.DEVICE)
        for _ in range(3):
            step8()
        x8 = xw.clone()
        step_dev()
        xdiff = float((torch.linalg.vector_norm(x8 - xw) / torch.linalg.vector_norm(xw)).item())
        torch.cuda.synchronize()
        k8 = max(3, min(args.steps, 10))
        s8 = []
        kkt8.timer_start()
        for _ in range(k8):
            step8()
            s8.append(kkt8.last_breakdown()["syrk_ms"])
        ms8 = kkt8.timer_stop() / k8
        extras["other_syrk_path"] = {
            "what": ("fp64 DMMA SYRK (CVXB_OZAKI=0)" if i8_default else "int8-slice SYRK on tcgen05.mma kind::i8 (CVXB_OZAKI=2)")
                    + ": same step, same inputs",
            "ms_per_step": ms8, "value": f_it / (ms8 * 1e-3) * 1e-9, "syrk_ms": float(np.mean(s8)),
            "syrk_fp64_equiv_tflops": float(n) * n * m / (float(np.mean(s8)) * 1e-3) * 1e-12,
            "direction_rel_diff_vs_default": xdiff}
        kkt8.close()
        del kkt8
    kkt.close()
    del kkt, d_d, d_di, xs, zs
    torch.cuda.empty_cache()
    if not args.no_ipm:
        # config 4 (BASELINE): 512 independent dense QPs, ALL held by rank 0, through the path north_star names:
        # NCCL scatter of the problem data -> device-resident lock-step IPM on every rank -> NCCL gather of the
        # iterates (cvxopt_b200.qp_batch_distributed).  Strong scaling: total work fixed as N grows.
        try:
            extras_b = run_batch_distributed(args.batch, 512, 1024, rank, world, dev)
            if rank == 0:
                extras["batch"] = extras_b
        except Exception as exc:            # noqa: BLE001  keep the headline line even if this extra leg fails
            if rank == 0:
                extras["batch"] = {"error": repr(exc)[:300]}
        # (ii) IPM iterations/s: a whole solve of the same-size QP, device resident (rank 0 only).  The device
        # IPM's factor takes the same SYRK path as `value` (int8 slices at this size; reported as syrk_path).
        if rank == 0:
            try:
                extras["ipm"] = run_ipm(n, m, args.seed, local_rank)
            except Exception as exc:        # noqa: BLE001
                extras["ipm"] = {"error": repr(exc)[:300]}
            if world == 1 and not args.no_driver:
                try:
                    extras["e2e_driver"] = run_e2e_driver(4096, 8192, args.seed, local_rank)
                except Exception as exc:    # noqa: BLE001
                    extras["e2e_driver"] = {"error": repr(exc)[:300]}
                try:
                    extras["e2e_cones"] = run_e2e_cones(local_rank)
                except Exception as exc:    # noqa: BLE001
                    extras["e2e_cones"] = {"error": repr(exc)[:300]}
    if rank == 0:
        out.update(extras)
        print(json.dumps(out))
    if world > 1:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


if __name__ == "__main__":
    main()
