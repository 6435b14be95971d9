#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 hot path (BASELINE.json metric):

    iLQR iterations/sec on batched Quadrotor (n=13, m=4, N=101, batch=4096 per GPU, goal + control-bound AL-iLQR)

A "step" is one iLQR iteration (dynamics expansion + Riccati backward pass + forward pass with line search) of
every instance in the batch.  `value` times K consecutive iterations of one solve with everything resident in HBM;
`e2e` times the same iteration through the public C ABI with HOST buffers (x0 + warm-start controls uploaded,
controls + merit downloaded every step).  `--impl reference` times the CPU oracle port of the same path on the
host cores (the Julia reference cannot run here: no Julia in the image).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs DIR     # also writes the last timed step's outputs to DIR/*.npy
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "quadrotor": dict(n=13, m=4, N=101, batch=4096, desc="Quadrotor point-to-point n=13 m=4 N=101, u in [0,10] + goal (AL-iLQR), Riccati on the Lie-group error state n_e=12 (what Altro does for this model)"),
    "quadrotor_fullstate": dict(n=13, m=4, N=101, batch=4096, desc="Quadrotor point-to-point n=13 m=4 N=101, u in [0,10] + goal (AL-iLQR), Riccati on the full 13-state (round-1 headline)"),
    "quadrotor_calm": dict(n=13, m=4, N=101, batch=4096, desc="the quadrotor workload with a 25x smaller perturbation of the hover controls (the open-loop rollout does not tumble): no regularisation restarts in the backward pass -- isolates the single-sweep speed of the Riccati kernel"),
    "cartpole": dict(n=4, m=1, N=101, batch=1024, desc="Cartpole swing-up n=4 m=1 N=101, unconstrained LQR cost"),
    "acrobot": dict(n=4, m=1, N=201, batch=8192, desc="Acrobot n=4 m=1 N=201, dense second-order cost + |u|<=15 + goal (AL)"),
    "quadrotor_lie": dict(n=13, m=4, N=101, batch=4096, desc="Quadrotor n=13 m=4 N=101 on the Lie-group error state (n_e=12), LQR cost, u in [0,10] + goal; materialised expansion (lie.cu)"),
}


def build_problem(workload, B, N, cls=None, device=0):
    import trajopt_b200 as TO
    P = TO.problems
    if workload == "quadrotor":
        return P.quadrotor(B=B, N=N, cls=cls, device=device, error_state=True)
    if workload == "quadrotor_calm":
        return P.quadrotor(B=B, N=N, cls=cls, device=device, error_state=True, u_noise=0.002)
    if workload == "quadrotor_fullstate":
        return P.quadrotor(B=B, N=N, cls=cls, device=device)
    if workload == "cartpole":
        return P.cartpole(B=B, N=N, cls=cls, device=device)
    if workload == "acrobot":
        return P.acrobot(B=B, N=N, cls=cls, device=device)
    if workload == "quadrotor_lie":
        return P.quadrotor_lie(B=B, N=N, cls=cls, device=device, quat_cost=False, quat_goal=False)
    raise SystemExit(f"unknown workload {workload}")


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons of one GPU while the timed region runs"""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = []
        for i, name in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap")):
            if any(len(r) > i and r[i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        # only the upper half of the samples are "under load" for short runs
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": (load[len(load) // 2] if load else None), "sm_max_mhz": (max(mx) if mx else None), "reasons": reasons, "samples": len(sm)}


def host_cpu_quota():
    """CPUs this process may actually use: min(affinity, cgroup quota) -- the GPU boxes expose 128 logical CPUs under a
    16-CPU cgroup quota, and oversubscribing the quota throttles the whole process."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(round(int(q) / int(per)))))
    except Exception:
        pass
    return n


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(prob, directory, suffix="", budget=DUMP_BYTES):
    """--dump-outputs: what the timed path left behind after its last step, i.e. what a caller of to_ilqr_step reads back -- states
    [B, N, n], controls [B, N-1, m], merit [B] and the accepted step size of the last line search [B] -- as <directory>/<name><suffix>.npy
    in float64, together with instance_index (the batch rows written).  The inputs are seeded, so two builds run with the same arguments
    can be compared array for array.  When the batch does not fit in `budget` bytes, a fixed seeded sample of the instances is written,
    the same rows of every array."""
    import trajopt_b200 as TO
    out = {"states": TO.states(prob), "controls": TO.controls(prob), "merit": TO.merit(prob), "step_size": TO.solver_state(prob)["alpha"]}
    B = prob.B
    per_instance = sum(a.nbytes for a in out.values()) // B + 8          # + 8: the instance_index entry
    keep = min(B, (budget - 1024 * (len(out) + 1)) // per_instance)      # 1 KB per file for the .npy headers
    rows = np.arange(B) if keep == B else np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    out = {k: v[rows] for k, v in out.items()}
    out["instance_index"] = rows
    os.makedirs(directory, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(directory, f"{k}{suffix}.npy"), np.ascontiguousarray(v, dtype=np.float64))


def cpu_arm(workload, B, N, warmup, steps, budget_s=None, dump=None):
    """The CPU arm: the oracle port of the same path on the host cores, on the SAME workload as the GPU arm -- the same B instances
    from the same initial state, `warmup` untimed iLQR iterations followed by `steps` timed ones of the same solve (one step = one
    iLQR iteration of every instance).  The warm-up iterations double as the thread-count probe (1x / 2x / 4x the CPU quota, best
    kept).  `budget_s` (cpu_baseline leg of the GPU arm): cap the timed steps so the leg stays near that many seconds -- the steps
    actually run are reported.  `dump`: directory the outputs of the last step go to (dump_outputs)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding as OB
    import trajopt_b200 as TO
    lib = OB.load_oracle()
    lib.orc_set_threads.restype = C.c_int
    quota = host_cpu_quota()
    ncpu = os.cpu_count() or quota
    prob = build_problem(workload, B, N, cls=OB.OracleProblem)
    TO.rollout(prob)
    cands = sorted({quota, min(2 * quota, ncpu), min(4 * quota, ncpu)})
    best = None
    warmup = max(warmup, 1)
    for i in range(warmup):
        thr = cands[i] if i < len(cands) else best[0]
        nthr = lib.orc_set_threads(int(thr))
        t0 = time.perf_counter(); TO.ilqr_step(prob, 1); t1 = time.perf_counter() - t0
        if best is None or t1 < best[1]:
            best = (nthr, t1)
    nthr = lib.orc_set_threads(best[0])
    if budget_s is not None:
        steps = max(1, min(steps, int(budget_s / max(best[1], 1e-6))))
    t0 = time.perf_counter()
    for _ in range(steps):
        TO.ilqr_step(prob, 1)
    wall = time.perf_counter() - t0
    if dump:
        dump_outputs(prob, dump)
    prob.close()
    return {"value": B * steps / wall, "unit": "instance-iterations/s", "cores": nthr, "kind": "port",
            "sample": f"{B} instances x {steps} iLQR iterations after {warmup} warm-up iterations of the same solve as the GPU arm ({wall:.2f} s wall; "
                      f"{nthr} OpenMP threads = best of 1x/2x/4x the host's {quota}-CPU quota, {ncpu} logical CPUs; g++ -O3 x86-64-v3)",
            "steps": steps, "ms_per_step": 1e3 * wall / steps, "wall_s": wall, "host_cpu_quota": quota, "nproc": ncpu}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path.  The Julia package cannot run in this image (no Julia, and
    its RK4 / AD / Riccati live in un-vendored packages), so the arm times the oracle port -- the documented CPU restatement -- on
    all host threads, on the GPU arm's own configuration: the global batch (batch per GPU x world, or the fixed global batch of
    --scaling strong), the same initial state, `warmup` + `steps` iterations of one solve.  Rank 0 only."""
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    N = args.N or w["N"]
    per_gpu, glob = batch_split(args, w, world)
    warmup = max(args.warmup, 3)
    base = cpu_arm(args.workload, glob, N, warmup, args.steps, dump=args.dump_outputs)
    out = {"impl": "reference", "metric": "ilqr_iterations_per_sec", "value": base["value"], "unit": "instance-iterations/s", "n_gpus": args.gpus,
           "steps": base["steps"], "warmup": warmup, "ms_per_step": base["ms_per_step"], "higher_is_better": True,
           "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": make_config(args, w, per_gpu, N, world),
           "details": {"note": "CPU arm: oracle port of the reference path (Julia unavailable) on the whole global batch, same initial state, warm-up and step count as the GPU arm"},
           "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
           "e2e": {"value": base["value"], "unit": "instance-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "host": {"cpu_quota": base["host_cpu_quota"], "nproc": base["nproc"], "threads": base["cores"]}}
    print(json.dumps(out), flush=True)


def make_config(args, w, per_gpu, N, world):
    """the `config` object of the JSON line -- identical for the GPU arm and the CPU (--impl reference) arm"""
    n_r, nm_r = (w["n"] - 1, w["n"] + w["m"] - 1) if args.workload in ("quadrotor", "quadrotor_lie", "quadrotor_calm") else (w["n"], w["n"] + w["m"])
    return {"workload": w["desc"], "batch_per_gpu": per_gpu, "N": N, "global_batch": per_gpu * world, "parallelism": f"batch-sharded x{world}",
            "step": "1 iLQR iteration = dynamics expansion + Riccati backward pass + forward pass/line search of every instance, K consecutive iterations of one solve",
            "merit_collective_every": (args.merit_every if world > 1 else None),
            "l2": "inputs larger than L2 (126 MB): the per-knot dynamics Jacobians alone are %.0f MB per GPU, rewritten and re-read every step"
                  % (per_gpu * (N - 1) * n_r * nm_r * 8 / 1e6)}


def batch_split(args, w, world):
    """(instances per GPU, global batch): weak scaling keeps the per-GPU batch, strong scaling the global one"""
    if args.scaling == "strong":
        glob = args.batch or w["batch"]
        return max(1, glob // world), max(1, glob // world) * world
    per = args.batch or w["batch"]
    return per, per * world


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="quadrotor", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU (default: the workload's BASELINE batch)")
    ap.add_argument("--N", type=int, default=0, help="knot points (default: the workload's)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: --batch instances per GPU; strong: --batch instances in total, split over the GPUs")
    ap.add_argument("--merit-every", type=int, default=5, help="N > 1: iterations between two {sum merit, max violation} collectives (a solver's convergence report)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-depth", type=int, default=2, help="problem handles in flight in the end-to-end measurement (1 = strictly serial, 2 = double-buffered)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the states, controls, merit and step sizes of the last step to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    import trajopt_b200 as TO
    K = TO.capi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    w = WORKLOADS[args.workload]
    B, global_batch = batch_split(args, w, world)
    N = args.N or w["N"]
    n, m = w["n"], w["m"]
    prob = build_problem(args.workload, B, N, device=local)
    lib, h = prob._lib, prob._h
    stream = torch.cuda.current_stream()
    K.check(lib, h, lib.to_set_stream(h, C.c_void_p(stream.cuda_stream)))
    x0_host = torch.from_numpy(prob.x0.copy()).pin_memory()
    U0_np = TO.controls(prob)
    U0_host = torch.from_numpy(U0_np.copy()).pin_memory()
    U_out = torch.empty_like(U0_host).pin_memory()
    J_out = torch.empty(B, dtype=torch.float64).pin_memory()
    merit2 = TO.multi_gpu.merit_device_tensor(prob, f"cuda:{local}")

    def dptr(t):
        return C.cast(t.data_ptr(), K.c_double_p)

    def reset():
        K.check(lib, h, lib.to_set_initial_state(h, dptr(x0_host)))
        K.check(lib, h, lib.to_set_controls(h, dptr(U0_host)))
        K.check(lib, h, lib.to_rollout(h))

    side = torch.cuda.Stream() if world > 1 else None
    gather = torch.empty((world, 2), dtype=torch.float64, device=f"cuda:{local}") if world > 1 else None
    step_no = [0]

    def step():
        K.check(lib, h, lib.to_ilqr_step(h, 1))
        step_no[0] += 1
        if world > 1 and step_no[0] % max(1, args.merit_every) == 0:
            # the path's only collective: {sum merit, max violation} over the ranks (SURVEY 8e) -- ONE all-gather of the 2-vectors every
            # `merit_every` iterations.  Nothing on the device consumes it, so it runs on a side stream behind the per-GPU reduction
            # kernel (to_reduce_merit_async queues that behind the iteration's last kernel and makes `side` wait on its event); the
            # main stream never waits for the collective: the previous one has long finished when the buffer is reduced again.
            K.check(lib, h, lib.to_reduce_merit_async(h, C.c_void_p(side.cuda_stream)))
            with torch.cuda.stream(side):
                TO.multi_gpu.all_reduce_merit(merit2, scratch=gather)

    def barrier():
        if world > 1:
            stream.wait_stream(side)
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ---------------------------------------------------------------------------------
    reset()
    for _ in range(args.warmup):
        step()
    if world > 1:   # the first collective sets up NCCL's channels (tens of ms): it belongs to the warm-up whatever --merit-every is
        K.check(lib, h, lib.to_reduce_merit_async(h, C.c_void_p(side.cuda_stream)))
        with torch.cuda.stream(side):
            TO.multi_gpu.all_reduce_merit(merit2, scratch=gather)
        step_no[0] = 0
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start(); time.sleep(0.3)
    barrier()
    launches0 = lib.to_launch_count(h)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    if side is not None:
        if args.steps % max(1, args.merit_every) != 0:   # the final merit report is part of the job
            K.check(lib, h, lib.to_reduce_merit_async(h, C.c_void_p(side.cuda_stream)))
            with torch.cuda.stream(side):
                TO.multi_gpu.all_reduce_merit(merit2, scratch=gather)
        stream.wait_stream(side)      # the last collective is inside the timed region
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = lib.to_launch_count(h) - launches0
    clocks = sampler.finish() if sampler else None
    tmax = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax.item())
    value = B * world * args.steps / (ms * 1e-3)
    st = TO.solver_state(prob)
    accepted_frac = float((st["alpha"] > 0).mean())
    if args.dump_outputs:   # before the passes below restart the solve on `prob`
        dump_outputs(prob, args.dump_outputs, f"_rank{rank}" if world > 1 else "", DUMP_BYTES // world)

    # ---- per-phase timing pass (CUDA events around each kernel on the launching stream) -> roofline -----------------
    reset()
    for _ in range(args.warmup):
        step()
    lib.to_set_phase_timing(h, 1)
    pms = (C.c_double * K.PHASE_COUNT)(); pl = (C.c_int64 * K.PHASE_COUNT)()
    lib.to_get_phase_times(h, pms, pl, 1)
    for _ in range(args.steps):
        K.check(lib, h, lib.to_ilqr_step(h, 1))
    lib.to_get_phase_times(h, pms, pl, 1)
    lib.to_set_phase_timing(h, 0)
    phase = {name: (pms[i] / max(1, pl[i])) for name, i in (("expand", K.PHASE_EXPAND), ("cost_expansion", K.PHASE_COSTEXP), ("backward", K.PHASE_BACKWARD), ("forward", K.PHASE_FORWARD), ("ladder", K.PHASE_LADDER), ("late_expansion", K.PHASE_LATE))}
    E, R, F = C.c_int64(), C.c_int64(), C.c_int64()
    lib.to_algorithmic_bytes(h, C.byref(E), C.byref(R), C.byref(F))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    r_ms = phase["backward"]
    achieved = (R.value * B / (r_ms * 1e-3)) / 1e9 if r_ms > 0 else 0.0
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "riccati_traffic.json"))).get(f"{args.workload}_B{B}_N{N}")
    except Exception:
        pass
    frag = args.workload in ("quadrotor", "quadrotor_lie", "quadrotor_calm") and not os.environ.get("TO_NO_FRAG")
    rk = "k_riccati_frag (riccati_frag.cu: register-resident tensor-core Riccati pass on the error state, timed alone)" if frag \
        else "k_expansion_compact + k_riccati_dense_mma (lie.cu: error-state expansion + shared-memory tensor-core Riccati pass)" if args.workload in ("quadrotor", "quadrotor_lie", "quadrotor_calm") \
        else "k_riccati (Riccati backward pass)"
    roofline = {"kernel": rk, "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": R.value * B, "avg_launch_ms": r_ms,
                "phase_ms": phase, "fp64_tflops_riccati": None}
    # FP64 view of the same kernel: 2 * (T + Qzz + Qz + S-update + solves) FMA per knot (DESIGN.md), counted analytically
    nm = n + m
    if args.workload in ("quadrotor", "quadrotor_lie", "quadrotor_calm"):
        n, nm = n - 1, nm - 1        # the recursion runs on the error state
    fma_knot = n * n * nm + n * nm * (nm + 1) // 2 + n * nm + m * n * (n + 1) // 2 + m * m * (n + 1) + m * m * m // 3
    roofline["fp64_tflops_riccati"] = (2.0 * fma_knot * (N - 1) * B / (r_ms * 1e-3)) / 1e12 if r_ms > 0 else None

    # ---- end to end through the C ABI with host buffers -------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        # Two problem handles (each its own stream) work on alternate steps: while one batch iterates, the other batch's inputs are uploaded
        # and the previous results downloaded -- the double buffering any caller streaming independent batches through the C ABI would use
        # (setters are asynchronous, getters synchronise their own handle only).  Every step still uploads ITS inputs and downloads ITS
        # results inside the timed region; --e2e-depth 1 gives the strictly serial upload -> iterate -> download of one handle.
        depth = max(1, min(2, args.e2e_depth))
        probs = [prob] + [build_problem(args.workload, B, N, device=local) for _ in range(depth - 1)]
        outs = [(U_out, J_out)] + [(torch.empty_like(U0_host).pin_memory(), torch.empty(B, dtype=torch.float64).pin_memory()) for _ in range(depth - 1)]

        def issue(i):
            hh = probs[i % depth]._h
            K.check(lib, hh, lib.to_set_initial_state(hh, dptr(x0_host)))     # H2D (pinned, asynchronous)
            K.check(lib, hh, lib.to_set_controls(hh, dptr(U0_host)))          # H2D (pinned, asynchronous)
            K.check(lib, hh, lib.to_rollout(hh))
            K.check(lib, hh, lib.to_ilqr_step(hh, 1))

        def collect(i):
            hh = probs[i % depth]._h
            K.check(lib, hh, lib.to_get_controls(hh, dptr(outs[i % depth][0])))   # D2H (synchronises this handle)
            K.check(lib, hh, lib.to_merit(hh, dptr(outs[i % depth][1])))          # D2H

        def e2e_run(k):
            for i in range(k):
                issue(i)
                if i >= depth - 1:
                    collect(i - (depth - 1))
            for i in range(max(0, k - (depth - 1)), k):
                collect(i)

        e2e_run(args.warmup)
        barrier()
        t0 = time.perf_counter()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        e2e_run(args.steps)
        g1.record(stream)
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        ems = max(g0.elapsed_time(g1), wall_ms)    # the host-blocking copies are part of the step
        t2 = torch.tensor([ems], dtype=torch.float64, device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        ems = float(t2.item())
        e2e = {"value": B * world * args.steps / (ems * 1e-3), "unit": "instance-iterations/s",
               "h2d_bytes_per_step": int(x0_host.numel() * 8 + U0_host.numel() * 8), "d2h_bytes_per_step": int(U_out.numel() * 8 + J_out.numel() * 8),
               "ms_per_step": ems / args.steps,
               "handles_in_flight": depth,
               "what": "per step: upload x0 + warm-start U (pinned host), rollout, 1 iLQR iteration, download U + merit J"
                       + ("; consecutive steps alternate between two problem handles so that one batch's copies overlap the other batch's iteration" if depth > 1 else "")}
        for pb in probs[1:]:
            pb.close()

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        try:
            cpu = cpu_arm(args.workload, B, N, max(args.warmup, 3), args.steps, budget_s=12.0)
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as ex:   # the oracle is only the reported baseline; never let it take the GPU number down
            cpu = {"value": None, "unit": "instance-iterations/s", "cores": 0, "kind": "port", "sample": f"failed: {ex}"}

    if rank == 0:
        out = {"metric": "ilqr_iterations_per_sec", "value": value, "unit": "instance-iterations/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
               "dtype": "f64", "data": "synthetic",
               "config": make_config(args, w, B, N, world),
               "details": {"batch_iterations_per_s": args.steps / (ms * 1e-3), "accepted_fraction_last_step": accepted_frac},
               "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu}
        print(json.dumps(out), flush=True)
    prob.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
