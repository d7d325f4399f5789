#!/usr/bin/env python
"""bench.py -- ms per LM iteration (linearize + QR + PCG + back-substitution) of the square-root BA inner loop.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU)
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host cores
  python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed (DIR/*.npy)

A "step" is ONE Levenberg-Marquardt iteration of the reference's loop (solver/bal_bundle_adjustment.cpp:291-521):
[compute_error + linearize at a new linearization point] + solve(lambda) + apply + compute_error + accept/reject.
Both arms run the same LM trajectory from the same seeded, perturbed synthetic problem.  The W warm-up iterations start at
the initial point; the state is then RESET to the initial point and K iterations are timed from there, so the number does
not depend on W.  When the reference's own stopping rule fires (function tolerance, max lambda or max_num_iterations,
bal_bundle_adjustment.cpp:174-201, 378-379, 291) the solve is over and the next step starts a new solve from the initial
point: every timed step is an iteration the reference's loop would execute, never an iteration past convergence.

Workload: N = 1 -> BASELINE.json configs[1] (BAL ladybug problem-1723-156502, float32); N > 1 -> configs[3] (BAL venice
problem-1778-993923, float32, landmarks sharded over the N GPUs); --workload final-13682 = configs[4].  Synthetic
stand-ins of the same shape (no BAL file exists on the box; SURVEY.md section 8d).  A line measured at N > 1 also
carries the N = 1 time of the SAME workload (rank 0 alone, same run), because the driver's own N = 1 line is configs[1].
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ms/LM-iter (linearize+QR+PCG) on BAL at 1/2/4/8 B200 vs CPU ref"


# ----------------------------------------------------------------------------------------------
# LM loop as a step machine (one call = one `it` of optimize_lm_ours)
# ----------------------------------------------------------------------------------------------
class LMStepper:
    def __init__(self, backend, dtype, initial_trust_region_radius=1e4, min_trust_region_radius=1e-32,
                 max_trust_region_radius=1e16, min_relative_decrease=0.0, initial_vee=2.0, vee_factor=2.0,
                 function_tolerance=1e-6, max_num_iterations=20):
        self.b = backend
        self.S = np.float32 if np.dtype(dtype) == np.float32 else np.float64
        S = self.S
        self.min_lambda, self.max_lambda = S(1.0 / max_trust_region_radius), S(1.0 / min_trust_region_radius)
        self.vee_factor, self.initial_vee = S(vee_factor), S(initial_vee)
        self.lam0 = S(1.0 / initial_trust_region_radius)
        self.min_relative_decrease = min_relative_decrease
        self.function_tolerance = function_tolerance
        self.max_num_iterations = max_num_iterations
        self.log = []
        self.solves = 0
        self._fresh()

    def _fresh(self):
        self.lam, self.vee = self.lam0, self.initial_vee
        self.new_outer = True
        self.ri = None
        self.it = 0  # LM iterations done in the current solve

    def restart(self):
        """a new solve from the initial point (same seeded start; bal_bundle_adjustment.cpp:249-290)"""
        self.b.reset()
        self.solves += 1
        self._fresh()

    def step(self):
        b, S = self.b, self.S
        rec = {"lambda": float(self.lam), "solve": self.solves, "it": self.it + 1}
        terminated = False
        with np.errstate(all="ignore"):
            fused = getattr(b, "fused", False)
            lin_first = self.new_outer
            if self.new_outer:
                self.ri = b.compute_error()
                if not fused:
                    b.linearize()
                self.new_outer = False
            if fused:  # rba_lm_step: [linearize] + solve + backup + apply + compute_error with one host synchronisation
                fr = b.lm_step(float(self.lam), lin_first)
                inc_ok = not fr["solve_failed"]
            else:
                inc_ok = b.solve(float(self.lam))
            rec["cg_iterations"] = b.cg_iterations()
            self.it += 1
            if not inc_ok:
                if fused:
                    b.restore()
                self.lam = S(self.vee * self.lam); self.vee = S(self.vee * self.vee_factor)
                rec["accepted"] = False
                terminated = bool(self.lam > self.max_lambda)
            else:
                if fused:
                    l_diff, ri2 = S(fr["l_diff"]), fr["cost"]
                else:
                    b.backup()
                    l_diff = S(b.apply())
                    ri2 = b.compute_error()
                ok = bool(np.isfinite(l_diff)) and ri2["is_numerically_valid"]
                success = False
                if ok:
                    f_diff = S(self.ri["all"]["error"] - ri2["all"]["error"])
                    q = S(f_diff / l_diff)
                    success = bool(l_diff > 0 and q > self.min_relative_decrease)
                rec.update(cost=ri2["all"]["error"], accepted=success)
                if success:
                    self.lam = max(self.min_lambda, S(self.lam * S(max(1.0 / 3, 1 - (2 * float(q) - 1) ** 3))))
                    self.vee = self.initial_vee
                    self.new_outer = True
                    # function tolerance (bal_bundle_adjustment.cpp:174-201)
                    terminated = bool(abs(self.ri["all"]["error"] - ri2["all"]["error"]) <= self.function_tolerance * ri2["all"]["error"])
                else:
                    self.lam = S(self.vee * self.lam); self.vee = S(self.vee * self.vee_factor)
                    b.restore()
                    terminated = bool(self.lam > self.max_lambda)
            if self.it >= self.max_num_iterations:
                terminated = True
        rec["terminated"] = terminated
        self.log.append(rec)
        if terminated:
            self.restart()
        return rec


class GpuBackend:
    """device-resident state and increment (what `value` measures); one host synchronisation per LM iteration (rba_lm_step)"""
    fused = True

    def __init__(self, lin):
        self.lin = lin
        bp = lin.bal_problem
        self._init = (bp.cams.copy(), bp.lms.copy())

    def reset(self):
        bp = self.lin.bal_problem
        bp.cams[:] = self._init[0]; bp.lms[:] = self._init[1]
        self.lin.upload_state()

    def compute_error(self): return self.lin.compute_error()
    def lm_step(self, lam, linearize_first): return self.lin.lm_step(lam, linearize_first)
    def linearize(self): self.lin.linearize()
    def solve(self, lam):
        self.lin.solve(lam, to_host=False)
        return self.lin.last_cg.termination_type != 2
    def cg_iterations(self): return self.lin.last_cg.num_iterations
    def backup(self): self.lin._backup()
    def apply(self): return self.lin.apply(None)
    def restore(self): self.lin._restore()


class GpuE2EBackend(GpuBackend):
    """every step moves its inputs host->device from pinned memory and its results device->host through the
    reference-facing API: state up, increment down, increment up (apply takes a host vector like
    LinearizorQR::apply(VecX&&)), state + l_diff + ResidualInfo down."""
    fused = False

    def __init__(self, lin):
        super().__init__(lin)
        import torch
        bp = lin.bal_problem
        # re-home the host arrays in pinned memory
        self._pin = [torch.from_numpy(bp.cams.copy()).pin_memory(), torch.from_numpy(bp.lms.copy()).pin_memory()]
        bp.cams, bp.lms = self._pin[0].numpy(), self._pin[1].numpy()
        self._bk = (bp.cams.copy(), bp.lms.copy())
        self._inc_pin = torch.zeros(9 * lin.nc, dtype=torch.float32 if lin.dtype == np.float32 else torch.float64).pin_memory()
        self.h2d = self.d2h = 0
        self.item = lin.dtype.itemsize

    def reset(self):
        bp = self.lin.bal_problem
        bp.cams[:] = self._init[0]; bp.lms[:] = self._init[1]
        self.lin.upload_state()  # compute_error / linearize of the new solve run before the next solve() uploads
        self.h2d += (10 * self.lin.nc + 3 * self.lin.nl) * self.item

    def solve(self, lam):
        lin = self.lin
        lin.upload_state()
        self.h2d += (10 * lin.nc + 3 * lin.nl) * self.item
        inc = lin.solve(lam, to_host=True)
        self._inc_pin.numpy()[:] = inc
        self.d2h += 9 * lin.nc * self.item
        return bool(np.all(np.isfinite(inc)))

    def backup(self):
        bp = self.lin.bal_problem
        self._bk[0][:] = bp.cams; self._bk[1][:] = bp.lms
        self.lin._backup()

    def apply(self):
        lin = self.lin
        l = lin.apply(self._inc_pin.numpy())
        lin.download_state()
        self.h2d += 9 * lin.nc * self.item
        self.d2h += (10 * lin.nc + 3 * lin.nl) * self.item + self.item
        return l

    def compute_error(self):
        self.d2h += 56
        return self.lin.compute_error()

    def restore(self):
        bp = self.lin.bal_problem
        bp.cams[:] = self._bk[0]; bp.lms[:] = self._bk[1]
        self.lin._restore()


class OracleBackend:
    def __init__(self, o):
        self.o = o
        self._inc = None
        self._it = 0
        c, l = o.get_state()
        self._init = (c.copy(), l.copy())

    def reset(self): self.o.set_state(*self._init)

    def compute_error(self): return self.o.compute_error()
    def linearize(self):
        if not self.o.linearize():
            raise RuntimeError("numerical failure during linearization")
    def solve(self, lam):
        self._inc, self._it = self.o.solve(lam)
        return bool(np.all(np.isfinite(self._inc)))
    def cg_iterations(self): return self._it
    def backup(self): self.o.backup()
    def apply(self): return self.o.apply(self._inc)
    def restore(self): self.o.restore()


# ----------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.split(",")]
                if len(f) >= 8:
                    self.samples.append(f)
        except Exception:
            pass

    def stop(self) -> dict:
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        mx = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def host_threads() -> int:
    """threads for the CPU arm: one per physical core (the landmark loop is memory-bound; SMT siblings only add contention)"""
    try:
        import psutil
        n = psutil.cpu_count(logical=False) or os.cpu_count()
    except Exception:
        n = os.cpu_count()
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return max(1, int(n))


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def make_problem(args):
    """the synthetic stand-in; with RBA_BENCH_CACHE_DIR set the generated arrays are kept there (npz) so that several
    bench invocations on one box (dense / implicit, the ranks of one torchrun) generate a large problem only once"""
    from rootba_b200.synthetic import BalArrays, synth_config
    cache = os.environ.get("RBA_BENCH_CACHE_DIR")
    path = os.path.join(cache, f"{args.workload}_s{args.seed}_x{args.scale}.npz") if cache else None
    if path and os.path.exists(path):
        z = np.load(path)
        return BalArrays(z["cams"], z["lms"], z["lm_off"], z["obs_cam"], z["obs_xy"])
    arrays = synth_config(args.workload, seed=args.seed, scale=args.scale)
    if path:
        os.makedirs(cache, exist_ok=True)
        tmp = f"{path}.{os.getpid()}.tmp.npz"
        np.savez(tmp, cams=arrays.cams, lms=arrays.lms, lm_off=arrays.lm_off, obs_cam=arrays.obs_cam, obs_xy=arrays.obs_xy)
        os.replace(tmp, path)
    return arrays


def tune_oracle_threads(o, n_vec, dtype, max_threads):
    """The CPU restatement scatters under per-camera locks like the reference (reduction_alg=1), which stops scaling well
    before 64 threads; so that the CPU arm is not handicapped, time the PCG operator at a few thread counts (after the
    warm-up steps, when the oracle is linearised) and keep the fastest.  Returns the thread count left configured."""
    from oracle import oracle_py as orc
    best, best_t = max_threads, None
    try:
        x = np.ones(n_vec, dtype=dtype)
        cands = sorted({max(1, max_threads >> k) for k in range(4)} | {min(8, max_threads)})
        for T in cands:
            o.set_options(orc.default_options(num_threads=T))
            o.right_multiply(x)
            t0 = time.perf_counter()
            for _ in range(3):
                o.right_multiply(x)
            dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best, best_t = T, dt
    except Exception:  # the sweep is a courtesy to the CPU arm; never let it take the measurement down
        best = max_threads
    o.set_options(orc.default_options(num_threads=best))
    return best


WORKLOAD_LABEL = {
    "ladybug-1723": "synthetic ladybug-1723 (BAL ladybug problem-1723-156502 shape, BASELINE configs[1])",
    "trafalgar-257": "synthetic trafalgar-257 (BAL trafalgar problem-257-65132 shape, BASELINE configs[2])",
    "venice-1778": "synthetic venice-1778 (BAL venice problem-1778-993923 shape, BASELINE configs[3])",
    "final-13682": "synthetic final-13682 (BAL final problem-13682-4456117 shape, BASELINE configs[4])",
}
SOLVER_LABEL = "SQUARE_ROOT/SCHUR_JACOBI/Householder, reference defaults"
PROTOCOL = ("W warm-up LM iterations from the initial point, state reset, then K timed LM iterations from the initial point; "
            "a solve that meets the reference's stopping rule is followed by a new solve from the initial point")


def default_workload(gpus: int) -> str:
    """N = 1: BASELINE configs[1]; N > 1: configs[3], the smallest config BASELINE.json shards over 8 GPUs"""
    return "ladybug-1723" if gpus <= 1 else "venice-1778"


def workload_config(args, arrays) -> dict:
    """the `config` object, identical in both arms"""
    return {"workload": WORKLOAD_LABEL.get(args.workload, f"synthetic {args.workload}"), "scale": args.scale, "seed": args.seed,
            **arrays.stats(), "solver": SOLVER_LABEL, "protocol": PROTOCOL}


def run_lm(backend, dtype, warmup, steps, timer=None, barrier=None, after_warmup=None, budget_s=None, on_step=None):
    """W warm-up steps, reset to the initial point, K timed steps (fewer if `budget_s` of wall time is exhausted; >= 1).
    Returns (seconds, wall seconds, stepper, steps timed)."""
    st = LMStepper(backend, dtype)
    for _ in range(warmup):
        st.step()
    st.restart()
    st.log.clear()
    st.solves = 0
    if after_warmup:
        after_warmup()
    if barrier:
        barrier()
    t0 = time.perf_counter()
    if timer:
        timer[0]()
    done = 0
    for _ in range(steps):
        rec = st.step()
        done += 1
        if on_step:
            on_step(rec)
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dev = timer[1]() if timer else None
    wall = time.perf_counter() - t0
    if barrier:
        barrier()
    return (dev if dev is not None else wall), wall, st, done


def trajectory_fields(st) -> dict:
    return {"cg_iterations": [r.get("cg_iterations") for r in st.log],
            "accepted": [bool(r.get("accepted")) for r in st.log],
            "solves_completed": int(sum(1 for r in st.log if r.get("terminated"))),
            "final_cost": next((r.get("cost") for r in reversed(st.log) if r.get("cost") is not None and r.get("cost") == r.get("cost")), None)}


LAST_STEP_FIELDS = ("lambda", "cost", "l_diff", "relative_decrease", "cg_iterations", "accepted", "terminated")
DUMP_BUDGET_BYTES = 64 * 10**6


def dump_outputs(out_dir, lin, last):
    """What the timed LM loop hands its caller after its last step, as DIR/<name>.npy: the camera and landmark state (the
    landmarks of this rank's shard) in the solver's scalar type, and that step's record (LAST_STEP_FIELDS, float64).
    Landmarks that would exceed DUMP_BUDGET_BYTES are cut to a fixed, seeded sample of rows, the same rows in every run."""
    lin.download_state()
    bp, stats = lin.bal_problem, lin.stats()
    lms = bp.lms[stats["landmark_begin"]:stats["landmark_end"]]
    room = (DUMP_BUDGET_BYTES - bp.cams.nbytes - 4096) // (3 * bp.lms.itemsize)
    if len(lms) > room:
        lms = lms[np.sort(np.random.default_rng(0).choice(len(lms), room, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("cameras", bp.cams), ("landmarks", lms),
                    ("last_step", np.array([last[k] for k in LAST_STEP_FIELDS], dtype=np.float64))):
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def bench_reference(args):
    """the reference's algorithm (CPU restatement, oracle/) on the host cores; rank 0 only"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle_py as orc
    dtype = np.float32 if args.dtype == "f32" else np.float64
    arrays = make_problem(args)
    cores = host_threads()
    o = orc.Oracle(arrays, dtype, orc.default_options(num_threads=cores))
    # thread count: fastest of a short sweep of the PCG operator on the linearised problem (the per-camera-lock scatter
    # of reduction_alg=1 stops scaling before all cores); done once, before the warm-up
    o.compute_error(); o.linearize(); o.solve(1e-4)
    used = tune_oracle_threads(o, 9 * arrays.nc, dtype, cores)
    be = OracleBackend(o)
    be.reset()
    warm = args.warmup if args.workload in ("ladybug-1723", "trafalgar-257") else min(args.warmup, 2)
    secs, wall, st, done = run_lm(be, dtype, warm, args.steps, budget_s=args.cpu_budget_s)
    ms = 1e3 * secs / done
    n_cg = sum(int(c) for c in trajectory_fields(st)["cg_iterations"] if c is not None)
    t = o.timings()
    sample = (f"LM iterations 1..{done} of the same trajectory (of the {args.steps} requested: wall-time budget {args.cpu_budget_s:.0f} s"
              f"{'' if done == args.steps else ', EXHAUSTED -- the early, cheaper iterations of the solve are over-represented'}), "
              f"{warm} warm-up iterations; OpenMP over landmarks with per-camera locks (reduction_alg=1); CPU restatement of the "
              f"reference (the reference itself cannot be built here); {used} of {cores} physical cores = the fastest of a short "
              f"sweep of the PCG operator")
    out = {
        "impl": "reference", "metric": METRIC, "value": ms, "unit": "ms/LM-iter", "n_gpus": args.gpus,
        "steps": args.steps, "steps_timed": done, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": False, "scaling": "strong",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": workload_config(args, arrays),
        "cpu_baseline": {"value": ms, "unit": "ms/LM-iter", "cores": used, "cores_available": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ms, "unit": "ms/LM-iter", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "pcg": {"iterations": n_cg},
        **trajectory_fields(st),
    }
    # SURVEY 8(d): "run with T = all cores and T = 1; report both": the PCG operator alone on one thread (bounded)
    if not args.no_single_thread:
        x = np.ones(9 * arrays.nc, dtype=dtype)
        o.set_options(orc.default_options(num_threads=1))
        t0 = time.perf_counter(); o.right_multiply(x); t1 = time.perf_counter() - t0
        o.set_options(orc.default_options(num_threads=used))
        t0 = time.perf_counter(); o.right_multiply(x); tn = time.perf_counter() - t0
        out["cpu_operator"] = {"ms_1_thread": 1e3 * t1, f"ms_{used}_threads": 1e3 * tn, "what": "one application of the PCG operator (ipp:400-441)"}
    del t
    print(json.dumps(out), flush=True)


def bench_ours(args):
    import torch
    import rootba_b200 as rb
    dtype = np.float32 if args.dtype == "f32" else np.float64
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    arrays = make_problem(args)

    def make_linearizor(single=False):
        bp = rb.BalProblem.from_arrays(arrays, dtype)
        so = rb.SolverOptions(use_double=(dtype == np.float64), device=local_rank, rank=0 if single else rank,
                              nranks=1 if single else world, operator_form=args.operator.upper())
        lin = rb.LinearizorQR.create(bp, so)
        if world > 1 and not single:
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid.copy_(torch.frombuffer(bytearray(rb.nccl_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            lin.comm_init(bytes(uid.cpu().numpy().tobytes()))
            # peer-memory exchange fused into the PCG kernels: all-gather the CUDA IPC handles
            mine = torch.frombuffer(bytearray(lin.ipc_export()), dtype=torch.uint8).cuda()
            allh = [torch.zeros(len(mine), dtype=torch.uint8, device="cuda") for _ in range(world)]
            dist.all_gather(allh, mine)
            lin.ipc_import(b"".join(bytes(t.cpu().numpy().tobytes()) for t in allh))
        return lin

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    PH = ("stage1_time", "stage2_time", "compute_preconditioner_time", "solve_reduced_system_time",
          "back_substitution_time", "update_cameras_time", "residual_evaluation_time")

    def timed_run(lin, sync=barrier):
        """device-resident run: returns (device seconds for K steps, wall, log holder, phases, per-step device ms, launches).
        The LM loop runs natively (rba_lm_run: optimize_lm_ours in the library, one host synchronisation per iteration, no
        interpreter between iterations); a solve that ends is followed by a new solve from the initial point."""
        be = GpuBackend(lin)
        phase = {k: 0.0 for k in PH}
        step_ms, log = [], []

        def run(nsteps, record):
            left = nsteps
            while left > 0:
                its, term, tot = lin.lm_run(left)
                if not its:
                    raise RuntimeError("rba_lm_run made no progress")
                left -= len(its)
                if record:
                    log.extend(its)
                    step_ms.extend(1e3 * i["device_seconds"] for i in its)
                    for k in PH:
                        phase[k] += tot[k]
                if left > 0:
                    be.reset()  # the solve ended: a new solve from the initial point
            # a solve that ends with the last step is not reset here: its state is the result of that step, and the
            # reset belongs to the next solve, which is not timed

        run(args.warmup, False)
        be.reset()
        sync()
        l0 = lin.timings()["kernel_launches"]
        t0 = time.perf_counter()
        lin.timer_start()
        run(args.steps, True)
        dev_s = lin.timer_stop()
        wall_s = time.perf_counter() - t0
        sync()

        class _Log:  # the fields trajectory_fields() reads
            pass
        st = _Log()
        st.log = log
        return dev_s, wall_s, st, phase, step_ms, lin.timings()["kernel_launches"] - l0

    # ---- device-resident run (value) ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    lin = make_linearizor()
    dev_s, wall_s, st, phase, step_ms, launches = timed_run(lin)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, lin, st.log[-1])
    secs = torch.tensor([dev_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(secs, op=dist.ReduceOp.MAX)
    ms = 1e3 * float(secs.item()) / args.steps
    # ---- roofline of the dominant kernel (rcs_matvec), timed alone with CUDA events ----
    mv_s = lin.time_matvec(200)
    stats = lin.stats()
    clocks = sampler.stop() if rank == 0 else {}
    mv_t = torch.tensor([mv_s], dtype=torch.float64, device="cuda")
    sz = 4 if dtype == np.float32 else 8
    dense_bytes = float(stats["matvec_algorithmic_bytes"])  # SURVEY 8(d): 18 M2 s + 18 Nobs s + 4 Nobs (dense Q2 panels)
    # implicit form: jp (18) + q1d (27) records + x gather (9) + per-observation y written and read back (9 + 9), cam index
    implicit_bytes = float(stats["num_observations_local"]) * (72 * sz + 4)
    mv_bytes = torch.tensor([implicit_bytes if args.operator == "implicit" else dense_bytes], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(mv_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(mv_bytes, op=dist.ReduceOp.SUM)
    peak, peak_src = hbm_peak()
    traffic = None
    try:  # DRAM bytes of the dominant kernel from the committed ncu --set full capture (same workload), per launch
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_matvec_traffic.json")))
        if args.workload == tj.get("workload") and args.scale == 1.0 and args.dtype == "f32" and world == 1 and args.operator == "dense":
            traffic = tj["traffic_bytes_per_launch"]
    except Exception:
        pass
    achieved = float(mv_bytes.item()) / float(mv_t.item()) / 1e9 / world  # per GPU
    traj = trajectory_fields(st)
    lin.close()
    # ---- end-to-end run through the host-buffer API ----
    lin2 = make_linearizor()
    be = GpuE2EBackend(lin2)

    def e2e_start():
        be.h2d = be.d2h = 0
    e2e_s, _, st2, _ = run_lm(be, dtype, args.warmup, args.steps, timer=(e2e_start, lambda: None), barrier=barrier)
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_ms = 1e3 * float(e2e_t.item()) / args.steps
    h2d, d2h = be.h2d // args.steps, be.d2h // args.steps
    lin2.close()
    # ---- the same workload on ONE GPU (rank 0 alone), so that a line measured at N > 1 carries its own N = 1 reference ----
    n1 = None
    if world > 1 and not args.no_n1:
        if rank == 0:
            lin1 = make_linearizor(single=True)
            d1, _, st1, ph1, _, _ = timed_run(lin1, sync=torch.cuda.synchronize)
            mv1 = lin1.time_matvec(50)
            cg1 = sum(int(c) for c in trajectory_fields(st1)["cg_iterations"] if c is not None)
            n1 = {"value": 1e3 * d1 / args.steps, "unit": "ms/LM-iter", "n_gpus": 1,
                  "what": "the same workload, protocol and trajectory on rank 0's GPU alone, measured in this run",
                  "pcg_us_per_iteration": 1e6 * ph1["solve_reduced_system_time"] / max(cg1, 1), "operator_us_per_launch": 1e6 * mv1,
                  "final_cost": trajectory_fields(st1)["final_cost"], "cg_iterations": trajectory_fields(st1)["cg_iterations"]}
            lin1.close()
        barrier()
    # ---- CPU baseline on a bounded sample (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle_py as orc
        cores = host_threads()
        o = orc.Oracle(arrays, dtype, orc.default_options(num_threads=cores))
        o.compute_error(); o.linearize(); o.solve(1e-4)
        used = tune_oracle_threads(o, 9 * arrays.nc, dtype, cores)
        bo = OracleBackend(o)
        bo.reset()
        n_cpu = min(args.steps, 6)
        cs, _, stc, done = run_lm(bo, dtype, 0, n_cpu, budget_s=30.0)
        cpu = {"value": 1e3 * cs / done, "unit": "ms/LM-iter", "cores": used, "cores_available": cores, "kind": "port",
               "sample": f"LM iterations 1..{done} of the same trajectory on the host cores (CPU restatement of the reference, OpenMP over "
                         f"landmarks with per-camera locks; thread count = fastest of a short sweep of the PCG operator; 30 s budget)",
               "cg_iterations": trajectory_fields(stc)["cg_iterations"]}
    if rank == 0:
        cfg = workload_config(args, arrays)
        cfg.update(parallelism=f"landmark-shard x{world}",
                   l2="inputs larger than L2 (Q2 panels %.0f MB per GPU vs 126 MB L2)" % (stats["panel_scalars"] * sz / 1e6))
        if args.operator == "implicit":
            cfg["solver"] += ", operator_form=IMPLICIT (opt-in)"
        out = {
            "metric": METRIC, "value": ms, "unit": "ms/LM-iter", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic", "config": cfg,
            "e2e": {"value": e2e_ms, "unit": "ms/LM-iter", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches),
            "clocks": {"sm_mhz": clocks.get("sm_mhz"), "sm_max_mhz": clocks.get("sm_max_mhz"), "reasons": clocks.get("reasons", [])},
            "roofline": {"bound": "hbm", "kernel": "rcs_matvec (k_matvec_implicit + camera reduction), bytes of the implicit form" if args.operator == "implicit"
                         else "rcs_matvec (k_matvec_small_tma + camera reduction)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": float(mv_bytes.item()) / world, "us_per_launch": 1e6 * float(mv_t.item())},
            "cpu_baseline": cpu,
            "phases_ms_per_step": {k: 1e3 * v / args.steps for k, v in phase.items()},
            "median_ms_per_step": float(np.median(step_ms)) if step_ms else None,
            "wall_ms_per_step": 1e3 * wall_s / args.steps,
            **traj,
        }
        # SURVEY 8(d): also report microseconds per PCG iteration (solve_reduced_system_time over the PCG iterations)
        n_cg = sum(int(c) for c in traj["cg_iterations"] if c is not None)
        out["pcg"] = {"iterations": n_cg,
                      "us_per_iteration": (1e6 * phase["solve_reduced_system_time"] / n_cg) if n_cg > 0 else None}
        if n1 is not None:
            out["same_workload_n1"] = n1
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOAD_LABEL),
                    help="default: ladybug-1723 at --gpus 1 (BASELINE configs[1]), venice-1778 at --gpus > 1 (configs[3])")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--seed", type=int, default=38401)
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-n1", action="store_true", help="N > 1: skip the single-GPU run of the same workload on rank 0")
    ap.add_argument("--no-single-thread", action="store_true", help="reference arm: skip the single-thread operator timing")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="reference arm: wall-time budget of the timed steps")
    ap.add_argument("--operator", default="dense", choices=["dense", "implicit"],
                    help="PCG operator form: dense = the reference's Q2-panel product (default, contract kernel); implicit = opt-in")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the state after the last one (cameras, landmarks) and that step's "
                         f"record (last_step: {', '.join(LAST_STEP_FIELDS)}) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computes (--impl ours)")
    if args.workload is None:
        args.workload = default_workload(args.gpus)
    if args.impl == "reference":
        bench_reference(args)
    else:
        bench_ours(args)


if __name__ == "__main__":
    main()
