#!/usr/bin/env python
"""bench.py -- LM iterations/s of the joint-optimisation hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU algorithm
                                                           (oracle port; the reference itself
                                                           cannot be built here, DESIGN.md)
  ... --dump-outputs DIR                                   also write the state and report of the
                                                           last timed step as DIR/<name>.npy

One "step" = one LM iteration = one call of OptimizeJointly(max_iteration_count=1): one H/b
build over all observations, >= 1 Schur solve, >= 1 trial-cost pass (SURVEY.md 8d).
Workload: BASELINE config 2 -- central-generic B-spline camera 2050x1450 (84x60 grid, 10 080
intrinsics), 500 imagesets, 2 000 pattern points, ~0.95 M observations, seed 2, synthetic.
Under torchrun the imagesets are sharded over the ranks (strong scaling: the problem is fixed).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree, which may be read-only

_emit = None
BYTES_PER_OBS = {0: 720, 1: 1488, 3: 400}  # SURVEY.md 8(d): algorithmic bytes of the Jacobian kernel (C = 1)
DUMP_LIMIT_BYTES = 64 * 1000 * 1000  # --dump-outputs: data bytes written in all


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [v.strip() for v in out.split(",")]
                self.samples.append((float(f[0]), float(f[1])))
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(s[1] for s in self.samples),
                "reasons": sorted(self.reasons), "samples": len(sm)}


def _workload_cache_path(args):
    """File of this user's private workload cache for these arguments, or None when no private
    directory is available. The name carries a digest of the generator's source, so a changed
    generator never reads a workload an older one wrote."""
    import hashlib
    from camera_calibration_b200 import cabi, synthetic
    h = hashlib.sha256()
    for m in (synthetic, cabi):
        with open(m.__file__, "rb") as f:
            h.update(f.read())
    d = os.path.join(tempfile.gettempdir(), f"b200ba_workload_{os.getuid()}")
    try:
        os.makedirs(d, mode=0o700, exist_ok=True)
        st = os.stat(d)
    except OSError:
        return None
    if st.st_uid != os.getuid() or st.st_mode & 0o077:
        return None  # another user could write there, and the cache is unpickled
    return os.path.join(d, f"c{args.config}_i{args.imagesets}_{h.hexdigest()[:16]}.pkl")


def make_workload(args):
    """Seeded synthetic problem: the same arguments give the same inputs on every run. Cached in a
    private temporary directory so that several bench invocations on one machine (and the ranks of
    one torchrun) do not regenerate it -- generation is deterministic and takes about a minute."""
    import pickle
    from camera_calibration_b200 import synthetic
    kw = {}
    if args.imagesets:
        kw["n_imagesets"] = args.imagesets
    cache = _workload_cache_path(args)
    if cache and os.path.exists(cache):
        try:
            d = pickle.load(open(cache, "rb"))
            from camera_calibration_b200.cabi import Camera, FlatProblem, FlatState
            cams = []
            for f in d["cams"]:
                c = Camera()
                for k, v in f.items():
                    setattr(c, k, v)
                cams.append(c)
            pb = FlatProblem(cams, d["n_imagesets"], d["n_points"], d["oi"], d["oc"], d["op"], d["oxy"])
            zlp = lambda a: a if a is not None else np.zeros((len(d["oi"]), 2))  # all-zero caches are not stored
            mk = lambda t: FlatState(t[0], t[1], t[2], t[3], zlp(t[4]))
            return synthetic.SyntheticProblem(d["name"], pb, mk(d["init"]), mk(d["gt"]), d["seed"], d["info"])
        except Exception:
            pass
    sp = synthetic.make_problem(args.config, **kw)
    if not cache:
        return sp
    try:
        p = sp.problem
        st = lambda s: (s.points, s.rig_tr_global, s.camera_tr_rig, s.intrinsics,
                        None if (s.last_projection is None or not np.any(s.last_projection)) else s.last_projection)
        d = dict(cams=[{k: getattr(c, k) for k, _ in c._fields_} for c in p.cameras], n_imagesets=p.n_imagesets,
                 n_points=p.n_points, oi=p.obs_imageset, oc=p.obs_camera, op=p.obs_point, oxy=p.obs_xy,
                 init=st(sp.init_state), gt=st(sp.gt_state), seed=sp.seed, info=sp.info, name=sp.name)
        tmp = cache + f".{os.getpid()}"
        pickle.dump(d, open(tmp, "wb"))
        os.replace(tmp, cache)
    except Exception:
        pass
    return sp


STOP_THRESHOLD = 1e-4  # cost_reduction_threshold of the product's final BA runs (APP/calibration.cc:1110,1124)
MAX_TRAJECTORY = 100   # their max_iteration_count


def cpu_baseline_sampled(sp, opt_numeric, budget_s=20.0):
    """FALLBACK (labelled as such in the output): the CPU port timed on a bounded sample and scaled to
    one full LM iteration = 1 Compute<true> + 1 Schur solve + 1 Compute<false>. Used only when the box
    has too few host cores for a complete iteration to fit the time budget."""
    from oracle import oracle
    p = sp.problem
    n_upd = sum(c.update_parameter_count() for c in p.cameras)
    nd = 6 * p.n_imagesets + (6 * p.n_cameras if p.n_cameras > 1 else 0) + n_upd
    nbd = 3 * p.n_points
    k = max(1, min(p.n_imagesets, 2))
    t_j = oracle.time_jacobian(p, sp.init_state, opt_numeric, 0, k, True)
    per = t_j / k
    k2 = int(max(k, min(p.n_imagesets, (0.45 * budget_s) / max(per, 1e-9))))
    if k2 > k:
        t_j = oracle.time_jacobian(p, sp.init_state, opt_numeric, 0, k2, True)
        k = k2
    obs_frac = float(np.sum(p.obs_imageset < k)) / max(1, p.n_obs)
    t_jac_full = t_j / max(obs_frac, 1e-12)
    t_r = oracle.time_jacobian(p, sp.init_state, opt_numeric, 0, k, False)
    t_res_full = t_r / max(obs_frac, 1e-12)
    nc = int(min(nd, 1200))
    t_c = oracle.time_contraction(nbd, nc)
    t_con_full = t_c * (nd / nc) ** 2
    nl = int(min(nd, 1800))
    t_l = oracle.time_ldlt(nl)
    t_ldlt_full = t_l * (nd / nl) ** 3
    total = t_jac_full + t_res_full + t_con_full + t_ldlt_full
    sample = (f"SAMPLED ESTIMATE (fallback): Compute<true> on {k} of {p.n_imagesets} imagesets ({t_j:.1f}s), Compute<false> on "
              f"the same ({t_r:.1f}s), B^T D^-1 B on {nc} of {nd} dense columns ({t_c:.1f}s, x(nd/nc)^2), pivoted LDLT at "
              f"n={nl} of {nd} ({t_l:.1f}s, x(nd/n)^3); single thread, unblocked loops")
    return {"value": 1.0 / total, "unit": "LM iterations/s", "cores": 1, "kind": "port", "sample": sample,
            "seconds_per_iteration": total,
            "breakdown_s": {"jacobian": t_jac_full, "residual": t_res_full, "contraction": t_con_full, "ldlt": t_ldlt_full}}


def physical_cores() -> int:
    """Physical cores of the host (hyper-threads do not help the FMA-bound dense kernels)."""
    try:
        seen = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    seen.add((phys, core))
                phys = core = None
        if seen:
            return len(seen)
    except OSError:
        pass
    return os.cpu_count() or 1


class CpuTrajectory:
    """The reference's CPU algorithm (oracle port, NUMERIC Jacobians like the reference) driven exactly
    like the GPU arm: single LM iterations from the start state under the stop rule of
    RunBundleAdjustment (APP/calibration.cc:298-300), restarted when it triggers. Every step is one
    COMPLETE LM iteration of the full workload -- nothing is sampled or extrapolated."""

    def __init__(self, sp, threads=0):
        from camera_calibration_b200 import cabi
        from oracle import oracle
        self.oracle = oracle
        # one thread per physical core, pinned and spread over the sockets (must be set before libgomp starts)
        os.environ.setdefault("OMP_PROC_BIND", "spread")
        os.environ.setdefault("OMP_PLACES", "cores")
        self.threads = oracle.use_native(threads if threads > 0 else physical_cores())  # -march=native, built for this CPU
        self.sp = sp
        self.opt = cabi.default_options(jacobian_mode=cabi.JACOBIAN_NUMERIC, max_iteration_count=1)
        # start state: the perturbed initial state with the projection cache warmed by one residual pass
        # (the product enters BA with PointFeature::last_projection filled by the previous stage)
        st = sp.init_state.copy()
        ev = oracle.evaluate(sp.problem, st, self.opt, False)
        if isinstance(ev, dict) and "last_projection" in ev:
            st.last_projection = ev["last_projection"]
        self.start = st
        self._reset()
        self.breakdown = {"cost_and_jacobian_s": 0.0, "solve_s": 0.0}
        self.attempts = []

    def _reset(self):
        self.state = self.start.copy()
        self.lam = -1.0
        self.last_cost = float("inf")
        self.n_in_traj = 0

    def step(self):
        self.opt.init_lambda = self.lam
        t0 = time.perf_counter()
        self.state, rep = self.oracle.optimize(self.sp.problem, self.state, self.opt)
        dt = time.perf_counter() - t0
        self.last = (self.state, rep)  # what this step returned, kept across a restart of the trajectory
        self.lam = rep.final_lambda
        self.breakdown["cost_and_jacobian_s"] += rep.cost_and_jacobian_evaluation_time
        self.breakdown["solve_s"] += rep.solve_time
        self.attempts.append(int(rep.trace_attempts[0]) if rep.trace_len else 0)
        cost = rep.final_cost
        self.n_in_traj += 1
        if cost >= self.last_cost - STOP_THRESHOLD or not rep.performed_an_iteration or self.n_in_traj >= MAX_TRAJECTORY:
            self._reset()
        else:
            self.last_cost = cost
        return dt, cost


def dump_outputs(out_dir, state, rep):
    """Writes what one timed step returns to its caller -- the state after the step and its report --
    as float64 DIR/<name>.npy, so that two builds can be compared output for output on the same
    inputs. last_projection (two values per observation) is the only array that grows with the
    workload: when everything would exceed DUMP_LIMIT_BYTES, a fixed, seeded sample of its rows is
    written instead, together with their indices (last_projection_rows)."""
    arrays = {"points": state.points, "rig_tr_global": state.rig_tr_global, "camera_tr_rig": state.camera_tr_rig}
    for c, a in enumerate(state.intrinsics):
        arrays[f"intrinsics_{c}"] = a
    for k in ("initial_cost", "final_cost", "final_lambda", "rmse", "n_valid", "n_invalid", "num_iterations_performed",
              "performed_an_iteration"):
        arrays[k] = getattr(rep, k)
    arrays["trace_cost"], arrays["trace_lambda"], arrays["trace_attempts"] = rep.trace()
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    lp = np.asarray(state.last_projection, dtype=np.float64)
    room = DUMP_LIMIT_BYTES - sum(a.nbytes for a in arrays.values())
    if lp.nbytes <= room:
        arrays["last_projection"] = lp
    else:
        per_row = lp[0].nbytes + 8  # the row and its index
        rows = np.sort(np.random.default_rng(0).choice(len(lp), room // per_row, replace=False))
        arrays["last_projection"] = lp[rows]
        arrays["last_projection_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)
    return {"dir": out_dir, "arrays": sorted(arrays), "bytes": int(sum(a.nbytes for a in arrays.values())),
            "last_projection_sampled": "last_projection_rows" in arrays}


def cpu_baseline(sp, budget_s=60.0):
    """One complete NUMERIC LM iteration of the oracle port at full size on all host cores (falls back
    to the labelled sampled estimate when the box has fewer than 4 cores)."""
    cores = os.cpu_count() or 1
    if cores < 4:
        from camera_calibration_b200 import cabi
        return cpu_baseline_sampled(sp, cabi.default_options(jacobian_mode=cabi.JACOBIAN_NUMERIC), budget_s=min(budget_s, 20.0))
    traj = CpuTrajectory(sp)
    dt, cost = traj.step()
    return {"value": 1.0 / dt, "unit": "LM iterations/s", "cores": traj.threads, "kind": "port",
            "sample": f"1 complete LM iteration (NUMERIC Jacobians, full workload, first iteration from the start state) in {dt:.1f} s on "
                      f"{traj.threads} host threads; blocked + OpenMP dense kernels (oracle/ba_dense_fast.h), -march=native",
            "seconds_per_iteration": dt, "cost_after": cost, "lm_attempts": traj.attempts[-1],
            "breakdown_s": dict(traj.breakdown)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sp = make_workload(args)
    traj = CpuTrajectory(sp, threads=args.cpu_threads)
    W = min(args.warmup, 1)  # a CPU code path needs no more than one untimed pass
    K = max(1, args.steps)
    for _ in range(W):
        traj.step()
    traj.attempts.clear()
    traj.breakdown = {"cost_and_jacobian_s": 0.0, "solve_s": 0.0}
    t_total, done, costs = 0.0, 0, []
    while done < K:
        dt, cost = traj.step()
        t_total += dt
        done += 1
        costs.append(cost)
        if t_total > args.cpu_budget and done >= 1:
            break  # bounded: as many COMPLETE iterations as fit the budget (steps reports the count)
    sec = t_total / done
    val = 1.0 / sec
    sample = (f"{done} complete LM iterations (NUMERIC Jacobians, full workload, trajectory from the start state under the reference's "
              f"stop rule) on {traj.threads} host threads; blocked + OpenMP dense kernels, -march=native; nothing sampled or extrapolated")
    line = {
        "impl": "reference", "metric": "LM iterations/sec", "value": val, "unit": "LM iterations/s",
        "n_gpus": args.gpus, "steps": done, "warmup": W, "ms_per_step": 1e3 * sec,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(sp, args, max(1, args.gpus)),  # the same config object as the b200 arm's line
        "cpu_baseline": {"value": val, "unit": "LM iterations/s", "cores": traj.threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "LM iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "attempts_per_step": traj.attempts, "costs": costs,
        "breakdown_s_per_step": {k: v / done for k, v in traj.breakdown.items()},
        "steps_requested": K,
    }
    if args.dump_outputs:
        line["dump_outputs"] = dump_outputs(args.dump_outputs, *traj.last)
    _emit(line)
    return 0


def workload_config(sp, args, world):
    c = sp.problem.cameras[0]
    return {"workload": f"BASELINE config {args.config}: " + {1: "CentralOpenCV 12-param", 2: "central-generic B-spline",
                                                              3: "noncentral-generic B-spline", 4: "2x central-generic rig",
                                                              5: "4x central-generic rig"}[args.config],
            "n_obs": sp.n_obs, "n_imagesets": sp.problem.n_imagesets, "n_points": sp.problem.n_points,
            "n_cameras": sp.problem.n_cameras, "grid": [c.grid_width, c.grid_height],
            "intrinsic_unknowns": sum(cc.update_parameter_count() for cc in sp.problem.cameras), "seed": sp.seed,
            "options": "eliminate_points=1 localize_only=0 huber=1 max_lm_attempts=50 init_lambda=-1",
            "step": ("one LM iteration = OptimizeJointly(max_iteration_count=1); iterations run as trajectories from the "
                     "(projection-cache-warmed) start state under the reference's stop rule cost >= last - 1e-4 "
                     "(calibration.cc:298-300), restarted from a device-side snapshot (untimed) when it triggers"),
            "parallelism": f"imageset-sharded x{world}" if world > 1 else "single GPU",
            "l2": "inputs larger than L2 (per step: B 0.6 GB, C 1.4 GB, S 1.4 GB >> 126 MB)"}


def measure_fp64_peak(torch):
    """Burst FP64 GEMM rate of the box (cuBLAS dgemm 8192^3, best of 3): the denominator of the
    rooflines of the two dense phases (MEASURED_PEAKS.json only carries bf16)."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def run_b200(args):
    import torch
    from camera_calibration_b200 import api, cabi, distributed
    rank, world, local = distributed.env_rank_world()
    dist = None
    if world > 1:
        dist = distributed.init_process_group("nccl")
    torch.cuda.set_device(local)
    sp = make_workload(args)
    opt = cabi.default_options(max_iteration_count=1)
    if world > 1:
        adj, idx = distributed.make_sharded_adjuster(sp.problem)
        state0 = distributed.shard_state(sp.init_state, idx)
    else:
        adj = api.BundleAdjuster(sp.problem, local)
        state0 = sp.init_state.copy()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    W, K = max(3, args.warmup), max(1, args.steps)
    sampler = ClockSampler(local)
    fp64_peak = measure_fp64_peak(torch) if rank == 0 else None

    # ---- start state: perturbed initial state + projection cache warmed by one residual pass -------
    adj.set_state(state0)
    adj.evaluate_device(opt)          # untimed; fills last_projection on the device
    adj.snapshot_state()              # device-side copy the trajectories restart from
    start_host = adj.get_state()      # the same start state in host buffers (e2e leg)

    class Traj:
        """Single LM iterations under the stop rule of RunBundleAdjustment, restarted from the snapshot."""

        def __init__(self):
            self.lam, self.last, self.n = -1.0, float("inf"), 0
            self.lengths = []

        def after(self, rep, restore):
            self.lam = rep.final_lambda
            self.n += 1
            cost = rep.final_cost
            if cost >= self.last - STOP_THRESHOLD or not rep.performed_an_iteration or self.n >= MAX_TRAJECTORY:
                self.lengths.append(self.n)
                restore()
                self.lam, self.last, self.n = -1.0, float("inf"), 0
            else:
                self.last = cost

    # ---- device-resident: the state stays in HBM between steps ---------------------------------------
    tr = Traj()
    first_traj_costs = []
    for _ in range(W):
        opt.init_lambda = tr.lam
        rep = adj.optimize(opt)
        if not tr.lengths:
            first_traj_costs.append(rep.final_cost)
        tr.after(rep, adj.restore_state)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    dev_ms = 0.0
    jac_ms, jac_n, launches = 0.0, 0, 0
    phases = {"jacobian": 0.0, "straggler": 0.0, "accumulate": 0.0, "schur": 0.0, "factor": 0.0, "solve": 0.0, "trial": 0.0,
              "update": 0.0, "allreduce": 0.0}
    attempts, builds, step_ms, costs = [], 0, [], []
    con_flops = fac_flops = 0.0
    rmse = None
    restore_wall = 0.0
    dumped, dump_wall = None, 0.0
    for i in range(K):
        opt.init_lambda = tr.lam
        rep = adj.optimize(opt)
        if args.dump_outputs and i == K - 1:
            # read back before the stop rule may restore the start state; untimed in `value` and in wall_ms
            tw = time.perf_counter()
            dumped = (adj.get_state(), rep)
            dump_wall = time.perf_counter() - tw
        t = adj.timings()
        dev_ms += t.total_ms
        step_ms.append(t.total_ms)
        jac_ms += t.jacobian_kernel_ms
        jac_n += t.jacobian_kernel_launches
        launches += t.kernel_launches
        attempts.append(int(t.lm_attempts))
        builds += int(t.build_count)
        con_flops += t.contraction_flops
        fac_flops += t.factor_flops
        for k, v in (("jacobian", t.jacobian_kernel_ms), ("straggler", t.straggler_ms), ("accumulate", t.accumulate_ms),
                     ("schur", t.schur_ms), ("factor", t.factor_ms - t.solve_ms), ("solve", t.solve_ms), ("trial", t.trial_cost_ms),
                     ("update", t.update_ms), ("allreduce", t.allreduce_ms)):
            phases[k] += v / K
        costs.append(rep.final_cost)
        if not tr.lengths:
            first_traj_costs.append(rep.final_cost)
        rmse = rep.rmse
        tr_before = len(tr.lengths)
        tw = time.perf_counter()
        tr.after(rep, adj.restore_state)
        if len(tr.lengths) != tr_before:
            restore_wall += time.perf_counter() - tw  # untimed in `value`; reported
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0 - restore_wall - dump_wall)
    traj_lengths = list(tr.lengths)

    # ---- end to end: host buffers in, host buffers out, every step (b200ba_optimize_host) ---------------
    # the caller's state buffers live in pinned host memory (the copies in the timed region are
    # plain DMA transfers, as the e2e contract asks)
    pinned = []

    def pin(a):
        try:
            t = torch.empty(a.shape, dtype=torch.float64).pin_memory()
        except Exception:  # pragma: no cover - pinning refused: stay pageable
            return a.copy()
        pinned.append(t)
        v = t.numpy()
        v[...] = a
        return v
    st = start_host.copy()
    st.points, st.rig_tr_global, st.camera_tr_rig = pin(st.points), pin(st.rig_tr_global), pin(st.camera_tr_rig)
    st.intrinsics = [pin(a) for a in st.intrinsics]
    st.last_projection = pin(st.last_projection)

    def restore_host():
        st.points[...] = start_host.points
        st.rig_tr_global[...] = start_host.rig_tr_global
        st.camera_tr_rig[...] = start_host.camera_tr_rig
        for a, b in zip(st.intrinsics, start_host.intrinsics):
            a[...] = b
        st.last_projection[...] = start_host.last_projection

    tr2 = Traj()
    for _ in range(W):
        opt.init_lambda = tr2.lam
        rep2 = adj.optimize_host(st, opt)
        tr2.after(rep2, restore_host)
    barrier()
    e2e_s = 0.0
    e2e_attempts = []
    for _ in range(K):
        opt.init_lambda = tr2.lam
        t1 = time.perf_counter()
        rep2 = adj.optimize_host(st, opt)   # returns after the D2H copy of the state has completed
        e2e_s += time.perf_counter() - t1
        e2e_attempts.append(int(adj.timings().lm_attempts))
        tr2.after(rep2, restore_host)       # host-side reset of the caller's buffers: untimed
    barrier()
    e2e_ms = 1e3 * e2e_s
    clocks = sampler.stop()  # sampled over both timed regions (device-resident and end-to-end)
    state_bytes = 8 * (st.points.size + st.rig_tr_global.size + st.camera_tr_rig.size + sum(a.size for a in st.intrinsics)
                       + st.last_projection.size)

    # max over ranks
    if dist is not None:
        tt = torch.tensor([dev_ms, wall_ms, e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, e2e_ms = [float(v) for v in tt.tolist()]
    ms_per_step = max(dev_ms, 0.0) / K
    value = 1e3 / ms_per_step
    peak, peak_src = _peaks()
    n_local = adj.problem.n_obs
    model = sp.problem.cameras[0].model_type
    bpo = BYTES_PER_OBS.get(model, 720) + (96 if sp.problem.n_cameras > 1 else 0)
    jac_avg_ms = jac_ms / max(1, jac_n)
    achieved = n_local * bpo / (jac_avg_ms * 1e-3) / 1e9 if jac_avg_ms > 0 else 0.0
    traffic = None
    prof = os.path.join(ROOT, "profiles", "jacobian_kernel_latest.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None

    if rank == 0:
        n_att = max(1, sum(attempts))
        schur_s = phases["schur"] * K * 1e-3
        fact_s = phases["factor"] * K * 1e-3
        line = {
            "metric": "LM iterations/sec", "value": value, "unit": "LM iterations/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(sp, args, world),
            "wall_ms_per_step": wall_ms / K, "final_cost": costs[-1], "rmse_px": rmse,
            "attempts_per_step": attempts, "attempts_mean": sum(attempts) / K, "step_ms": [round(v, 3) for v in step_ms],
            "trajectory_lengths": traj_lengths, "first_trajectory_costs": first_traj_costs,
            "phases_ms_per_step": phases,
            "phases_ms_per_attempt": {k: phases[k] * K / n_att for k in ("schur", "factor", "solve", "trial", "update")},
            "roofline": {"kernel": "residual_jacobian_kernel", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_obs": bpo, "obs_per_launch": n_local, "avg_launch_ms": jac_avg_ms},
            "roofline_dense": {
                "peak_tflops": fp64_peak, "peak_source": "cuBLAS dgemm 8192^3 measured in this run (burst, best of 3)",
                "contraction": {"flops_per_step": con_flops / K, "tflops": con_flops / max(schur_s, 1e-12) / 1e12,
                                "frac": con_flops / max(schur_s, 1e-12) / 1e12 / fp64_peak if fp64_peak else None,
                                "note": "whole Schur phase (block factorisations, gathers, rank-k updates, scatters)"},
                "factor": {"flops_per_step": fac_flops / K, "tflops": fac_flops / max(fact_s, 1e-12) / 1e12,
                           "frac": fac_flops / max(fact_s, 1e-12) / 1e12 / fp64_peak if fp64_peak else None}},
            "e2e": {"value": 1e3 / (e2e_ms / K), "unit": "LM iterations/s", "h2d_bytes_per_step": int(state_bytes),
                    "d2h_bytes_per_step": int(state_bytes), "ms_per_step": e2e_ms / K, "attempts_mean": sum(e2e_attempts) / K,
                    "host_memory": "pinned" if pinned else "pageable"},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        # parity across GPU counts: the first trajectory against the committed 1-GPU trajectory of this config
        tp = os.path.join(ROOT, "profiles", f"r02_config{args.config}_trajectory.json")
        if os.path.exists(tp) and not args.imagesets:
            try:
                ref = json.load(open(tp))["first_trajectory_costs"]
                m = min(len(ref), len(first_traj_costs))
                if m:
                    line["parity_vs_1gpu"] = {"iterations_compared": m, "reference": os.path.relpath(tp, ROOT),
                                              "max_rel_cost_diff": max(abs(a - b) / abs(b) for a, b in zip(first_traj_costs[:m], ref[:m]))}
            except Exception:
                pass
        line["dense_path"] = ("in-tree sm_100a kernels: DMMA contraction with scatter epilogue, blocked Cholesky on packed "
                              "panels (fused tile factor + inverse launch), packed triangular solves (ba_dense.cu, ba_tile.cuh)") if os.environ.get("B200BA_DENSE", "own") not in ("lib", "0") \
            else "cuBLAS dsyrk + cuSOLVER potrf / potrs (B200BA_DENSE=lib)"
        if dumped is not None:
            line["dump_outputs"] = dump_outputs(args.dump_outputs, *dumped)
    adj.close()
    adj = None
    if rank == 0:
        if world == 1 and os.environ.get("B200BA_DENSE", "own") not in ("lib", "0") and not args.no_library_comparison:
            # the same steps with the dense phase on cuBLAS / cuSOLVER: the bar the in-tree kernels are measured against
            os.environ["B200BA_DENSE"] = "lib"
            try:
                ladj = api.BundleAdjuster(sp.problem, local)
                ladj.set_state(state0)
                ladj.evaluate_device(opt)
                lam_l, tot, n_l = -1.0, 0.0, 0
                lph = {"schur": 0.0, "factor": 0.0, "solve": 0.0}
                for i in range(7):
                    opt.init_lambda = lam_l
                    r_l = ladj.optimize(opt)
                    lam_l = r_l.final_lambda
                    if i >= 2:
                        t_l = ladj.timings()
                        tot += t_l.total_ms
                        n_l += 1
                        lph["schur"] += t_l.schur_ms
                        lph["factor"] += t_l.factor_ms - t_l.solve_ms
                        lph["solve"] += t_l.solve_ms
                ladj.close()
                line["library_path"] = {"ms_per_step": tot / n_l, "steps": n_l,
                                        "phases_ms_per_step": {k: v / n_l for k, v in lph.items()},
                                        "what": "cuBLAS dsyrk + cuSOLVER potrf / potrs for the dense phase, everything else identical"}
            finally:
                os.environ.pop("B200BA_DENSE", None)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(sp, budget_s=args.cpu_budget)
        _emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed LM iterations (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--imagesets", type=int, default=0, help="shrink the workload (debugging only)")
    ap.add_argument("--cpu-budget", type=float, default=600.0,
                    help="--impl reference: stop after the first complete iteration that ends beyond this many seconds")
    ap.add_argument("--cpu-threads", type=int, default=0, help="host threads of the CPU arm (0 = all cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-comparison", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the state and report the last one returned as DIR/<name>.npy "
                         "(float64, at most 64 MB; with several GPUs, rank 0's view: its shard of last_projection)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # Exactly ONE line goes to stdout (the JSON line): libraries (NCCL prints its version banner)
    # write to fd 1 directly, so fd 1 is pointed at stderr until the result is ready.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    result = {}

    def emit(line):
        result["line"] = line

    global _emit
    _emit = emit
    try:
        rc = run_reference(args) if args.impl == "reference" else run_b200(args)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if "line" in result:
        print(json.dumps(result["line"]), flush=True)
    return rc


if __name__ == "__main__":
    sys.exit(main())
