#!/usr/bin/env python
"""Benchmark of the hot path: Quadruped (flat) Predictive Sampling, 256 candidates x 64-step horizon, fp32.

A "step" is one planning iteration's rollout batch (SamplingPlanner::Rollouts + ranking).  Metric: env-steps/sec
(BASELINE.json).

N = 1   256 x 64 = 16384 simulated environment steps per iteration (BASELINE configs[1]).
N > 1   ONE planning problem on all ranks: the same nominal policy everywhere, N x 256 candidates (weak scaling) drawn with
        GLOBAL candidate indices in the Philox counter, rank g rolls out its contiguous shard, one ncclAllGather of the
        per-candidate returns per iteration on the engine stream (mjpc_b200_rollout_spline_sharded), ranking on the device,
        winner trajectory broadcast from its owner.  The line also carries "strong": the 256-candidate problem of N = 1
        split over the N ranks, and the bitwise check of the sharded returns against a single-GPU run of the same problem.

  value      device-timed throughput (CUDA events on the engine's stream, per iteration; at N > 1 the span covers
             rollout kernel + all-gather + compaction + ranking), inputs resident in HBM at N = 1
  e2e        same metric through the public call with HOST buffers: H2D of state/mocap/knots, kernel(s), the collective at
             N > 1, D2H of returns/order and of the winner trajectory, all inside the timed region
  roofline   dominant kernel vs the measured HBM copy peak; algorithmic bytes per env-step are SURVEY.md 8(d)'s figure.
             The kernel is latency-bound by construction (DESIGN.md), so issue-slot evidence rides along.
  cpu_baseline  the CPU oracle (a port - the reference binary cannot be built offline) on this box's usable host cores,
             with the reference's own thread rule (nproc - 3) and the fp32 instantiation beside it.

--impl reference times that CPU path as its own arm.

Inputs: the nominal comes from a burn-in on the fp64 CPU oracle and the candidate noise from seeded Philox counters,
so the same arguments give the same inputs bit for bit, whichever build of the engine runs.
--dump-outputs DIR writes what the last timed step returned (DIR/<name>.npy, float32 / float64): the headline
launch's returns, failure flags, ranking and every candidate trajectory, and the end-to-end call's returns, failure
flags, ranking and winner trajectory (prefix e2e_).  Two builds are compared output for output on these files.

The bench runs on the library that build() left in the tree and writes nothing into the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # the tree may be read-only: no __pycache__ from the imports below

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_CAND, HORIZON, INTERP = 256, 64, 2
METRIC, UNIT = "env-steps/sec", "env-steps/s"
WORKLOAD = "Quadruped (flat) Predictive Sampling, 256 candidates x 64-step horizon, fp32"

BURN_IN = 30  # planning iterations (untimed, part of set-up) that take the zero policy to the steady-state nominal


def usable_cores():
    """Threads this process may actually run on: scheduler affinity capped by the cgroup CPU quota (os.cpu_count()
    reports the machine, not the container)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


class OracleBackend:
    """CPU oracle behind the same rollout_spline signature (only used by the CPU arms)."""

    def __init__(self, m, threads, precision=64):
        from mujoco_mpc_b200.blob import to_blob
        from oracle import pyoracle
        self.o, self.threads = pyoracle.Oracle(to_blob(m), m, precision), threads

    def rollout_spline(self, state, time, mocap, knots, kt, interp, H):
        r = self.o.rollout_spline(state, time, mocap, knots, kt, interp, H, nthreads=self.threads, full=False)
        return r["returns"], r["failure"], np.argsort(r["returns"], kind="stable")


def load_inputs(backend, n_iter, n_cand=N_CAND, burn_cand=N_CAND):
    """Model at the home keyframe (testspeed.cc:71-76); nominal spline = the planner's steady state: BURN_IN
    Predictive-Sampling iterations (burn_cand candidates) starting from the repeated initial action (SURVEY.md 8d);
    candidates of timed iteration i = nominal + Philox noise with counter (BURN_IN + i, GLOBAL candidate, knot, dof),
    candidate 0 un-noised.  Deterministic: every rank computes the same nominal."""
    from conftest import get_model, mocap_of
    from mujoco_mpc_b200.planner import SamplingPlanner, candidate_knots
    m = get_model("quadruped")
    state = np.concatenate([m.key_qpos[0], np.zeros(m.nv)])
    mocap = mocap_of(m)
    pl = SamplingPlanner(m, backend, num_trajectory=burn_cand, horizon=HORIZON, seed=0x5EED)
    pl.reset()
    pl.set_state(state, 0.0, mocap)
    for _ in range(BURN_IN):
        pl.optimize_policy()
    pl.make_candidates()  # resample the winner onto the knot grid
    knots = [candidate_knots(pl.values, pl.sigma, pl.ctrlrange, BURN_IN + it, n_cand, seed=pl.seed).astype(np.float32)
             for it in range(n_iter)]
    return m, state, mocap, knots, pl.times.copy(), float(np.min(pl.returns))


def algorithmic_bytes_per_env_step(m, P):
    ds, nu, nr, ntr = m.nq + m.nv, m.nu, m.task_num_residual, m.task_num_trace
    return 4 * (ds + nu + nr + 3 * ntr + 2) + 4 * (P * nu + ds + 7 * m.nmocap + m.nuserdata) / HORIZON


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index, self.t_mark = [], None, index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def mark(self):
        """Start of the timed region: only samples taken from here on are reported."""
        self.t_mark = time.time()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
        rows = [r for t, r in self.rows if self.t_mark is None or t >= self.t_mark]
        if not rows and self.rows:
            rows = [self.rows[-1][1]]

        def num(x):
            try:
                return float(x)
            except ValueError:
                return None
        sm = [num(r[0]) for r in rows if r and num(r[0]) is not None]
        mx = [num(r[1]) for r in rows if len(r) > 1 and num(r[1]) is not None]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_arm(m, state, mocap, knots, kt, threads, precision=64, budget_s=8.0, max_steps=3):
    """Time the CPU port on the given candidate sets: one untimed warm-up, then up to max_steps full steps or budget_s."""
    be = OracleBackend(m, threads, precision)
    be.rollout_spline(state, 0.0, mocap, knots[0][:max(threads, 8)], kt, INTERP, HORIZON)      # thread pool / page warm-up
    times, ret = [], None
    t_all = time.perf_counter()
    for it in range(max_steps):
        t0 = time.perf_counter()
        ret, _, _ = be.rollout_spline(state, 0.0, mocap, knots[it % len(knots)], kt, INTERP, HORIZON)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:
            break
    return float(np.mean(times)), len(times), ret


def ilqg_probe(m, eng, mocap, cpu_threads):
    """BASELINE config 4 (Quadruped iLQG, H=64, 10 line-search rollouts, centred FD with eps 3e-4 - the fp32 setting with
    which the planner follows the fp64 reference, csrc/host/ilqg_planner.h - skip 0, differentiable model):
    per-sweep device time (CUDA events around the kernels) and host wall time with host buffers, the roofline entry of
    each sweep kernel, and the same sweeps on the CPU port.  Reported beside the headline, not part of it."""
    from mujoco_mpc_b200.ilqg import ILQGPlanner
    pl = ILQGPlanner(m, eng, horizon=HORIZON, num_rollouts=10, fd_tolerance=3e-4, fd_mode=1)
    pl.set_state(np.concatenate([m.key_qpos[0], np.zeros(m.nv)]), 0.0, mocap)
    pl.nominal_trajectory()
    descent = [float(pl.cand["total_return"])]
    for _ in range(3):
        pl.optimize_policy(); descent.append(float(pl.total_return))
    pl.nominal_trajectory()
    c = pl.cand

    def tm(f, reps=5):
        f(); t0 = time.perf_counter(); dev = []
        for _ in range(reps):
            out = f(); dev.append(eng.last_kernel_ms)
        return (time.perf_counter() - t0) / reps * 1e3, float(np.mean(dev)), out
    t_fd, d_fd, (A, B, C, D) = tm(lambda: eng.model_derivatives(c["states"], c["actions"], c["times"], pl.mocap, 3e-4, mode=1))
    t_cd, d_cd, cd = tm(lambda: eng.cost_derivatives(c["residual"], C, D))
    t_bp, d_bp, bp = tm(lambda: eng.backward_pass(A, B, cd[0], cd[1], cd[2], cd[4], cd[3], c["actions"], mu=pl.regularization))
    t_ro, d_ro, _ = tm(lambda: eng.rollout_feedback(pl.state, 0.0, pl.mocap, c["actions"], c["states"], c["times"], bp["K"], bp["du"],
                                                    pl._steps(), 3))
    t_it, _, _ = tm(lambda: pl.optimize_policy())
    n, nu, nr, H = 2 * m.nv, m.nu, m.task_num_residual, HORIZON
    fd_steps = H * (1 + 2 * (nu + 2 * m.nv))          # centred: two evaluations per column + the centre
    peak = hbm_peak()[0]
    by_fd = 4 * H * (n * n + n * nu + nr * n + nr * nu)                       # A, B, C, D written once
    by_cd = 4 * H * (nr + nr * n + nr * nu + n + nu + n * n + nu * nu + n * nu)   # C, D, residual read; cx..cxu written
    by_bp = 4 * H * (n * n + n * nu + n + nu + n * n + n * nu + nu * nu + nu + nu * n + nu)
    fl_cd = 2.0 * H * nr * (n * n + n * nu + nu * nu)                           # Gauss-Newton products (upper bound: dense norm Hessian blocks)
    fl_bp = 2.0 * (H - 1) * (2 * n * n * n + 3 * n * n * nu + 2 * n * nu * nu + nu * nu * nu / 3)

    def roof(name, ms, nbytes, flops=None, note=""):
        r = {"kernel": name, "kernel_ms": ms, "bound": "latency (neither HBM nor tensor)", "algorithmic_bytes": nbytes,
             "achieved_gbs": nbytes / (ms * 1e-3) / 1e9, "hbm_frac": nbytes / (ms * 1e-3) / 1e9 / peak, "note": note}
        if flops:
            r["fp32_gflops"] = flops / (ms * 1e-3) / 1e9
        return r
    out = {"workload": "Quadruped (flat) iLQG, H=64, 10 line-search rollouts, centred FD (eps 3e-4: the fp32 setting; the CPU arm uses the reference's 1e-6 one-sided in fp64), skip 0, MakeDifferentiable on",
           "return_per_iteration_from_home_keyframe": descent,
           "fd_sweep_ms": t_fd, "fd_mj_step_equivalents": fd_steps, "fd_steps_per_s": fd_steps / (d_fd * 1e-3),
           "cost_derivatives_ms": t_cd, "backward_pass_ms": t_bp, "line_search_rollouts_ms": t_ro, "optimize_policy_ms": t_it,
           "device_ms": {"fd_sweep": d_fd, "cost_derivatives": d_cd, "backward_pass": d_bp, "line_search_rollouts": d_ro},
           "timing": "host wall clock around each C-ABI call with host buffers (…_ms) and CUDA events around the kernels (device_ms)",
           "roofline": [roof("fd_center_kernel + fd_column_kernel (%d one-warp mj_steps)" % fd_steps, d_fd, by_fd,
                             note="same device code as the rollout: dependent-instruction latency; the warps fill the SMs two per SM (shared memory)"),
                        roof("cost_derivatives_kernel", d_cd, by_cd, fl_cd, "one CTA per time step, shared-memory FMA"),
                        roof("backward_pass_kernel", d_bp, by_bp, fl_bp,
                             "strictly sequential in t: one CTA, 63 dependent Riccati steps (36 us each)")]}
    # the same sweeps on the CPU port (fp64 oracle; FD parallel over time steps as ModelDerivatives::Compute does)
    try:
        from conftest import OracleBackend as FullOracle
        ob = FullOracle(m, threads=cpu_threads)
        if pl.settings.differentiable:
            ob.set_differentiable(True)
        t0 = time.perf_counter(); Ao, Bo, Co, Do = ob.model_derivatives(c["states"], c["actions"], c["times"], pl.mocap, 1e-6); c_fd = time.perf_counter() - t0
        t0 = time.perf_counter(); cdo = ob.cost_derivatives(c["residual"], Co, Do); c_cd = time.perf_counter() - t0
        t0 = time.perf_counter(); ob.backward_pass(Ao, Bo, cdo[0], cdo[1], cdo[2], cdo[4], cdo[3], c["actions"], mu=pl.regularization); c_bp = time.perf_counter() - t0
        t0 = time.perf_counter()
        ob.rollout_feedback(pl.state, 0.0, pl.mocap, c["actions"], c["states"], c["times"], bp["K"], bp["du"], pl._steps(), 3)
        c_ro = time.perf_counter() - t0
        out["cpu_baseline"] = {"kind": "port", "cores": cpu_threads, "precision": "f64", "fd_sweep_ms": c_fd * 1e3,
                               "fd_steps_per_s": fd_steps / c_fd, "cost_derivatives_ms": c_cd * 1e3, "backward_pass_ms": c_bp * 1e3,
                               "line_search_rollouts_ms": c_ro * 1e3, "sample": "one pass of each sweep on the same nominal trajectory"}
    except Exception as e:  # noqa: BLE001 - the probe must never take the headline down
        out["cpu_baseline"] = {"error": repr(e)}
    return out


def humanoid_probe():
    """BASELINE config 3 task (Humanoid Track PS, H=128, 16 cubic knots, dt 0.005) at its per-GPU share of the 8-GPU
    configuration (128 of 1024 candidates): device-timed kernel of one planning iteration on the reference's keyframes."""
    from conftest import get_model
    from mujoco_mpc_b200.engine import Engine
    m = get_model("humanoid_track")
    N, H, P = 128, 128, 16
    e = Engine(m, N, H)
    mocap = np.concatenate([m.key_mpos[0].reshape(-1, 3), np.tile([1.0, 0, 0, 0], (m.nmocap, 1))], 1).reshape(-1)
    state = np.concatenate([m.key_qpos[0], m.key_qvel[0]])
    kt = np.arange(P) * (H - 1) * 0.005 / (P - 1)
    knots = np.clip(0.15 * np.random.default_rng(0).standard_normal((N, P, m.nu)), -1, 1); knots[0] = 0
    ms = []
    for i in range(6):
        ret, fail, _ = e.rollout_spline(state, 0.0, mocap, knots, kt, 2, H)
        if i >= 2:
            ms.append(e.last_kernel_ms)
    out = {"workload": "Humanoid Track PS, 128 candidates (1/8 of 1024) x 128 steps, 16 cubic knots, dt 0.005, fp32",
           "keyframes": getattr(m, "key_source", "?"),
           "kernel_ms": float(np.mean(ms)), "env_steps_per_s_per_gpu": N * H / (float(np.mean(ms)) * 1e-3),
           "static_kernel": bool(e.last_kernel_static), "failures": int(fail.sum())}
    e.close()
    return out


def shadow_probe(cpu_threads):
    """BASELINE config 5 task (Shadow Hand cube reorientation, PS 512 x 48, 5 cubic knots, dt 0.01) on the documented
    primitive-geom stand-in hand (mujoco_menagerie's meshes are not in the tree): generic kernels, device-timed, with
    the fp64 oracle on a 128-candidate share beside it."""
    from conftest import get_model
    from mujoco_mpc_b200.blob import to_blob
    from mujoco_mpc_b200.engine import Engine
    from mujoco_mpc_b200.planner import candidate_knots
    from oracle import pyoracle
    m = get_model("shadow_reorient")
    N, H, P = 512, 48, 5
    q0 = m.key_qpos[0]
    hold = np.zeros(m.nu)
    for i in range(m.nu):
        if m.actuator_trntype[i] == 0:
            hold[i] = q0[m.jnt_qposadr[m.actuator_trnid[i]]]
        else:
            t = m.actuator_trnid[i]
            hold[i] = sum(m.wrap_coef[w] * q0[m.wrap_qposadr[w]] for w in range(m.tendon_adr[t], m.tendon_adr[t] + m.tendon_num[t]))
    knots = candidate_knots(np.tile(hold, (P, 1)), 0.1, np.asarray(m.actuator_ctrlrange, float), 0, N, seed=7).astype(np.float32)
    kt = np.linspace(0.0, (H - 1) * m.opt_timestep, P)
    state = np.concatenate([q0, np.zeros(m.nv)])
    mocap = np.zeros(7 * m.nmocap)
    e = Engine(m, N, H)
    ms = []
    for i in range(6):
        ret, fail, _ = e.rollout_spline(state, 0.0, mocap, knots, kt, 2, H)
        if i >= 2:
            ms.append(e.last_kernel_ms)
    o = pyoracle.Oracle(to_blob(m), m, 64)
    o.rollout_spline(state, 0.0, mocap, knots[:16], kt, 2, H, nthreads=cpu_threads, full=False)
    t0 = time.perf_counter()
    r = o.rollout_spline(state, 0.0, mocap, knots[:128], kt, 2, H, nthreads=cpu_threads, full=False)
    cpu_s = time.perf_counter() - t0
    rel = np.abs(ret[:128] - r["returns"]) / np.abs(r["returns"])
    out = {"workload": "Shadow-Hand-shaped cube reorientation PS (STAND-IN hand: primitive geoms, same tree / dof / actuator / "
                       "tendon structure and task as shadow_reorient/task.xml), 512 candidates x 48 steps, 5 cubic knots, dt 0.01, fp32",
           "nq_nv_nu": [int(m.nq), int(m.nv), int(m.nu)], "residuals": int(m.task_num_residual),
           "kernel_ms": float(np.mean(ms)), "env_steps_per_s": N * H / (float(np.mean(ms)) * 1e-3),
           "static_kernel": bool(e.last_kernel_static), "failures": int(fail.sum()),
           "cpu_oracle_fp64": {"value": 128 * H / cpu_s, "threads": cpu_threads, "sample": "128 of the 512 candidates x 48 steps"},
           "parity_vs_fp64_oracle_128": {"median_rel": float(np.median(rel)), "max_rel": float(rel.max()), "above_1e-4": int((rel > 1e-4).sum())}}
    e.close()
    return out


def model_fidelity(m):
    """What of the reference model the compiled model keeps (recorded in the bench line so that the workload is auditable)."""
    import collections
    names = {0: "plane", 2: "sphere", 3: "capsule", 4: "ellipsoid", 5: "cylinder", 6: "box"}
    kept, dropped = collections.Counter(), collections.Counter()
    for a, b in zip(m.pair_geom1, m.pair_geom2):
        kept["-".join(sorted((names[int(m.geom_type[a])], names[int(m.geom_type[b])])))] += 1
    for a, b in getattr(m, "pairs_dropped", []):
        dropped["-".join(sorted((names[int(m.geom_type[a])], names[int(m.geom_type[b])])))] += 1
    return {"nq": int(m.nq), "nv": int(m.nv), "nu": int(m.nu), "ngeom": int(m.ngeom), "collision_pairs": dict(kept),
            "collision_pairs_dropped_no_narrow_phase": dict(dropped),
            "note": "pairs MuJoCo's filters keep; dropped types have no narrow phase here (cylinder / box against capsule, "
                    "cylinder, box - MuJoCo's convex / box-box routines) and are dropped on BOTH the device and the oracle"}


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT = 64 << 20   # bytes, all --dump-outputs files together


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as out_dir/<name>.npy; flags and indices are stored as float64 (exact)."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes (limit %d)" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_reference(args, rank, world):
    """--impl reference: the CPU port of the path (the reference binary cannot be built offline: MuJoCo is fetched at
    configure time) on all usable host cores, its own burn-in, bounded sample."""
    if rank != 0:
        return
    from conftest import get_model
    threads = usable_cores()
    be = OracleBackend(get_model("quadruped"), threads)
    m, state, mocap, knots, kt, _ = load_inputs(be, args.steps + args.warmup)
    times = []
    for it in range(args.steps + args.warmup):
        t0 = time.perf_counter()
        be.rollout_spline(state, 0.0, mocap, knots[it], kt, INTERP, HORIZON)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = float(np.mean(times))
    value = N_CAND * HORIZON / ms
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "backend": "CPU oracle (restatement of mj_step + Trajectory::Rollout, ThreadPool dispatch); "
                       "the reference binary cannot be built offline (MuJoCo is fetched at configure time)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "machine_threads": os.cpu_count(), "kind": "port",
                             "sample": "full workload: 256 candidates x 64 steps per step"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-probes", action="store_true", help="skip the iLQG / Humanoid Track probes (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", 0)); local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from mujoco_mpc_b200.engine import Engine
    n_iter = args.steps + args.warmup
    from conftest import get_model
    n_total = world * N_CAND                                   # one problem: N x 256 candidates
    clocks = ClockSampler(local)
    clocks.start()          # nvidia-smi needs ~0.5 s to produce its first row: started before the set-up / burn-in
    eng = Engine(get_model("quadruped"), N_CAND, HORIZON, device=local)
    if world > 1:
        eng.comm_init_torch(dist)                              # ncclCommInitRank inside libmjpc_b200.so
    # the burn-in runs on the fp64 CPU oracle with 256 candidates (its result does not depend on the thread count):
    # every rank, and every build of the engine, gets the same nominal
    burn_in = OracleBackend(get_model("quadruped"), max(1, usable_cores() // world))
    m, state, mocap, knots, kt, nominal_return = load_inputs(burn_in, n_iter, n_cand=n_total)
    P = knots[0].shape[1]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-timed region: one event pair per iteration, L2 flushed in between
    if world == 1:
        eng.upload_spline_inputs(state, 0.0, mocap, knots[0], kt, INTERP, HORIZON)
        eng.sync()
    kern_ms = []
    launches0 = 0
    for it in range(n_iter):
        if it == args.warmup:
            barrier()
            clocks.mark()
            launches0 = eng.launch_count
            t_wall0 = time.perf_counter()
        flush.zero_()
        barrier() if world > 1 else torch.cuda.synchronize()
        if world == 1:
            eng.launch_resident()
            eng.sync()
        else:
            sharded_out = eng.rollout_spline_sharded(state, 0.0, mocap, knots[it], kt, INTERP, HORIZON)
        if it >= args.warmup:
            kern_ms.append(eng.last_kernel_ms)
    barrier()
    wall = time.perf_counter() - t_wall0
    gpu_launches = eng.launch_count - launches0
    ms_per_step = max_over_ranks(float(np.sum(kern_ms))) / args.steps
    value = n_total * HORIZON / (ms_per_step * 1e-3)
    outputs = {}
    if args.dump_outputs and rank == 0:      # read back after the timed region: what the last timed step computed
        ret, fail, order = eng.read_returns() if world == 1 else sharded_out
        outputs.update(returns=ret, failure=fail, order=order)
        if world == 1:
            outputs.update(eng.fetch_all())

    # ---------------- end-to-end through the public call with host buffers (collective included at N > 1)
    ds, nu, nr, ntr = eng.ds, eng.nu, eng.nr, eng.ntr
    h2d = 4 * (ds + 7 * m.nmocap + eng.info.task_state_size + (n_total // world) * P * nu + P)
    d2h = n_total * (4 + 4 + 1) + HORIZON * (4 * (ds + nu + nr + ntr + 1) + 8)

    def e2e_step(it):
        if world == 1:
            ret, fail, order = eng.rollout_spline(state, 0.0, mocap, knots[it], kt, INTERP, HORIZON)
            best = eng.fetch_trajectory(int(order[0]))
        else:
            ret, fail, order = eng.rollout_spline_sharded(state, 0.0, mocap, knots[it], kt, INTERP, HORIZON)
            best = eng.fetch_trajectory_sharded(int(order[0]))     # ncclBroadcast from the winner's owner
        return ret, fail, order, best
    for it in range(args.warmup):
        e2e_step(it)
    barrier()
    t0 = time.perf_counter()
    for it in range(args.steps):
        ret, fail, order, best = e2e_step(args.warmup + it)
    barrier()
    e2e_value = n_total * HORIZON / max_over_ranks((time.perf_counter() - t0) / args.steps)
    if args.dump_outputs and rank == 0:
        outputs.update(e2e_returns=ret, e2e_failure=fail, e2e_order=order, **{"e2e_winner_" + k: v for k, v in best.items()})
    clk = clocks.stop()      # samples cover both timed regions (device-timed and end-to-end), 50 ms apart

    # ---------------- N > 1: one-problem evidence + strong scaling of the 256-candidate problem
    multi = None
    if world > 1:
        # identical returns / order / winner on every rank
        h = torch.tensor([float(np.sum(ret.astype(np.float64) * np.arange(1, n_total + 1))), float(order[0]),
                          float(np.abs(best["states"]).sum())], dtype=torch.float64, device="cuda")
        hmin, hmax = h.clone(), h.clone()
        dist.all_reduce(hmin, op=dist.ReduceOp.MIN); dist.all_reduce(hmax, op=dist.ReduceOp.MAX)
        identical = bool(torch.equal(hmin, hmax))
        # strong scaling: the N = 1 problem (256 candidates) over all ranks
        kn = knots[-1][:N_CAND]
        s_ms = []
        for it in range(args.warmup + min(args.steps, 20)):
            flush.zero_(); barrier()
            sret, sfail, sorder = eng.rollout_spline_sharded(state, 0.0, mocap, kn, kt, INTERP, HORIZON)
            if it >= args.warmup:
                s_ms.append(eng.last_kernel_ms)
        strong_ms = max_over_ranks(float(np.mean(s_ms)))
        bitwise = None
        if rank == 0:
            single = Engine(get_model("quadruped"), N_CAND, HORIZON, device=local)     # no communicator: one GPU, same problem
            r1, f1, o1 = single.rollout_spline(state, 0.0, mocap, kn, kt, INTERP, HORIZON)
            bitwise = bool(np.array_equal(r1.view(np.uint32), sret.view(np.uint32)) and np.array_equal(o1, sorder))
            single.close()
        multi = {"one_problem": True, "candidates_total": n_total, "identical_returns_order_winner_on_all_ranks": identical,
                 "sharded_equals_single_gpu_bitwise": bitwise, "comm": "ncclAllGather of (return, failure) per candidate on the engine stream "
                 "inside libmjpc_b200.so; ranking on the device; winner trajectory ncclBroadcast from its owner",
                 "strong": {"workload": "256 candidates total x 64 steps over %d GPUs" % world, "ms_per_step": strong_ms,
                            "value": N_CAND * HORIZON / (strong_ms * 1e-3), "unit": UNIT}}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---------------- parity + roofline + CPU baseline (rank 0)
    peak, peak_src = hbm_peak()
    bytes_per_launch = algorithmic_bytes_per_env_step(m, P) * (n_total // world) * HORIZON
    kernel_ms = float(np.mean(kern_ms))
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "kernel": "rollout_kernel_quadruped" if eng.last_kernel_static else "rollout_kernel", "kernel_ms": kernel_ms, "peak_source": peak_src,
                "algorithmic_bytes_per_env_step": algorithmic_bytes_per_env_step(m, P),
                "note": "latency/occupancy-bound by construction: 256 candidates, 64 dependent steps each; one main warp per candidate plus helper warps for the wide phases (DESIGN.md section 5)",
                "kernel_shape": int(eng.last_kernel_shape)}
    for prof in ("traffic_r02.json", "traffic_r01.json"):
        pp = os.path.join(ROOT, "profiles", prof)
        if os.path.exists(pp):
            pj = json.load(open(pp))
            roofline["traffic"] = pj.get("dram_bytes_per_launch")
            # what actually bounds the kernel (from the committed ncu capture of the same launch): issue-slot use and stalls
            roofline["latency_bound_evidence"] = {k: pj[k] for k in ("smsp__issue_active_pct", "sm__warps_active_pct_of_peak",
                                                                     "warp_instructions_per_env_step", "warp_instructions_per_env_step_main_warp",
                                                                     "stall_mix_pct", "stall_mix_pct_main_warp",
                                                                     "counters_from") if k in pj}
            break
    cores = usable_cores()
    probes = world == 1 and not args.no_probes
    ilqg = ilqg_probe(m, eng, mocap, cores) if probes else None
    config3 = humanoid_probe() if probes else None
    config5 = shadow_probe(cores) if probes else None
    cpu = None
    parity = None
    if not args.no_cpu_baseline and world == 1:     # the CPU arm is reported at N = 1 only
        # same inputs as the GPU arm (the last timed candidate sets); bounded: <= 3 steps or ~8 s per arm
        cpu_s, n_s, cpu_ret = cpu_arm(m, state, mocap, knots[-3:], kt, cores)
        ref_threads = max(1, cores - 3)              # the reference's own rule: planner_threads = nproc - 3 (agent.cc:153-154)
        ref_s, _, _ = cpu_arm(m, state, mocap, knots[-3:], kt, ref_threads, max_steps=2)
        f32_s, _, r32 = cpu_arm(m, state, mocap, knots[-3:], kt, cores, precision=32, max_steps=2)
        cpu = {"value": N_CAND * HORIZON / cpu_s, "unit": UNIT, "cores": cores, "machine_threads": os.cpu_count(), "kind": "port",
               "sample": "%d full steps (256 candidates x 64 steps each) on the GPU arm's own candidate sets, fp64 oracle, "
                         "ThreadPool over all usable host threads (affinity / cgroup quota)" % n_s,
               "reference_thread_rule": {"threads": ref_threads, "value": N_CAND * HORIZON / ref_s,
                                         "note": "planner_threads = nproc - 3 (agent.cc:153-154)"},
               "fp32_oracle": {"threads": cores, "value": N_CAND * HORIZON / f32_s,
                               "note": "same arithmetic width as the kernels (BASELINE.md section 3)"}}
        # parity on identical inputs: the CPU arm's last candidate set through the device path
        c_knots = knots[-3:][(n_s - 1) % 3]
        gret, _, gorder = eng.rollout_spline(state, 0.0, mocap, c_knots, kt, INTERP, HORIZON)
        from mujoco_mpc_b200.blob import to_blob
        from oracle import pyoracle
        ops, _ = pyoracle.count_flops(to_blob(m), state, 0.0, mocap, c_knots[:4], kt, INTERP, HORIZON)
        roofline["oracle_ops_per_env_step"] = ops
        roofline["achieved_tflops_at_oracle_op_count"] = ops * value / world / 1e12
        roofline["fp32_note"] = "operation count of the dense CPU restatement (instrumented scalar); the kernel exploits the dof-tree sparsity and executes fewer"
        rel = np.abs(gret - cpu_ret) / np.maximum(np.abs(cpu_ret), 1e-12)
        o32 = pyoracle.Oracle(to_blob(m), m, 32)
        r32 = o32.rollout_spline(state, 0.0, mocap, c_knots, kt, INTERP, HORIZON, nthreads=cores, full=False)["returns"]
        floor = np.abs(r32 - cpu_ret) / np.maximum(np.abs(cpu_ret), 1e-12)
        # conditioning of each candidate's return, from the fp64 oracle alone: inputs rounded to fp32 and 5 random
        # perturbations of the initial velocity of size 1e-5 (= one teacher-forced fp32 step error); a return that moves
        # by > 2e-5 under ONE of them cannot be pinned to 1e-4 through 64 such steps (tests/test_gpu_teacher_forced.py)
        o64 = pyoracle.Oracle(to_blob(m), m, 64)
        rng = np.random.default_rng(12345)
        variants = [np.asarray(state, np.float32).astype(float)]
        for _ in range(5):
            sv = np.asarray(state, float).copy(); sv[m.nq:] += 1e-5 * rng.standard_normal(m.nv)
            variants.append(sv)
        worst = np.zeros(len(cpu_ret))
        for sv in variants:
            rp = o64.rollout_spline(sv, 0.0, mocap, c_knots.astype(float), kt, INTERP, HORIZON, nthreads=cores, full=False)["returns"]
            worst = np.maximum(worst, np.abs(rp - cpu_ret) / np.abs(cpu_ret))
        stable = worst <= 2e-5
        parity = {"max_rel_return_err_vs_fp64_oracle": float(rel.max()), "mean_rel": float(rel.mean()),
                  "median_rel_vs_fp64_oracle": float(np.median(rel)),
                  "candidates_above_1e-4_vs_fp64": int((rel > 1e-4).sum()),
                  "well_conditioned_candidates": int(stable.sum()),
                  "max_rel_on_well_conditioned_candidates": float(rel[stable].max()) if stable.any() else None,
                  "well_conditioned_candidates_above_1e-4": int((rel[stable] > 1e-4).sum()),
                  "fp32_oracle_vs_fp64_oracle": {"max_rel": float(floor.max()), "median_rel": float(np.median(floor)),
                                                 "candidates_above_1e-4": int((floor > 1e-4).sum())},
                  "argmin_agrees": bool(int(gorder[0]) == int(np.argmin(cpu_ret))),
                  "note": "well-conditioned = the fp64 oracle's own return moves < 2e-5 when the inputs are rounded to fp32 or the "
                          "initial velocity is perturbed by 1e-5 (one teacher-forced fp32 step error); teacher-forced per-step "
                          "parity at 256x64 is asserted in tests/test_gpu_teacher_forced.py"}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD if world == 1 else WORKLOAD + "; N GPUs: one planning problem, %d candidates sharded %d per GPU" % (n_total, N_CAND),
                       "model": model_fidelity(m), "candidates_per_gpu": N_CAND, "candidates_total": n_total, "horizon": HORIZON, "spline_points": P,
                       "nominal": "steady-state policy after %d planning iterations of the fp64 CPU oracle from the zero policy (return %.4f)" % (BURN_IN, nominal_return),
                       "l2": "flushed between timed iterations (256 MB memset)",
                       "sharding": "one problem, contiguous candidate ranges, one ncclAllGather of returns per iteration" if world > 1 else "single GPU",
                       "e2e_call": ("Engine.rollout_spline (mjpc_b200_rollout_spline) + fetch_trajectory(winner), host buffers" if world == 1 else
                                    "Engine.rollout_spline_sharded (mjpc_b200_rollout_spline_sharded: H2D, kernel, ncclAllGather, rank, D2H) + "
                                    "fetch_trajectory_sharded(winner: ncclBroadcast), host buffers")},
            "clocks": clk, "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(gpu_launches), "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "ilqg": ilqg, "humanoid_track": config3, "shadow_reorient_standin": config5,
            "multi_gpu": multi, "wall_s_timed_region": wall}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
