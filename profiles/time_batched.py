"""One batched launch of M planning problems (mjpc_b200_rollout_spline_batched) against M sequential single-problem
calls (mjpc_b200_rollout_spline) on the same handle.  Quadruped, H = 64, P = 3, for several (M, N), plus Humanoid Track
(4, 32) at H = 128.  The two ways alternate within each case (which goes first alternates too); the L2 is flushed
(256 MB memset) before each of them.  Device ms = CUDA events of the engine (rollout + ranking; summed over the M
sequential calls), end-to-end ms = host clock around the call(s) including staging and copies.  The outputs of the two
ways are compared bit for bit.  Prints one JSON line; with an argument, also writes it to that file."""
import json
import os
import subprocess
import sys
import time

import numpy as np

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
sys.path.insert(0, os.path.join(R, "tests"))
sys.dont_write_bytecode = True

WARMUP, ITERS = 3, 30


def problems(m, name, M, N, H):
    from conftest import mocap_of
    from mujoco_mpc_b200.planner import candidate_knots
    rng = np.random.default_rng(M * 1000 + N)
    cr = np.asarray(m.actuator_ctrlrange, float).reshape(-1, 2)
    q0 = m.key_qpos[0] if name == "quadruped" else m.qpos0
    st, tm, kn, kt = [], [], [], []
    for p in range(M):
        s = np.concatenate([q0, np.zeros(m.nv)])
        s[7: m.nq] += 0.01 * p * rng.standard_normal(m.nq - 7)
        t = 0.1 * p
        st.append(s); tm.append(t)
        kn.append(candidate_knots(np.zeros((3, m.nu)), 0.04, cr, p, N))
        kt.append(t + np.arange(3) * (H - 1) * m.opt_timestep / 2)
    return np.array(st), np.array(tm), np.tile(mocap_of(m), (M, 1)), np.array(kn), np.array(kt)


def stats(x):
    x = np.asarray(x)
    return {"median": float(np.median(x)), "min": float(x.min()), "p10": float(np.percentile(x, 10)),
            "p90": float(np.percentile(x, 90)), "max": float(x.max())}


def run_case(e, m, name, M, N, H, flush):
    import torch
    st, tm, mc, kn, kt = problems(m, name, M, N, H)
    dev = {"batched": [], "sequential": []}
    e2e = {"batched": [], "sequential": []}
    equal = True

    def batched():
        t0 = time.perf_counter()
        r = e.rollout_spline_batched(st, tm, mc, kn, kt, 2, H)
        return time.perf_counter() - t0, e.last_kernel_ms, r

    def sequential():
        t0, ms, out = time.perf_counter(), 0.0, []
        for p in range(M):
            out.append(e.rollout_spline(st[p], tm[p], mc[p], kn[p], kt[p], 2, H))
            ms += e.last_kernel_ms
        return time.perf_counter() - t0, ms, tuple(np.stack(x) for x in zip(*out))

    for it in range(WARMUP + ITERS):
        res = {}
        for way in (("batched", "sequential") if it % 2 == 0 else ("sequential", "batched")):
            flush.zero_()
            torch.cuda.synchronize()
            res[way] = (batched if way == "batched" else sequential)()
        if it >= WARMUP:
            for way, (s, ms, _) in res.items():
                e2e[way].append(1e3 * s); dev[way].append(ms)
        equal &= all(np.array_equal(a, b) for a, b in zip(res["batched"][2], res["sequential"][2]))
    med = {k: float(np.median(v)) for k, v in dev.items()}
    med_e2e = {k: float(np.median(v)) for k, v in e2e.items()}
    return {"model": name, "M": M, "N": N, "H": H, "candidates": M * N, "bitwise_equal": bool(equal),
            "device_ms": {k: stats(v) for k, v in dev.items()}, "end_to_end_ms": {k: stats(v) for k, v in e2e.items()},
            "speedup_device": med["sequential"] / med["batched"], "speedup_end_to_end": med_e2e["sequential"] / med_e2e["batched"]}


def main():
    import torch
    from conftest import get_model
    from mujoco_mpc_b200.engine import Engine
    if not torch.cuda.is_available():
        raise SystemExit("time_batched.py measures on a CUDA device; none is visible")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    try:
        power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = None
    cases = []
    m = get_model("quadruped")
    e = Engine(m, 300, 64)
    for M, N in ((8, 32), (4, 64), (2, 128), (4, 74), (3, 100), (16, 16)):
        cases.append(run_case(e, m, "quadruped", M, N, 64, flush))
    e.close()
    h = get_model("humanoid_track")
    e = Engine(h, 128, 128)
    cases.append(run_case(e, h, "humanoid_track", 4, 32, 128, flush))
    e.close()
    line = {"script": "profiles/time_batched.py", "gpu": torch.cuda.get_device_name(0), "power_limit_and_max_sm_clock": power,
            "warmup": WARMUP, "iterations": ITERS, "l2": "flushed (256 MB memset) before each timed way", "cases": cases}
    text = json.dumps(line)
    print(text, flush=True)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
