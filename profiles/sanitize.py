"""Small invocations of every kernel for compute-sanitizer (memcheck / racecheck / initcheck are slow: tiny sizes)."""
import os, sys
import numpy as np
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, R); sys.path.insert(0, os.path.join(R, "tests"))
from conftest import get_model, mocap_of, quadruped_inputs
from mujoco_mpc_b200.engine import Engine
from mujoco_mpc_b200.ilqg import ILQGPlanner
which = sys.argv[1] if len(sys.argv) > 1 else "all"
m = get_model("quadruped")
e = Engine(m, 8, 12)
state, mocap, knots, kt = quadruped_inputs(m, N=4, H=10)
if which in ("all", "rollout"):
    for shape in ("wide", "plain"):                                            # static instances: helper warps / one warp
        os.environ["MJPC_B200_SHAPE"] = shape
        e.rollout_spline(state, 0.0, mocap, knots, kt, 2, 10)
        assert e.last_kernel_shape == (1 if shape == "wide" else 2)
    del os.environ["MJPC_B200_SHAPE"]
    os.environ["MJPC_B200_NO_STATIC"] = "1"
    e.rollout_spline(state, 0.0, mocap, knots, kt, 2, 10)                      # generic instance
    del os.environ["MJPC_B200_NO_STATIC"]
    e.set_xfrc_noise(1.0, 0.1, 3); e.rollout_spline(state, 0.0, mocap, knots, kt, 2, 10); e.set_xfrc_noise(0.0)
if which in ("all", "ilqg"):
    pl = ILQGPlanner(m, e, horizon=8, num_rollouts=4, fd_tolerance=1e-3)
    pl.set_state(state, 0.0, mocap)
    pl.optimize_policy()
if which in ("all", "humanoid"):
    mh = get_model("humanoid_track")
    eh = Engine(mh, 4, 10)
    mc = np.concatenate([mh.key_mpos[0].reshape(-1, 3), np.tile([1.0, 0, 0, 0], (mh.nmocap, 1))], 1).reshape(-1)
    sh = np.concatenate([mh.key_qpos[0], np.zeros(mh.nv)])
    kh = np.clip(0.1 * np.random.default_rng(0).standard_normal((2, 16, mh.nu)), -1, 1)
    for shape in ("wide", "plain"):
        os.environ["MJPC_B200_SHAPE"] = shape
        eh.rollout_spline(sh, 0.0, mc, kh, np.arange(16) * 0.003, 2, 8)
    del os.environ["MJPC_B200_SHAPE"]
    os.environ["MJPC_B200_NO_STATIC"] = "1"
    eh.rollout_spline(sh, 0.0, mc, kh, np.arange(16) * 0.003, 2, 8)
    del os.environ["MJPC_B200_NO_STATIC"]
    g = eh.step_debug(mh.qpos0, np.zeros(mh.nv), np.zeros(mh.nu), mc)
if which in ("all", "batched"):                                                # batched instances: 2 problems x 3 candidates
    M2 = 2
    args = (np.tile(state, (M2, 1)), np.arange(M2) * 0.1, np.tile(mocap, (M2, 1)), np.stack([knots[:3]] * M2),
            np.stack([kt + 0.1 * p for p in range(M2)]), 2, 10)
    for shape in ("wide", "plain"):
        os.environ["MJPC_B200_SHAPE"] = shape
        e.rollout_spline_batched(*args)
        assert e.last_kernel_shape == (1 if shape == "wide" else 2)
    del os.environ["MJPC_B200_SHAPE"]
    os.environ["MJPC_B200_NO_STATIC"] = "1"
    e.rollout_spline_batched(*args)                                            # generic instance
    del os.environ["MJPC_B200_NO_STATIC"]
print("sanitize run done:", which)
