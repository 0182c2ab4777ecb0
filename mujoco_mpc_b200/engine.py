"""ctypes binding of libmjpc_b200.so - the reference-facing call a user makes.

Every method goes through the C ABI in include/mjpc_b200.h; there is no Python/NumPy compute path and no
CPU fallback: if the library is missing or no B200 is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .blob import to_blob
from .build import SO

_fp = C.POINTER(C.c_float)
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_bp = C.POINTER(C.c_uint8)

EXPORTS = ["mjpc_b200_version", "mjpc_b200_last_error", "mjpc_b200_create", "mjpc_b200_destroy",
           "mjpc_b200_get_info", "mjpc_b200_set_task", "mjpc_b200_set_differentiable", "mjpc_b200_set_xfrc_noise", "mjpc_b200_rollout_spline", "mjpc_b200_rollout_spline_batched", "mjpc_b200_rollout_feedback",
           "mjpc_b200_fetch_trajectory", "mjpc_b200_fetch_all", "mjpc_b200_model_derivatives",
           "mjpc_b200_cost_derivatives", "mjpc_b200_backward_pass", "mjpc_b200_step_debug", "mjpc_b200_step_batch", "mjpc_b200_comm_unique_id", "mjpc_b200_comm_init",
           "mjpc_b200_comm_info", "mjpc_b200_rollout_spline_sharded", "mjpc_b200_fetch_trajectory_sharded",
           "mjpc_b200_fetch_stats", "mjpc_b200_launch_count", "mjpc_b200_last_kernel_ms", "mjpc_b200_last_kernel_static",
           "mjpc_b200_spec_words", "mjpc_b200_upload_spline_inputs",
           "mjpc_b200_launch_resident", "mjpc_b200_sync", "mjpc_b200_read_returns", "mjpc_b200_stream",
           "mjpc_b200_device_returns", "mjpc_b200_host_spline_sample", "mjpc_b200_host_philox_normal",
           "mjpc_b200_planner_create", "mjpc_b200_planner_destroy", "mjpc_b200_planner_set_exploration", "mjpc_b200_planner_reset",
           "mjpc_b200_planner_set_state", "mjpc_b200_planner_optimize_policy",
           "mjpc_b200_planner_action_from_policy", "mjpc_b200_planner_get_result",
           "mjpc_b200_batch_planner_create", "mjpc_b200_batch_planner_destroy", "mjpc_b200_batch_planner_reset",
           "mjpc_b200_batch_planner_set_state", "mjpc_b200_batch_planner_set_task", "mjpc_b200_batch_planner_optimize_policy",
           "mjpc_b200_batch_planner_action_from_policy", "mjpc_b200_batch_planner_get_result",
           "mjpc_b200_ce_planner_create", "mjpc_b200_ce_planner_destroy", "mjpc_b200_ce_planner_reset",
           "mjpc_b200_ce_planner_set_state", "mjpc_b200_ce_planner_optimize_policy",
           "mjpc_b200_ce_planner_action_from_policy", "mjpc_b200_ce_planner_get_result",
           "mjpc_b200_ilqg_planner_create", "mjpc_b200_ilqg_planner_destroy", "mjpc_b200_ilqg_planner_set_fd",
           "mjpc_b200_gradient_planner_set_fd", "mjpc_b200_ilqs_planner_set_fd", "mjpc_b200_ilqg_planner_reset",
           "mjpc_b200_ilqg_planner_set_state", "mjpc_b200_ilqg_planner_nominal_trajectory",
           "mjpc_b200_ilqg_planner_optimize_policy", "mjpc_b200_ilqg_planner_action_from_policy",
           "mjpc_b200_ilqg_planner_get_result", "mjpc_b200_host_ilqg_policy_action",
           "mjpc_b200_robust_planner_create", "mjpc_b200_robust_planner_destroy", "mjpc_b200_robust_planner_reset",
           "mjpc_b200_robust_planner_set_state", "mjpc_b200_robust_planner_optimize_policy",
           "mjpc_b200_robust_planner_action_from_policy", "mjpc_b200_robust_planner_get_result",
           "mjpc_b200_gradient_planner_create", "mjpc_b200_gradient_planner_destroy", "mjpc_b200_gradient_planner_reset",
           "mjpc_b200_gradient_planner_set_state", "mjpc_b200_gradient_planner_optimize_policy",
           "mjpc_b200_gradient_planner_action_from_policy", "mjpc_b200_gradient_planner_get_result",
           "mjpc_b200_host_spline_mapping", "mjpc_b200_ilqs_planner_create", "mjpc_b200_ilqs_planner_destroy",
           "mjpc_b200_ilqs_planner_reset", "mjpc_b200_ilqs_planner_set_state", "mjpc_b200_ilqs_planner_set_exploration",
           "mjpc_b200_ilqs_planner_optimize_policy", "mjpc_b200_ilqs_planner_action_from_policy",
           "mjpc_b200_ilqs_planner_get_result",
           "mjpc_b200_set_options", "mjpc_b200_agent_steps", "mjpc_b200_agent_create", "mjpc_b200_agent_destroy",
           "mjpc_b200_agent_reset", "mjpc_b200_agent_set_state", "mjpc_b200_agent_set_task", "mjpc_b200_agent_set_plan_enabled",
           "mjpc_b200_agent_plan_iteration", "mjpc_b200_agent_get_steps", "mjpc_b200_agent_action_from_policy",
           "mjpc_b200_quadruped_transition_create", "mjpc_b200_quadruped_transition_destroy",
           "mjpc_b200_quadruped_transition_step", "mjpc_b200_quadruped_transition_set", "mjpc_b200_track_transition_create",
           "mjpc_b200_track_transition_destroy", "mjpc_b200_track_transition_step", "mjpc_b200_shadow_transition_create",
           "mjpc_b200_shadow_transition_destroy", "mjpc_b200_shadow_transition_step"]


class ModelBlob(C.Structure):
    _fields_ = [("data", C.c_void_p), ("nbytes", C.c_size_t)]


class TaskDesc(C.Structure):
    _fields_ = [("weight", _dp), ("parameters", _dp), ("task_state", _dp), ("risk", C.c_double)]


class TaskBatch(C.Structure):
    _fields_ = [("weight", _dp), ("parameters", _dp), ("task_state", _dp)]


class Info(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("nq", "nv", "nu", "na", "nmocap", "nuserdata", "dim_state", "dim_dstate",
                                       "num_residual", "num_term", "num_trace", "num_parameters", "task_state_size",
                                       "max_candidates", "max_horizon", "device", "smem_bytes_per_warp")]


_LIB = None


def load_library():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO):
            raise RuntimeError(f"{SO} not built: run `python -m mujoco_mpc_b200.build` (no fallback path exists)")
        lib = C.CDLL(SO)
        lib.mjpc_b200_version.restype = C.c_char_p
        lib.mjpc_b200_last_error.restype = C.c_char_p
        lib.mjpc_b200_launch_count.restype = C.c_int64
        lib.mjpc_b200_last_kernel_ms.restype = C.c_float
        lib.mjpc_b200_stream.restype = C.c_void_p
        lib.mjpc_b200_device_returns.restype = C.c_void_p
        lib.mjpc_b200_host_philox_normal.restype = C.c_double
        lib.mjpc_b200_planner_destroy.argtypes = [C.c_void_p]
        lib.mjpc_b200_planner_set_exploration.argtypes = [C.c_void_p, C.c_double, C.c_double]
        lib.mjpc_b200_ce_planner_destroy.argtypes = [C.c_void_p]
        lib.mjpc_b200_batch_planner_destroy.argtypes = [C.c_void_p]
        lib.mjpc_b200_ilqg_planner_destroy.argtypes = [C.c_void_p]
        for n in ("mjpc_b200_ilqg_planner_set_fd", "mjpc_b200_gradient_planner_set_fd", "mjpc_b200_ilqs_planner_set_fd"):
            getattr(lib, n).argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_int]
            getattr(lib, n).restype = None
        lib.mjpc_b200_robust_planner_destroy.argtypes = [C.c_void_p]
        lib.mjpc_b200_gradient_planner_destroy.argtypes = [C.c_void_p]
        lib.mjpc_b200_agent_destroy.argtypes = [C.c_void_p]
        lib.mjpc_b200_agent_steps.argtypes = [C.c_double, C.c_double]
        lib.mjpc_b200_set_options.argtypes = [C.c_void_p, C.c_double, C.c_int]
        lib.mjpc_b200_ilqs_planner_destroy.argtypes = [C.c_void_p]
        lib.mjpc_b200_ilqs_planner_set_exploration.argtypes = [C.c_void_p, C.c_double]
        lib.mjpc_b200_shadow_transition_destroy.argtypes = [C.c_void_p]
        for n in ("mjpc_b200_quadruped_transition_create", "mjpc_b200_track_transition_create", "mjpc_b200_shadow_transition_create"):
            getattr(lib, n).restype = C.c_void_p
        lib.mjpc_b200_quadruped_transition_destroy.argtypes = [C.c_void_p]
        lib.mjpc_b200_track_transition_destroy.argtypes = [C.c_void_p]
        for n in ("mjpc_b200_destroy", "mjpc_b200_fetch_stats", "mjpc_b200_launch_count", "mjpc_b200_last_kernel_ms", "mjpc_b200_stream",
                  "mjpc_b200_device_returns", "mjpc_b200_sync", "mjpc_b200_launch_resident"):
            getattr(lib, n).argtypes = [C.c_void_p]
        _LIB = lib
    return _LIB


class EngineError(RuntimeError):
    pass


def host_ilqg_policy_action(model, u_nom, x_nom, t_nom, gains, representation, feedback_scaling, state, time):
    """iLQGPolicy::Action (ilqg/policy.cc:82-161) on the host through mjpc_b200_host_ilqg_policy_action (no device)."""
    lib = load_library()
    blob = to_blob(model)
    buf = C.create_string_buffer(blob, len(blob))
    mb = ModelBlob(C.cast(buf, C.c_void_p), len(blob))
    u, x, t, g = _f(u_nom), _f(x_nom), _d(t_nom), _f(gains)
    st = _d(state)
    out = np.zeros(model.nu)
    rc = lib.mjpc_b200_host_ilqg_policy_action(C.byref(mb), _pf(u), _pf(x), _pd(t), _pf(g), int(u.shape[0]), int(representation),
                                               C.c_double(feedback_scaling), _pd(st), C.c_double(time), _pd(out))
    if rc != 0:
        raise EngineError(f"host_ilqg_policy_action failed ({rc})")
    return out


def _f(a):
    return None if a is None else np.ascontiguousarray(a, np.float32)


def _d(a):
    return None if a is None else np.ascontiguousarray(a, np.float64)


def _pf(a):
    return None if a is None else a.ctypes.data_as(_fp)


def _pd(a):
    return None if a is None else a.ctypes.data_as(_dp)


def batched_inputs(m, state, time, mocap, knots, knot_times, weight=None, parameters=None, task_state=None):
    """The arguments of Engine.rollout_spline_batched for model m as contiguous arrays of the C ABI's types; raises
    ValueError when a shape does not fit knots [M][N][P][nu]."""
    knots = _f(knots)
    if knots.ndim != 4 or knots.shape[3] != m.nu or min(knots.shape) < 1:
        raise ValueError(f"knots must be [M][N][P][{m.nu}], got {knots.shape}")
    M, N, P, _ = knots.shape

    def rows(a, width, conv, name, optional=False):
        if a is None:
            if optional:
                return None
            raise ValueError(f"{name} is required")
        a = conv(a)
        if a.shape != (M, width):
            raise ValueError(f"{name} must be [{M}][{width}], got {a.shape}")
        return a
    tm = _d(time)
    if tm.shape != (M,):
        raise ValueError(f"time must be [{M}], got {tm.shape}")
    return (rows(state, m.nq + m.nv, _f, "state"), tm, rows(mocap, 7 * m.nmocap, _f, "mocap") if m.nmocap else None,
            knots, rows(knot_times, P, _d, "knot_times"), rows(weight, len(m.task_weight), _d, "weight", True),
            rows(parameters, len(m.task_parameters), _d, "parameters", True),
            rows(task_state, len(m.task_state), _d, "task_state", True))


class Engine:
    """One handle = one GPU's share of the candidates (Planner::Initialize/Allocate analogue)."""

    def __init__(self, model, max_candidates=256, max_horizon=64, device=0):
        self.lib = load_library()
        self.m = model
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_create(C.byref(mb), int(max_candidates), int(max_horizon), int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"mjpc_b200_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h = h
        info = Info()
        self._check(self.lib.mjpc_b200_get_info(self.h, C.byref(info)))
        self.info = info
        self.ds, self.n, self.nu, self.nr = info.dim_state, info.dim_dstate, info.nu, info.num_residual
        self.ntr = 3 * info.num_trace
        self.lastN = self.lastH = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc):
        if rc != 0:
            raise EngineError(f"mjpc_b200 error {rc}: {self.lib.mjpc_b200_last_error().decode()}")

    # ---- task snapshot (Agent::PlanIteration, agent.cc:316-319)
    def set_task(self, weight=None, parameters=None, task_state=None, risk=None):
        w, p, s = _d(weight), _d(parameters), _d(task_state)
        td = TaskDesc(_pd(w), _pd(p), _pd(s), float(self.m.task_risk if risk is None else risk))
        self._check(self.lib.mjpc_b200_set_task(self.h, C.byref(td)))

    def set_options(self, timestep, integrator=0):
        """Agent::PlanIteration's planning-model overrides (agent.cc:288-289)."""
        self._check(self.lib.mjpc_b200_set_options(self.h, C.c_double(timestep), int(integrator)))

    def set_differentiable(self, on=True):
        """MakeDifferentiable (utilities.cc:60-75): solimp[0] = 0 for joints and geoms while planning with gradients."""
        self._check(self.lib.mjpc_b200_set_differentiable(self.h, int(bool(on))))

    # ---- SamplingPlanner::Rollouts
    def rollout_spline(self, state, time, mocap, knots, knot_times, interp, H, want_order=True):
        knots = _f(knots)
        N, P, nu = knots.shape
        st, mc, kt = _f(state), _f(mocap), _d(knot_times)
        ret = np.zeros(N, np.float32); fail = np.zeros(N, np.uint8); order = np.zeros(N, np.int32)
        self._check(self.lib.mjpc_b200_rollout_spline(self.h, _pf(st), C.c_double(time), _pf(mc), None, _pf(knots),
                                                      _pd(kt), int(interp), P, N, int(H), _pf(ret),
                                                      fail.ctypes.data_as(_bp), order.ctypes.data_as(_ip)))
        self.lastN, self.lastH = N, H
        return ret, fail, order

    def rollout_spline_batched(self, state, time, mocap, knots, knot_times, interp, H, weight=None, parameters=None,
                               task_state=None):
        """M independent problems in one launch (mjpc_b200_rollout_spline_batched): state [M][dim_state], time [M],
        mocap [M][7 nmocap], knots [M][N][P][nu], knot_times [M][P] (absolute), optional task rows [M][...] (None = the
        handle's current value for every problem).  Returns returns [M][N], failure [M][N], order [M][N] (problem-local)."""
        st, tm, mc, knots, kt, w, p, ts = batched_inputs(self.m, state, time, mocap, knots, knot_times, weight, parameters,
                                                         task_state)
        M, N, P, _ = knots.shape
        task = TaskBatch(_pd(w), _pd(p), _pd(ts)) if any(a is not None for a in (w, p, ts)) else None
        ret = np.zeros((M, N), np.float32); fail = np.zeros((M, N), np.uint8); order = np.zeros((M, N), np.int32)
        self._check(self.lib.mjpc_b200_rollout_spline_batched(self.h, M, _pf(st), _pd(tm), _pf(mc),
                                                              C.byref(task) if task is not None else None, _pf(knots),
                                                              _pd(kt), int(interp), P, N, int(H), _pf(ret),
                                                              fail.ctypes.data_as(_bp), order.ctypes.data_as(_ip)))
        self.lastN, self.lastH = M * N, H
        return ret, fail, order

    # ---- multi-GPU: one planning problem sharded over an NCCL communicator owned by the handle
    @staticmethod
    def comm_unique_id():
        buf = (C.c_uint8 * 128)()
        lib = load_library()
        rc = lib.mjpc_b200_comm_unique_id(buf, C.c_size_t(128))
        if rc != 0:
            raise EngineError(f"comm_unique_id failed ({rc}): {lib.mjpc_b200_last_error().decode()}")
        return bytes(buf)

    def comm_init(self, nranks, rank, unique_id: bytes):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self._check(self.lib.mjpc_b200_comm_init(self.h, int(nranks), int(rank), buf, C.c_size_t(128)))
        self.nranks, self.rank = int(nranks), int(rank)

    def comm_init_torch(self, dist):
        """Distribute rank 0's ncclUniqueId over an existing torch.distributed group, then ncclCommInitRank."""
        import torch
        world, rank = dist.get_world_size(), dist.get_rank()
        t = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            t = torch.tensor(list(self.comm_unique_id()), dtype=torch.uint8)
        if dist.get_backend() == "nccl":
            t = t.cuda()
        dist.broadcast(t, 0)
        self.comm_init(world, rank, bytes(t.cpu().numpy().tobytes()))

    def rollout_spline_sharded(self, state, time, mocap, knots, knot_times, interp, H):
        knots = _f(knots)
        N, P, nu = knots.shape
        st, mc, kt = _f(state), _f(mocap), _d(knot_times)
        ret = np.zeros(N, np.float32); fail = np.zeros(N, np.uint8); order = np.zeros(N, np.int32)
        self._check(self.lib.mjpc_b200_rollout_spline_sharded(self.h, _pf(st), C.c_double(time), _pf(mc), None, _pf(knots),
                                                              _pd(kt), int(interp), P, N, int(H), _pf(ret),
                                                              fail.ctypes.data_as(_bp), order.ctypes.data_as(_ip)))
        nr, rk = getattr(self, "nranks", 1), getattr(self, "rank", 0)
        self.lastN, self.lastH = N // nr + (1 if rk < N % nr else 0), H     # fetch_all / fetch_stats are per shard
        return ret, fail, order

    def fetch_trajectory_sharded(self, i):
        H = self.lastH
        o = dict(states=np.zeros((H, self.ds), np.float32), actions=np.zeros((H, self.nu), np.float32),
                 times=np.zeros(H), residual=np.zeros((H, self.nr), np.float32), costs=np.zeros(H, np.float32),
                 trace=np.zeros((H, self.ntr), np.float32))
        self._check(self.lib.mjpc_b200_fetch_trajectory_sharded(self.h, int(i), _pf(o["states"]), _pf(o["actions"]),
                                                                _pd(o["times"]), _pf(o["residual"]), _pf(o["costs"]),
                                                                _pf(o["trace"])))
        return o

    def upload_spline_inputs(self, state, time, mocap, knots, knot_times, interp, H):
        knots = _f(knots)
        N, P, nu = knots.shape
        st, mc, kt = _f(state), _f(mocap), _d(knot_times)
        self._check(self.lib.mjpc_b200_upload_spline_inputs(self.h, _pf(st), C.c_double(time), _pf(mc), None,
                                                            _pf(knots), _pd(kt), int(interp), P, N, int(H)))
        self.lastN, self.lastH = N, H

    def launch_resident(self):
        self._check(self.lib.mjpc_b200_launch_resident(self.h))

    def sync(self):
        self._check(self.lib.mjpc_b200_sync(self.h))

    def read_returns(self):
        N = self.lastN
        ret = np.zeros(N, np.float32); fail = np.zeros(N, np.uint8); order = np.zeros(N, np.int32)
        self._check(self.lib.mjpc_b200_read_returns(self.h, _pf(ret), fail.ctypes.data_as(_bp), order.ctypes.data_as(_ip)))
        return ret, fail, order

    # ---- iLQGPlanner::FeedbackRollouts / ActionRollouts
    def rollout_feedback(self, state, time, mocap, u_nom, x_nom, t_nom, gains, du, step_sizes, mode):
        u, x, t, g = _f(u_nom), _f(x_nom), _d(t_nom), _f(gains)
        dd = _f(du)
        ss = _f(step_sizes)
        K, H = len(ss), u.shape[0]
        st, mc = _f(state), _f(mocap)
        ret = np.zeros(K, np.float32); fail = np.zeros(K, np.uint8); order = np.zeros(K, np.int32)
        self._check(self.lib.mjpc_b200_rollout_feedback(self.h, _pf(st), C.c_double(time), _pf(mc), None, _pf(u), _pf(x),
                                                        _pd(t), _pf(g), _pf(dd), _pf(ss), int(mode), K, H, _pf(ret),
                                                        fail.ctypes.data_as(_bp), order.ctypes.data_as(_ip)))
        self.lastN, self.lastH = K, H
        return ret, fail, order

    def fetch_trajectory(self, i):
        H = self.lastH
        o = dict(states=np.zeros((H, self.ds), np.float32), actions=np.zeros((H, self.nu), np.float32),
                 times=np.zeros(H), residual=np.zeros((H, self.nr), np.float32), costs=np.zeros(H, np.float32),
                 trace=np.zeros((H, self.ntr), np.float32))
        self._check(self.lib.mjpc_b200_fetch_trajectory(self.h, int(i), _pf(o["states"]), _pf(o["actions"]),
                                                        _pd(o["times"]), _pf(o["residual"]), _pf(o["costs"]),
                                                        _pf(o["trace"])))
        return o

    def fetch_all(self):
        N, H = self.lastN, self.lastH
        o = dict(states=np.zeros((N, H, self.ds), np.float32), actions=np.zeros((N, H, self.nu), np.float32),
                 times=np.zeros((N, H)), residual=np.zeros((N, H, self.nr), np.float32),
                 costs=np.zeros((N, H), np.float32), trace=np.zeros((N, H, self.ntr), np.float32))
        self._check(self.lib.mjpc_b200_fetch_all(self.h, _pf(o["states"]), _pf(o["actions"]), _pd(o["times"]),
                                                 _pf(o["residual"]), _pf(o["costs"]), _pf(o["trace"])))
        return o

    def step_debug(self, qpos, qvel, ctrl, mocap, time=0.0, warmstart=None):
        nv, nq = self.info.nv, self.info.nq
        o = dict(qacc=np.zeros(nv, np.float32), residual=np.zeros(max(self.nr, 1), np.float32),
                 next_qpos=np.zeros(nq, np.float32), next_qvel=np.zeros(nv, np.float32),
                 qM=np.zeros((nv, nv), np.float32), efc_force=np.zeros(256, np.float32))
        counts = np.zeros(4, np.int32)
        q, v, u, mc, ws = _f(qpos), _f(qvel), _f(ctrl), _f(mocap), _f(warmstart)
        self._check(self.lib.mjpc_b200_step_debug(self.h, _pf(q), _pf(v), _pf(u), _pf(mc), C.c_double(time), _pf(ws),
                                                  _pf(o["qacc"]), _pf(o["residual"]), _pf(o["next_qpos"]),
                                                  _pf(o["next_qvel"]), _pf(o["qM"]), _pf(o["efc_force"]),
                                                  counts.ctypes.data_as(_ip)))
        o.update(ncon=int(counts[0]), nefc=int(counts[1]), niter=int(counts[2]), warning=int(counts[3]))
        o["efc_force"] = o["efc_force"][: o["nefc"]]
        return o

    def step_batch(self, qpos, qvel, ctrl, mocap, times, time0=0.0, warmstart=None):
        """B independent single steps (mjpc_b200_step_batch): teacher-forced per-step parity at planner sizes."""
        q, v, u, mc, ws, t = _f(qpos), _f(qvel), _f(ctrl), _f(mocap), _f(warmstart), _d(times)
        B, nv, nq = q.shape[0], self.info.nv, self.info.nq
        o = dict(qacc=np.zeros((B, nv), np.float32), next_qpos=np.zeros((B, nq), np.float32),
                 next_qvel=np.zeros((B, nv), np.float32), residual=np.zeros((B, max(self.nr, 1)), np.float32),
                 cost=np.zeros(B, np.float32))
        counts = np.zeros((B, 4), np.int32)
        self._check(self.lib.mjpc_b200_step_batch(self.h, B, _pf(q), _pf(v), _pf(u), _pf(ws), _pf(mc), C.c_double(time0),
                                                  _pd(t), _pf(o["qacc"]), _pf(o["next_qpos"]), _pf(o["next_qvel"]),
                                                  _pf(o["residual"]), _pf(o["cost"]), counts.ctypes.data_as(_ip)))
        o.update(ncon=counts[:, 0], nefc=counts[:, 1], niter=counts[:, 2], warning=counts[:, 3])
        return o

    # ---- iLQG sweeps
    def model_derivatives(self, x, u, t, mocap, tol, skip=0, mode=0):
        x, u, t, mc = _f(x), _f(u), _d(t), _f(mocap)
        H = x.shape[0]
        n, nu, nr = self.n, self.nu, self.nr
        A = np.zeros((H, n, n), np.float32); B = np.zeros((H, n, nu), np.float32)
        Cm = np.zeros((H, nr, n), np.float32); D = np.zeros((H, nr, nu), np.float32)
        self._check(self.lib.mjpc_b200_model_derivatives(self.h, _pf(x), _pf(u), _pd(t), _pf(mc), H, int(skip), C.c_float(tol), int(mode),
                                                         _pf(A), _pf(B), _pf(Cm), _pf(D)))
        return A, B, Cm, D

    def cost_derivatives(self, residual, Cm, D):
        r, c, d = _f(residual), _f(Cm), _f(D)
        H = r.shape[0]
        n, nu = self.n, self.nu
        cx = np.zeros((H, n), np.float32); cu = np.zeros((H, nu), np.float32)
        cxx = np.zeros((H, n, n), np.float32); cuu = np.zeros((H, nu, nu), np.float32)
        cxu = np.zeros((H, n, nu), np.float32)
        self._check(self.lib.mjpc_b200_cost_derivatives(self.h, _pf(r), _pf(c), _pf(d), H, _pf(cx), _pf(cu), _pf(cxx),
                                                        _pf(cuu), _pf(cxu)))
        return cx, cu, cxx, cuu, cxu

    def backward_pass(self, A, B, cx, cu, cxx, cxu, cuu, actions, mu=0.0, reg_type=0, limits=1):
        a = [_f(v) for v in (A, B, cx, cu, cxx, cxu, cuu, actions)]
        H, n, nu = a[1].shape
        K = np.zeros((H, nu, n), np.float32); du = np.zeros((H, nu), np.float32); dV = np.zeros(2, np.float32)
        Vx = np.zeros((H, n), np.float32); Vxx = np.zeros((H, n, n), np.float32)
        status = C.c_int(0)
        self._check(self.lib.mjpc_b200_backward_pass(self.h, *[_pf(v) for v in a], H, C.c_float(mu), int(reg_type),
                                                     int(limits), _pf(K), _pf(du), _pf(dV), _pf(Vx), _pf(Vxx),
                                                     C.byref(status)))
        return dict(K=K, du=du, dV=dV, Vx=Vx, Vxx=Vxx, status=status.value)

    def fetch_stats(self):
        st = np.zeros((self.lastN, 12), np.int64)
        self._check(self.lib.mjpc_b200_fetch_stats(self.h, st.ctypes.data_as(C.POINTER(C.c_int64))))
        return st

    @property
    def launch_count(self):
        return int(self.lib.mjpc_b200_launch_count(self.h))

    def set_xfrc_noise(self, std, rate=1.0, seed=0):
        """NoisyRollout perturbation for the following rollouts (mjpc_b200_set_xfrc_noise); std 0 = off."""
        self._check(self.lib.mjpc_b200_set_xfrc_noise(self.h, C.c_double(std), C.c_double(rate), C.c_uint32(seed)))

    @property
    def last_kernel_ms(self):
        return float(self.lib.mjpc_b200_last_kernel_ms(self.h))

    @property
    def last_kernel_static(self):
        """True if the last rollout launch ran a statically specialised kernel instance (csrc/spec_*.h)."""
        return bool(self.lib.mjpc_b200_last_kernel_static(self.h))

    @property
    def last_kernel_shape(self):
        """0 generic kernel, 1 static helper-warp instance (shipped), 2 its one-warp twin (MJPC_B200_SHAPE=plain);
        include/mjpc_b200.h."""
        return int(self.lib.mjpc_b200_last_kernel_static(self.h))


class CppSamplingPlanner:
    """The C++ host planner (csrc/host/sampling_planner.cc) through its C wrappers."""

    def __init__(self, model, num_trajectory, horizon, seed=0x5EED, device=0):
        self.lib = load_library()
        m = self.m = model
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        num = m.numeric
        self.P = int(num.get("sampling_spline_points", [3])[0])
        self.horizon, self.N, self.nu = int(horizon), int(num_trajectory), m.nu
        cr = _d(np.asarray(m.actuator_ctrlrange, float).reshape(-1))
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_planner_create(C.byref(mb), self.N, self.P, int(num.get("sampling_representation", [2])[0]),
                                               C.c_double(float(num.get("sampling_exploration", [0.1])[0])),
                                               C.c_double(float(m.opt_timestep)), _pd(cr), C.c_uint32(seed), self.horizon,
                                               int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"mjpc_b200_planner_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_planner_destroy(self.h)
            self.h = None

    __del__ = close

    def set_exploration(self, exploration, exploration2=0.0):
        self.lib.mjpc_b200_planner_set_exploration(self.h, C.c_double(exploration), C.c_double(exploration2))

    def reset(self, initial_repeated_action=None):
        a = _d(initial_repeated_action)
        self.lib.mjpc_b200_planner_reset(self.h, self.horizon, _pd(a))

    def set_state(self, state, time, mocap):
        s, mc = _d(state), _d(mocap)
        self.lib.mjpc_b200_planner_set_state(self.h, _pd(s), C.c_double(time), _pd(mc))

    def optimize_policy(self):
        rc = self.lib.mjpc_b200_planner_optimize_policy(self.h, self.horizon)
        if rc != 0:
            raise EngineError(f"planner_optimize_policy failed: {self.lib.mjpc_b200_last_error().decode()}")
        return self.result()

    def result(self):
        winner, imp = C.c_int(), C.c_double()
        ret = np.zeros(self.N, np.float32); knots = np.zeros((self.P, self.nu)); kt = np.zeros(self.P)
        self.lib.mjpc_b200_planner_get_result(self.h, C.byref(winner), C.byref(imp), _pf(ret), _pd(knots), _pd(kt))
        return dict(winner=winner.value, improvement=imp.value, returns=ret, knots=knots, knot_times=kt)

    def action_from_policy(self, time, use_previous=False):
        a = np.zeros(self.nu)
        self.lib.mjpc_b200_planner_action_from_policy(self.h, _pd(a), C.c_double(time), int(use_previous))
        return a


class BatchSamplingPlanner:
    """The C++ batched Predictive Sampling planner (csrc/host/batch_sampling_planner.cc): num_agents independent agents,
    agent p seeded with seeds[p], every iteration ONE batched launch on one engine handle."""

    def __init__(self, model, num_agents, num_trajectory, horizon, seeds=None, device=0):
        self.lib = load_library()
        m = self.m = model
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        num = m.numeric
        self.P = int(num.get("sampling_spline_points", [3])[0])
        self.M, self.horizon, self.N, self.nu = int(num_agents), int(horizon), int(num_trajectory), m.nu
        sd = np.ascontiguousarray([0x5EED] * self.M if seeds is None else seeds, np.uint32)
        if sd.shape != (self.M,):
            raise ValueError(f"seeds must have {self.M} entries")
        cr = _d(np.asarray(m.actuator_ctrlrange, float).reshape(-1))
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_batch_planner_create(
            C.byref(mb), self.M, sd.ctypes.data_as(C.POINTER(C.c_uint32)), self.N, self.P,
            int(num.get("sampling_representation", [2])[0]), C.c_double(float(num.get("sampling_exploration", [0.1])[0])),
            C.c_double(float(m.opt_timestep)), _pd(cr), self.horizon, int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"mjpc_b200_batch_planner_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_batch_planner_destroy(self.h)
            self.h = None

    __del__ = close

    def _agent(self, agent):
        if not 0 <= int(agent) < self.M:
            raise IndexError(f"agent {agent} outside [0, {self.M})")
        return int(agent)

    def reset(self, agent, initial_repeated_action=None):
        a = _d(initial_repeated_action)
        self.lib.mjpc_b200_batch_planner_reset(self.h, self._agent(agent), self.horizon, _pd(a))

    def set_state(self, agent, state, time, mocap):
        s, mc = _d(state), _d(mocap)
        self.lib.mjpc_b200_batch_planner_set_state(self.h, self._agent(agent), _pd(s), C.c_double(time), _pd(mc))

    def set_task(self, agent, weight=None, parameters=None, task_state=None, risk=None):
        w, p, s = _d(weight), _d(parameters), _d(task_state)
        td = TaskDesc(_pd(w), _pd(p), _pd(s), float(self.m.task_risk if risk is None else risk))
        rc = self.lib.mjpc_b200_batch_planner_set_task(self.h, self._agent(agent), C.byref(td))
        if rc != 0:
            raise EngineError(f"batch_planner_set_task failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")

    def optimize_policy(self):
        rc = self.lib.mjpc_b200_batch_planner_optimize_policy(self.h, self.horizon)
        if rc != 0:
            raise EngineError(f"batch_planner_optimize_policy failed: {self.lib.mjpc_b200_last_error().decode()}")
        return [self.result(p) for p in range(self.M)]

    def result(self, agent):
        winner, imp = C.c_int(), C.c_double()
        ret = np.zeros(self.N, np.float32); knots = np.zeros((self.P, self.nu)); kt = np.zeros(self.P)
        self.lib.mjpc_b200_batch_planner_get_result(self.h, self._agent(agent), C.byref(winner), C.byref(imp), _pf(ret),
                                                    _pd(knots), _pd(kt))
        return dict(winner=winner.value, improvement=imp.value, returns=ret, knots=knots, knot_times=kt)

    def action_from_policy(self, agent, time, use_previous=False):
        a = np.zeros(self.nu)
        self.lib.mjpc_b200_batch_planner_action_from_policy(self.h, self._agent(agent), _pd(a), C.c_double(time),
                                                            int(use_previous))
        return a


class CppCrossEntropyPlanner:
    """The C++ Cross-Entropy planner (csrc/host/cross_entropy_planner.cc) through its C wrappers."""

    def __init__(self, model, num_trajectory, horizon, n_elite=0, seed=0x5EED, device=0):
        self.lib = load_library()
        m = self.m = model
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        num = m.numeric
        self.P = int(num.get("sampling_spline_points", [3])[0])
        self.horizon, self.N, self.nu = int(horizon), int(num_trajectory), m.nu
        cr = _d(np.asarray(m.actuator_ctrlrange, float).reshape(-1))
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_ce_planner_create(
            C.byref(mb), self.N, int(n_elite), self.P, int(num.get("sampling_representation", [2])[0]),
            C.c_double(float(num.get("sampling_exploration", [0.1])[0])), C.c_double(float(num.get("std_min", [0.01])[0])),
            C.c_double(float(num.get("explore_fraction", [0.0])[0])), C.c_double(float(m.opt_timestep)), _pd(cr),
            C.c_uint32(seed), self.horizon, int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"mjpc_b200_ce_planner_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_ce_planner_destroy(self.h)
            self.h = None

    __del__ = close

    def reset(self, initial_repeated_action=None):
        a = _d(initial_repeated_action)
        self.lib.mjpc_b200_ce_planner_reset(self.h, self.horizon, _pd(a))

    def set_state(self, state, time, mocap):
        s, mc = _d(state), _d(mocap)
        self.lib.mjpc_b200_ce_planner_set_state(self.h, _pd(s), C.c_double(time), _pd(mc))

    def optimize_policy(self):
        rc = self.lib.mjpc_b200_ce_planner_optimize_policy(self.h, self.horizon)
        if rc != 0:
            raise EngineError(f"ce_planner_optimize_policy failed: {self.lib.mjpc_b200_last_error().decode()}")
        return self.result()

    def result(self):
        imp = C.c_double()
        ret = np.zeros(self.N + 1, np.float32); order = np.zeros(self.N, np.int32)
        knots = np.zeros((self.P, self.nu)); kt = np.zeros(self.P); var = np.zeros((self.P, self.nu))
        self.lib.mjpc_b200_ce_planner_get_result(self.h, C.byref(imp), _pf(ret), order.ctypes.data_as(C.POINTER(C.c_int)),
                                                 _pd(knots), _pd(kt), _pd(var))
        return dict(improvement=imp.value, returns=ret, order=order, knots=knots, knot_times=kt, variance=var)

    def action_from_policy(self, time, use_previous=False):
        a = np.zeros(self.nu)
        self.lib.mjpc_b200_ce_planner_action_from_policy(self.h, _pd(a), C.c_double(time), int(use_previous))
        return a


class CppILQGPlanner:
    """The C++ iLQG planner (csrc/host/ilqg_planner.cc) through its C wrappers."""

    def __init__(self, model, horizon, num_rollouts=10, representation=1, fd_tolerance=3e-4, device=0, fd_mode=1, derivative_skip=0):
        self.lib = load_library()
        m = self.m = model
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        self.H, self.nu, self.ds = int(horizon), m.nu, m.nq + m.nv
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_ilqg_planner_create(C.byref(mb), int(num_rollouts), int(representation),
                                                    C.c_double(fd_tolerance), self.H, int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"mjpc_b200_ilqg_planner_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h = h
        self.lib.mjpc_b200_ilqg_planner_set_fd(self.h, C.c_double(fd_tolerance), int(fd_mode), int(derivative_skip))

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_ilqg_planner_destroy(self.h)
            self.h = None

    __del__ = close

    def reset(self, initial_repeated_action=None):
        a = _d(initial_repeated_action)
        self.lib.mjpc_b200_ilqg_planner_reset(self.h, self.H, _pd(a))

    def set_state(self, state, time, mocap):
        s, mc = _d(state), _d(mocap)
        self.lib.mjpc_b200_ilqg_planner_set_state(self.h, _pd(s), C.c_double(time), _pd(mc))

    def nominal_trajectory(self):
        return self.lib.mjpc_b200_ilqg_planner_nominal_trajectory(self.h, self.H)

    def optimize_policy(self):
        rc = self.lib.mjpc_b200_ilqg_planner_optimize_policy(self.h, self.H)
        if rc < 0:
            raise EngineError(f"ilqg_planner_optimize_policy failed: {self.lib.mjpc_b200_last_error().decode()}")
        return rc

    def result(self):
        sc = np.zeros(6); st = np.zeros((self.H, self.ds), np.float32); ac = np.zeros((self.H, self.nu), np.float32)
        tm = np.zeros(self.H)
        self.lib.mjpc_b200_ilqg_planner_get_result(self.h, _pd(sc), _pf(st), _pf(ac), _pd(tm))
        return dict(total_return=sc[0], regularization=sc[1], improvement=sc[2], expected=sc[3], surprise=sc[4],
                    winner=int(sc[5]), states=st, actions=ac, times=tm)

    def action_from_policy(self, time, state=None):
        a = np.zeros(self.nu)
        s = _d(state)
        self.lib.mjpc_b200_ilqg_planner_action_from_policy(self.h, _pd(a), _pd(s), C.c_double(time))
        return a


class CppRobustPlanner:
    """The C++ Robust planner (csrc/host/robust_planner.cc) through its C wrappers."""

    def __init__(self, model, num_trajectory, horizon, ncandidates=-1, nrepetitions=5, xfrc_std=0.1, xfrc_rate=0.1,
                 seed=0x5EED, device=0):
        self.lib = load_library()
        m = self.m = model
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        num = m.numeric
        self.P = int(num.get("sampling_spline_points", [3])[0])
        self.horizon, self.N, self.nu = int(horizon), int(num_trajectory), m.nu
        self.nc = int(ncandidates if ncandidates != -1 else num_trajectory // nrepetitions)
        cr = _d(np.asarray(m.actuator_ctrlrange, float).reshape(-1))
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_robust_planner_create(
            C.byref(mb), self.N, self.P, int(num.get("sampling_representation", [2])[0]),
            C.c_double(float(num.get("sampling_exploration", [0.1])[0])), C.c_double(float(m.opt_timestep)), _pd(cr),
            C.c_uint32(seed), int(ncandidates), int(nrepetitions), C.c_double(xfrc_std), C.c_double(xfrc_rate),
            self.horizon, int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"mjpc_b200_robust_planner_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_robust_planner_destroy(self.h)
            self.h = None

    __del__ = close

    def reset(self, initial_repeated_action=None):
        a = _d(initial_repeated_action)
        self.lib.mjpc_b200_robust_planner_reset(self.h, self.horizon, _pd(a))

    def set_state(self, state, time, mocap):
        s, mc = _d(state), _d(mocap)
        self.lib.mjpc_b200_robust_planner_set_state(self.h, _pd(s), C.c_double(time), _pd(mc))

    def optimize_policy(self):
        rc = self.lib.mjpc_b200_robust_planner_optimize_policy(self.h, self.horizon)
        if rc != 0:
            raise EngineError(f"robust_planner_optimize_policy failed: {self.lib.mjpc_b200_last_error().decode()}")
        return self.result()

    def result(self):
        winner = C.c_int()
        scores = np.zeros(max(self.nc, 1)); ret = np.zeros(self.N, np.float32)
        knots = np.zeros((self.P, self.nu)); kt = np.zeros(self.P)
        n = self.lib.mjpc_b200_robust_planner_get_result(self.h, C.byref(winner), _pd(scores), _pf(ret), _pd(knots), _pd(kt))
        return dict(winner=winner.value, scores=scores[:n], returns=ret, knots=knots, knot_times=kt)

    def action_from_policy(self, time, use_previous=False):
        a = np.zeros(self.nu)
        self.lib.mjpc_b200_robust_planner_action_from_policy(self.h, _pd(a), C.c_double(time), int(use_previous))
        return a


def host_spline_mapping(representation, input_times, output_times):
    """SplineMapping::Compute (gradient/spline_mapping.cc) as scalar weights W [num_output][num_input]."""
    lib = load_library()
    ti, to = _d(input_times), _d(output_times)
    W = np.zeros((len(to), len(ti)))
    lib.mjpc_b200_host_spline_mapping(int(representation), _pd(ti), len(ti), _pd(to), len(to), _pd(W))
    return W


class CppGradientPlanner:
    """The C++ GradientPlanner (csrc/host/gradient_planner.cc) through its C wrappers."""

    def __init__(self, model, horizon, num_trajectory=8, num_spline_points=5, representation=1, fd_tolerance=3e-4, device=0, fd_mode=1):
        self.lib = load_library()
        self.m = model
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        cr = _d(np.asarray(model.actuator_ctrlrange, float).reshape(-1))
        self.horizon, self.P, self.nu = int(horizon), int(num_spline_points), model.nu
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_gradient_planner_create(C.byref(mb), int(num_trajectory), self.P, int(representation),
                                                        C.c_double(fd_tolerance), C.c_double(float(model.opt_timestep)), _pd(cr),
                                                        self.horizon, int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"gradient_planner_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h = h
        self.lib.mjpc_b200_gradient_planner_set_fd(self.h, C.c_double(fd_tolerance), int(fd_mode), -1)

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_gradient_planner_destroy(self.h)
            self.h = None

    __del__ = close

    def reset(self, initial_repeated_action=None):
        a = _d(initial_repeated_action)
        self.lib.mjpc_b200_gradient_planner_reset(self.h, self.horizon, _pd(a))

    def set_state(self, state, time, mocap):
        s, mc = _d(state), _d(mocap)
        self.lib.mjpc_b200_gradient_planner_set_state(self.h, _pd(s), C.c_double(time), _pd(mc))

    def optimize_policy(self):
        rc = self.lib.mjpc_b200_gradient_planner_optimize_policy(self.h, self.horizon)
        if rc < 0:
            raise EngineError(f"gradient_planner_optimize_policy failed: {self.lib.mjpc_b200_last_error().decode()}")
        return rc

    def result(self):
        sc = np.zeros(6); p = np.zeros((self.P, self.nu)); t = np.zeros(self.P)
        self.lib.mjpc_b200_gradient_planner_get_result(self.h, _pd(sc), _pd(p), _pd(t))
        return dict(total_return=sc[0], winner=int(sc[1]), action_step=sc[2], expected=sc[3], improvement=sc[4],
                    surprise=sc[5], parameters=p, times=t)

    def action_from_policy(self, time, use_previous=False):
        a = np.zeros(self.nu)
        self.lib.mjpc_b200_gradient_planner_action_from_policy(self.h, _pd(a), C.c_double(time), int(use_previous))
        return a


class CppILQSPlanner:
    """The C++ iLQSPlanner (csrc/host/gradient_planner.cc) through its C wrappers."""

    def __init__(self, model, horizon, num_trajectory=8, num_rollouts=6, fd_tolerance=3e-4, seed=0x5EED, device=0, fd_mode=1):
        self.lib = load_library()
        m = self.m = model
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        num = m.numeric
        cr = _d(np.asarray(m.actuator_ctrlrange, float).reshape(-1))
        self.horizon, self.nu = int(horizon), m.nu
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_ilqs_planner_create(C.byref(mb), int(num_trajectory), int(num.get("sampling_spline_points", [3])[0]),
                                                    int(num.get("sampling_representation", [2])[0]),
                                                    C.c_double(float(num.get("sampling_exploration", [0.1])[0])),
                                                    C.c_double(float(m.opt_timestep)), _pd(cr), C.c_uint32(seed), int(num_rollouts),
                                                    int(num.get("ilqg_representation", [1])[0]), C.c_double(fd_tolerance),
                                                    self.horizon, int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"ilqs_planner_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h = h
        self.lib.mjpc_b200_ilqs_planner_set_fd(self.h, C.c_double(fd_tolerance), int(fd_mode), -1)

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_ilqs_planner_destroy(self.h)
            self.h = None

    __del__ = close

    def reset(self, initial_repeated_action=None):
        a = _d(initial_repeated_action)
        self.lib.mjpc_b200_ilqs_planner_reset(self.h, self.horizon, _pd(a))

    def set_state(self, state, time, mocap):
        s, mc = _d(state), _d(mocap)
        self.lib.mjpc_b200_ilqs_planner_set_state(self.h, _pd(s), C.c_double(time), _pd(mc))

    def set_exploration(self, sigma):
        self.lib.mjpc_b200_ilqs_planner_set_exploration(self.h, C.c_double(sigma))

    def optimize_policy(self):
        rc = self.lib.mjpc_b200_ilqs_planner_optimize_policy(self.h, self.horizon)
        if rc < 0:
            raise EngineError(f"ilqs_planner_optimize_policy failed: {self.lib.mjpc_b200_last_error().decode()}")
        return rc

    def result(self):
        sc = np.zeros(4)
        self.lib.mjpc_b200_ilqs_planner_get_result(self.h, _pd(sc))
        return dict(active_policy=int(sc[0]), sampling_return=sc[1], ilqg_return=sc[2], sampling_winner=int(sc[3]))

    def action_from_policy(self, time, state=None, use_previous=False):
        a = np.zeros(self.nu); st = _d(state)
        self.lib.mjpc_b200_ilqs_planner_action_from_policy(self.h, _pd(a), _pd(st), C.c_double(time), int(use_previous))
        return a


class CppAgent:
    """Agent::PlanIteration glue (csrc/host/agent.cc) through its C wrappers; settings mirror the task XML numerics."""
    PLANNERS = {"sampling": 0, "gradient": 1, "ilqg": 2, "ilqs": 3, "robust": 4, "cross_entropy": 5}

    def __init__(self, model, planner="sampling", horizon=None, timestep=None, integrator=0, differentiable=-1, num_trajectory=None,
                 num_spline_points=None, representation=None, exploration=None, ilqg_num_rollouts=10, ilqg_representation=1,
                 fd_tolerance=3e-4, seed=0x5EED, device=0):
        self.lib = load_library()
        m = self.m = model
        num = m.numeric
        self._blob = to_blob(model)
        self._buf = C.create_string_buffer(self._blob, len(self._blob))
        mb = ModelBlob(C.cast(self._buf, C.c_void_p), len(self._blob))
        g = lambda k, d: float(num.get(k, [d])[0])
        st = np.array([self.PLANNERS[planner] if isinstance(planner, str) else planner,
                       g("agent_horizon", 0.5) if horizon is None else horizon,
                       g("agent_timestep", 0.01) if timestep is None else timestep, integrator, differentiable,
                       g("sampling_trajectories", 10) if num_trajectory is None else num_trajectory,
                       g("sampling_spline_points", 3) if num_spline_points is None else num_spline_points,
                       g("sampling_representation", 2) if representation is None else representation,
                       g("sampling_exploration", 0.1) if exploration is None else exploration,
                       ilqg_num_rollouts, ilqg_representation, fd_tolerance, 0, g("std_min", 0.01), g("explore_fraction", 0.0),
                       g("robust_candidates", -1), g("robust_repetitions", 5), g("robust_xfrc", 0.1), g("robust_xfrc_rate", 0.1),
                       seed], float)
        cr = _d(np.asarray(m.actuator_ctrlrange, float).reshape(-1))
        h = C.c_void_p()
        rc = self.lib.mjpc_b200_agent_create(C.byref(mb), _pd(st), _pd(cr), int(device), C.byref(h))
        if rc != 0:
            raise EngineError(f"agent_create failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        self.h, self.nu = h, m.nu

    def close(self):
        if getattr(self, "h", None):
            self.lib.mjpc_b200_agent_destroy(self.h)
            self.h = None

    __del__ = close

    @property
    def steps(self):
        return int(self.lib.mjpc_b200_agent_get_steps(self.h))

    def reset(self, initial_repeated_action=None):
        a = _d(initial_repeated_action)
        self.lib.mjpc_b200_agent_reset(self.h, _pd(a))

    def set_state(self, state, time, mocap):
        s, mc = _d(state), _d(mocap)
        self.lib.mjpc_b200_agent_set_state(self.h, _pd(s), C.c_double(time), _pd(mc))

    def set_task(self, weight=None, parameters=None, task_state=None, risk=None):
        w, p, s = _d(weight), _d(parameters), _d(task_state)
        td = TaskDesc(_pd(w), _pd(p), _pd(s), float(self.m.task_risk if risk is None else risk))
        self.lib.mjpc_b200_agent_set_task(self.h, C.byref(td))

    def set_plan_enabled(self, on):
        self.lib.mjpc_b200_agent_set_plan_enabled(self.h, int(bool(on)))

    def plan_iteration(self):
        rc = self.lib.mjpc_b200_agent_plan_iteration(self.h)
        if rc < 0:
            raise EngineError(f"agent_plan_iteration failed ({rc}): {self.lib.mjpc_b200_last_error().decode()}")
        return rc

    def action_from_policy(self, time, state=None, use_previous=False):
        a = np.zeros(self.nu); st = _d(state)
        self.lib.mjpc_b200_agent_action_from_policy(self.h, _pd(a), _pd(st), C.c_double(time), int(use_previous))
        return a
