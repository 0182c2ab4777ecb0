"""GPU: batched planning - mjpc_b200_rollout_spline_batched and the planners on top of it.  Problem p of a batched launch
must be bit for bit what mjpc_b200_rollout_spline computes for that problem alone on the same handle: returns, failure,
problem-local order and every trajectory array, under every kernel-shape setting and launch regime."""
import numpy as np
import pytest

from conftest import get_model, mocap_of

pytestmark = pytest.mark.gpu

TRAJ = ("states", "actions", "times", "residual", "costs", "trace")


def _problems(m, M, N, H, seed=0, task_state=None):
    """M different problems: perturbed states, absolute times, mocap, knots (and optional task-state rows)."""
    from mujoco_mpc_b200.planner import candidate_knots
    rng = np.random.default_rng(100 + seed)
    q0 = m.key_qpos[0] if len(m.key_qpos) else m.qpos0
    P = 3
    cr = np.asarray(m.actuator_ctrlrange, float).reshape(-1, 2)
    st, tm, mc, kn, kt = [], [], [], [], []
    for p in range(M):
        s = np.concatenate([q0, np.zeros(m.nv)])
        if p:
            s[7 if m.nq > 7 else 0: m.nq] += 0.01 * rng.standard_normal(m.nq - (7 if m.nq > 7 else 0))
            s[m.nq:] = 0.05 * rng.standard_normal(m.nv)
        t = 0.25 * p + 0.125 * seed
        mo = mocap_of(m).copy()
        if p and m.nmocap:
            for k in range(m.nmocap):
                mo[7 * k: 7 * k + 3] += 0.02 * rng.standard_normal(3)
        st.append(s); tm.append(t); mc.append(mo)
        kn.append(candidate_knots(np.zeros((P, m.nu)) + 0.05 * p, 0.1, cr, iteration=p, N=N, seed=0x5EED + seed))
        kt.append(t + np.arange(P) * (H - 1) * m.opt_timestep / (P - 1))
    return dict(state=np.array(st), time=np.array(tm), mocap=np.array(mc), knots=np.array(kn), knot_times=np.array(kt),
                task_state=task_state)


def _singles(e, m, pr, interp, H, task=None):
    """Each problem alone: set_task (when it has task rows), rollout_spline, fetch_all."""
    out = []
    M = len(pr["knots"])
    for p in range(M):
        rows = {k: v[p] for k, v in (task or {}).items() if v is not None}
        if pr.get("task_state") is not None:
            rows["task_state"] = pr["task_state"][p]
        if rows:
            e.set_task(**rows)
        r, f, o = e.rollout_spline(pr["state"][p], pr["time"][p], pr["mocap"][p], pr["knots"][p], pr["knot_times"][p],
                                   interp, H)
        out.append((r, f, o, e.fetch_all()))
        if rows:    # back to the model's task for the next problem and the batched call
            e.set_task(weight=m.task_weight, parameters=m.task_parameters, task_state=m.task_state)
    return out


def _assert_batched_equals_singles(e, m, pr, interp=2, H=32, task=None):
    single = _singles(e, m, pr, interp, H, task)
    kw = dict(task or {})
    if pr.get("task_state") is not None:
        kw["task_state"] = pr["task_state"]
    ret, fail, order = e.rollout_spline_batched(pr["state"], pr["time"], pr["mocap"], pr["knots"], pr["knot_times"],
                                                interp, H, **kw)
    allb = e.fetch_all()
    M, N = ret.shape
    ok = 0
    for p, (r, f, o, tr) in enumerate(single):
        np.testing.assert_array_equal(ret[p], r, err_msg=f"returns of problem {p}")
        np.testing.assert_array_equal(fail[p], f, err_msg=f"failure of problem {p}")
        np.testing.assert_array_equal(order[p], o, err_msg=f"order of problem {p}")
        for i in range(N):
            if f[i]:       # a failed rollout stops early: the rest of its rows are not outputs
                continue
            ok += 1
            for k in TRAJ:
                np.testing.assert_array_equal(allb[k][p * N + i], tr[k][i], err_msg=f"{k} of problem {p}, candidate {i}")
    assert ok >= M * N // 2, "most candidates must complete for the comparison to mean something"
    # the problems differ: a batched launch is not M copies of one problem
    assert len({float(ret[p, 0]) for p in range(M)}) == M
    return ret


def _engine(m, cap, H, monkeypatch=None, wpc=None):
    from mujoco_mpc_b200.engine import Engine
    if wpc is not None:
        monkeypatch.setenv("MJPC_B200_WARPS_PER_CTA", str(wpc))     # read by create()
    e = Engine(m, cap, H)
    if wpc is not None:
        monkeypatch.delenv("MJPC_B200_WARPS_PER_CTA")
    return e


def test_quadruped_static_batched_equals_singles():
    m = get_model("quadruped")
    e = _engine(m, 64, 32)
    from mujoco_mpc_b200 import task as T
    pr = _problems(m, 4, 16, 32)
    ts = np.tile(np.asarray(m.task_state, float), (4, 1))
    ts[:, T.QS_PHASE_START] = [0.0, 0.5, 1.0, 1.5]
    ts[:, T.QS_PHASE_START_TIME] = pr["time"] - np.array([0.0, 0.1, 0.2, 0.3])     # absolute: rebased per problem
    pr["task_state"] = ts
    _assert_batched_equals_singles(e, m, pr)
    assert e.last_kernel_shape == 1
    e.close()


def test_humanoid_track_static_batched_equals_singles():
    """Different clip (mode) and reference time per problem: the task state is rebased per problem."""
    m = get_model("humanoid_track")
    e = _engine(m, 64, 32)
    pr = _problems(m, 4, 12, 32)
    ts = np.tile(np.asarray(m.task_state, float), (4, 1))
    ts[:, 0] = [0, 1, 0, 1]
    ts[:, 1] = pr["time"] - np.array([0.0, 0.05, 0.1, 0.15])
    pr["task_state"] = ts
    _assert_batched_equals_singles(e, m, pr)
    assert e.last_kernel_shape == 1
    e.close()


@pytest.mark.parametrize("name", ["cartpole", "shadow_reorient"])
def test_generic_kernel_batched_equals_singles(name):
    m = get_model(name)
    e = _engine(m, 64, 32)
    _assert_batched_equals_singles(e, m, _problems(m, 4, 10, 32))
    assert e.last_kernel_shape == 0
    e.close()


@pytest.mark.parametrize("setting", ["plain", "no_static", "wpc2"])
def test_every_shape_setting(setting, monkeypatch):
    m = get_model("quadruped")
    e = _engine(m, 64, 32, monkeypatch, wpc=2 if setting == "wpc2" else None)
    if setting == "plain":
        monkeypatch.setenv("MJPC_B200_SHAPE", "plain")
    if setting == "no_static":
        monkeypatch.setenv("MJPC_B200_NO_STATIC", "1")
    N = 15 if setting == "wpc2" else 16      # odd N: with two candidates per CTA a CTA would otherwise span two problems
    _assert_batched_equals_singles(e, m, _problems(m, 4, N, 32, seed=1))
    assert e.last_kernel_shape == {"plain": 2, "no_static": 0, "wpc2": 0}[setting]
    e.close()


@pytest.mark.parametrize("M,N", [(8, 32), (3, 150)])
def test_launch_regimes(M, N):
    """8 x 32 = 256 candidates: co-resident pairs (pair synchronisation on); 3 x 150 = 450: two waves."""
    m = get_model("quadruped")
    e = _engine(m, M * N, 32)
    _assert_batched_equals_singles(e, m, _problems(m, M, N, 32, seed=2))
    e.close()


def test_per_problem_task_snapshot():
    """Different weights, gait parameters and task state per problem == set_task + a single call, bitwise."""
    m = get_model("quadruped")
    e = _engine(m, 64, 32)
    M = 4
    w = np.tile(np.asarray(m.task_weight, float), (M, 1)) * np.array([1.0, 1.5, 0.5, 2.0])[:, None]
    prm = np.tile(np.asarray(m.task_parameters, float), (M, 1))
    prm[:, 0] = [0, 1, 2, 3]      # gait
    from mujoco_mpc_b200 import task as T
    pr = _problems(m, M, 16, 32, seed=3)
    ts = np.tile(np.asarray(m.task_state, float), (M, 1))
    ts[:, T.QS_PHASE_START_TIME] = pr["time"] - 0.2
    ts[:, T.QS_PHASE_START] = [0.0, 1.0, 2.0, 3.0]
    pr["task_state"] = ts
    _assert_batched_equals_singles(e, m, pr, task=dict(weight=w, parameters=prm))
    e.close()


def test_single_problem_and_xfrc_noise():
    m = get_model("quadruped")
    e = _engine(m, 64, 32)
    pr = _problems(m, 1, 16, 32, seed=4)
    single = _singles(e, m, pr, 2, 32)[0]
    ret, fail, order = e.rollout_spline_batched(pr["state"], pr["time"], pr["mocap"], pr["knots"], pr["knot_times"], 2, 32)
    np.testing.assert_array_equal(ret[0], single[0]); np.testing.assert_array_equal(order[0], single[2])
    allb = e.fetch_all()
    for k in TRAJ:
        np.testing.assert_array_equal(allb[k], single[3][k])
    e.set_xfrc_noise(2.0, 0.05, seed=9)          # the noise stream is the problem-local candidate index
    r_noisy = _assert_batched_equals_singles(e, m, _problems(m, 3, 16, 32, seed=5))
    e.set_xfrc_noise(0.0, 0.05, 0)
    r_clean = e.rollout_spline_batched(**{k: v for k, v in _problems(m, 3, 16, 32, seed=5).items() if k != "task_state"},
                                       interp=2, H=32)[0]
    assert not np.array_equal(r_noisy, r_clean)
    e.close()


def test_errors_leave_the_handle_usable():
    from mujoco_mpc_b200.engine import EngineError
    m = get_model("quadruped")
    e = _engine(m, 32, 32)
    pr = _problems(m, 3, 11, 32, seed=6)          # 33 > 32 candidates
    with pytest.raises(EngineError, match="error -3"):
        e.rollout_spline_batched(pr["state"], pr["time"], pr["mocap"], pr["knots"], pr["knot_times"], 2, 32)
    pr = _problems(m, 2, 8, 32, seed=6)
    with pytest.raises(EngineError, match="error -1"):
        e.rollout_spline_batched(pr["state"], pr["time"], pr["mocap"], pr["knots"], pr["knot_times"], 2, 0)
    with pytest.raises(EngineError, match="error -1"):
        e.rollout_spline_batched(pr["state"], pr["time"], pr["mocap"], pr["knots"], pr["knot_times"], 7, 32)
    with pytest.raises(EngineError, match="error -3"):
        e.rollout_spline_batched(pr["state"], pr["time"], pr["mocap"], pr["knots"], pr["knot_times"], 2, 33)
    _assert_batched_equals_singles(e, m, pr)
    e.close()


def _agent_inputs(m, M):
    rng = np.random.default_rng(11)
    out = []
    for p in range(M):
        s = np.concatenate([m.key_qpos[0], np.zeros(m.nv)])
        s[7: m.nq] += 0.01 * p * rng.standard_normal(m.nq - 7)
        out.append((s, 0.3 * p, mocap_of(m)))
    return out


def test_cpp_batch_planner_equals_single_planners_and_mirror():
    from mujoco_mpc_b200.engine import BatchSamplingPlanner as CppBatch, CppSamplingPlanner, Engine
    from mujoco_mpc_b200.planner import BatchSamplingPlanner
    m = get_model("quadruped")
    M, N, H = 3, 16, 32
    seeds = [0x5EED + 7 * p for p in range(M)]
    inp = _agent_inputs(m, M)
    cpp = CppBatch(m, M, N, H, seeds=seeds)
    singles = [CppSamplingPlanner(m, N, H, seed=s) for s in seeds]
    e = Engine(m, M * N, H)
    py = BatchSamplingPlanner(m, e, M, num_trajectory=N, horizon=H, seeds=seeds)
    for p in range(M):
        cpp.reset(p, np.zeros(m.nu)); singles[p].reset(np.zeros(m.nu)); py.reset(p, np.zeros(m.nu))
    for it in range(5):
        for p, (s, t, mo) in enumerate(inp):
            tt = t + it * m.opt_timestep
            cpp.set_state(p, s, tt, mo); singles[p].set_state(s, tt, mo); py.set_state(p, s, tt, mo)
        res = cpp.optimize_policy()
        ret_py, _ = py.optimize_policy()
        for p in range(M):
            r1 = singles[p].optimize_policy()
            assert res[p]["winner"] == r1["winner"], (it, p)
            for k in ("returns", "knots", "knot_times"):
                np.testing.assert_array_equal(res[p][k], r1[k], err_msg=f"{k}, iteration {it}, agent {p}")
            assert res[p]["improvement"] == r1["improvement"]
            tq = inp[p][1] + it * m.opt_timestep + 0.013
            np.testing.assert_array_equal(cpp.action_from_policy(p, tq), singles[p].action_from_policy(tq))
            # the Python mirror drives the same ABI with the same noise (host arithmetic may differ in the last bits)
            ag = py.agents[p]
            assert res[p]["winner"] == ag.winner, (it, p)
            np.testing.assert_allclose(res[p]["knot_times"], ag.times, atol=1e-12)
            np.testing.assert_allclose(res[p]["knots"], ag.values, atol=1e-6)
            np.testing.assert_allclose(res[p]["returns"], ret_py[p], rtol=1e-5)
    cpp.close(); e.close()
    for s in singles:
        s.close()


def test_closed_loop_batched_equals_single_agent_loops(oracle_lib):
    """M quadrupeds from perturbed home states on the fp64 oracle plant, one batched planning iteration per plant step:
    every agent's cost sequence equals its own single-agent loop exactly (test_closed_loop.py's pattern)."""
    from mujoco_mpc_b200.blob import to_blob
    from mujoco_mpc_b200.engine import Engine
    from mujoco_mpc_b200.planner import BatchSamplingPlanner, SamplingPlanner
    m = get_model("quadruped")
    plant = oracle_lib.Oracle(to_blob(m), m, 64)
    M, N, H, steps = 4, 32, 32, 30
    rng = np.random.default_rng(5)
    starts = []
    for p in range(M):
        q = m.key_qpos[0].copy()
        q[7:] += 0.02 * p * rng.standard_normal(m.nq - 7)
        starts.append(q)
    mocap = mocap_of(m)

    def plant_step(q, v, u, t, warm):
        r = plant.forward_debug(q, v, u, mocap, time=t, warmstart=warm)
        return r["next_qpos"], r["next_qvel"], r["qacc"], plant.cost_value(r["residual"][: m.task_num_residual])

    e = Engine(m, M * N, H)
    single_costs = []
    for p in range(M):
        pl = SamplingPlanner(m, e, num_trajectory=N, horizon=H, seed=0x5EED + p)
        pl.reset(np.zeros(m.nu))
        q, v, t, warm, cs = starts[p].copy(), np.zeros(m.nv), 0.0, None, []
        for k in range(steps):
            pl.set_state(np.concatenate([q, v]), t, mocap)
            pl.optimize_policy()
            q, v, warm, c = plant_step(q, v, pl.action_from_policy(t), t, warm)
            cs.append(c); t += m.opt_timestep
        single_costs.append(np.array(cs))
    bp = BatchSamplingPlanner(m, e, M, num_trajectory=N, horizon=H, seeds=[0x5EED + p for p in range(M)])
    xs = [[starts[p].copy(), np.zeros(m.nv), None] for p in range(M)]
    costs, t = [[] for _ in range(M)], 0.0
    for p in range(M):
        bp.reset(p, np.zeros(m.nu))
    for k in range(steps):
        for p in range(M):
            bp.set_state(p, np.concatenate(xs[p][:2]), t, mocap)
        bp.optimize_policy()
        for p in range(M):
            q, v, warm, c = plant_step(xs[p][0], xs[p][1], bp.action_from_policy(p, t), t, xs[p][2])
            xs[p] = [q, v, warm]; costs[p].append(c)
        t += m.opt_timestep
    e.close()
    for p in range(M):
        np.testing.assert_array_equal(np.array(costs[p]), single_costs[p], err_msg=f"agent {p}")
    assert np.isfinite(np.array(costs)).all()
