"""CPU: batched planning without a device - the Python BatchSamplingPlanner on the fp64 oracle equals M independent
SamplingPlanners, through both of its paths (per-problem loop and rollout_spline_batched), and the argument checks of
Engine.rollout_spline_batched."""
import numpy as np
import pytest

from conftest import OracleBackend, get_model, mocap_of


class TaskOracleBackend(OracleBackend):
    """The oracle backend plus the task snapshot call the batched planner's per-problem loop makes."""

    def set_task(self, weight=None, parameters=None, task_state=None, risk=None):
        self.o.set_task(weight=weight, parameters=parameters, task_state=task_state, risk=risk)


class BatchedOracleBackend(TaskOracleBackend):
    """rollout_spline_batched restated as one oracle call per problem (each with its own task rows)."""

    def rollout_spline_batched(self, state, time, mocap, knots, knot_times, interp, H, weight=None, parameters=None,
                               task_state=None):
        m = self.m
        out = []
        for p in range(len(knots)):
            self.set_task(weight=m.task_weight if weight is None else weight[p],
                          parameters=m.task_parameters if parameters is None else parameters[p],
                          task_state=m.task_state if task_state is None else task_state[p])
            out.append(self.rollout_spline(state[p], time[p], mocap[p], knots[p], knot_times[p], interp, H))
        return tuple(np.stack(x) for x in zip(*out))


def _agents(m, M):
    """Different states, absolute times, seeds and task snapshots per agent."""
    rng = np.random.default_rng(7)
    base = np.concatenate([m.key_qpos[0] if len(m.key_qpos) else m.qpos0, np.zeros(m.nv)])
    out = []
    for p in range(M):
        st = base.copy()
        st[: m.nq] += 0.01 * rng.standard_normal(m.nq) * (p > 0)
        task = {}
        if p % 2 == 1 and len(m.task_parameters):
            task["parameters"] = np.asarray(m.task_parameters, float) * (1 + 0.1 * p)
        if p == 2:
            task["weight"] = np.asarray(m.task_weight, float) * 1.5
        out.append(dict(state=st, time=0.37 * p + 0.01, mocap=mocap_of(m), seed=0x5EED + 11 * p, task=task))
    return out


def _independent(m, agents, N, H, iters):
    from mujoco_mpc_b200.planner import SamplingPlanner
    hist = []
    planners = []
    for a in agents:
        be = TaskOracleBackend(m, threads=2)
        if a["task"]:
            be.set_task(**a["task"])
        pl = SamplingPlanner(m, be, num_trajectory=N, horizon=H, seed=a["seed"])
        pl.reset()
        planners.append(pl)
    for it in range(iters):
        row = []
        for pl, a in zip(planners, agents):
            pl.set_state(a["state"], a["time"] + it * m.opt_timestep, a["mocap"])
            ret, _ = pl.optimize_policy()
            row.append((pl.winner, np.array(ret), pl.values.copy(), pl.times.copy()))
        hist.append(row)
    return hist


def _batched(m, agents, N, H, iters, backend):
    from mujoco_mpc_b200.planner import BatchSamplingPlanner
    bp = BatchSamplingPlanner(m, backend, len(agents), num_trajectory=N, horizon=H, seeds=[a["seed"] for a in agents])
    for p, a in enumerate(agents):
        bp.reset(p)
        if a["task"]:
            bp.set_task(p, **a["task"])
    hist = []
    for it in range(iters):
        for p, a in enumerate(agents):
            bp.set_state(p, a["state"], a["time"] + it * m.opt_timestep, a["mocap"])
        ret, fail = bp.optimize_policy()
        assert ret.shape == (len(agents), N) and fail.shape == (len(agents), N)
        hist.append([(ag.winner, np.array(ret[p]), ag.values.copy(), ag.times.copy()) for p, ag in enumerate(bp.agents)])
    return hist, bp


@pytest.mark.parametrize("name,M,N,H,iters", [("cartpole", 3, 8, 24, 4), ("particle", 3, 8, 11, 4),
                                              ("quadruped", 3, 6, 12, 2)])
@pytest.mark.parametrize("path", ["loop", "batched"])
def test_batch_planner_equals_independent_planners(name, M, N, H, iters, path):
    m = get_model(name)
    agents = _agents(m, M)
    ref = _independent(m, agents, N, H, iters)
    backend = (TaskOracleBackend if path == "loop" else BatchedOracleBackend)(m, threads=2)
    got, bp = _batched(m, agents, N, H, iters, backend)
    for it in range(iters):
        for p in range(M):
            (w0, r0, v0, t0), (w1, r1, v1, t1) = ref[it][p], got[it][p]
            assert w0 == w1, (it, p)
            np.testing.assert_array_equal(r0, r1)
            np.testing.assert_array_equal(v0, v1)
            np.testing.assert_array_equal(t0, t1)
    # the agents really are different problems
    assert len({float(got[-1][p][1][0]) for p in range(M)}) == M
    t = agents[0]["time"]
    np.testing.assert_array_equal(bp.action_from_policy(0, t), bp.agents[0].action_from_policy(t))


def test_batch_planner_rejects_wrong_seed_count():
    from mujoco_mpc_b200.planner import BatchSamplingPlanner
    m = get_model("cartpole")
    with pytest.raises(ValueError):
        BatchSamplingPlanner(m, TaskOracleBackend(m), 3, seeds=[1, 2])


def test_rollout_spline_batched_argument_shapes():
    from mujoco_mpc_b200.engine import batched_inputs
    m = get_model("quadruped")
    M, N, P, ds, nm = 3, 5, 3, m.nq + m.nv, 7 * m.nmocap
    ok = dict(state=np.zeros((M, ds)), time=np.arange(M) * 0.1, mocap=np.zeros((M, nm)), knots=np.zeros((M, N, P, m.nu)),
              knot_times=np.zeros((M, P)))
    st, tm, mc, kn, kt, w, p, ts = batched_inputs(m, **ok)
    assert st.dtype == np.float32 and st.shape == (M, ds) and mc.dtype == np.float32 and kn.dtype == np.float32
    assert tm.dtype == np.float64 and kt.dtype == np.float64 and kt.shape == (M, P)
    assert w is None and p is None and ts is None
    *_, w, p, ts = batched_inputs(m, **ok, weight=np.ones((M, len(m.task_weight))),
                                  parameters=np.ones((M, len(m.task_parameters))), task_state=np.ones((M, len(m.task_state))))
    assert w.shape == (M, len(m.task_weight)) and p.dtype == np.float64 and ts.shape == (M, len(m.task_state))
    bad = [dict(knots=np.zeros((N, P, m.nu))), dict(knots=np.zeros((M, N, P, m.nu + 1))), dict(state=np.zeros((M, ds - 1))),
           dict(state=np.zeros((M + 1, ds))), dict(time=np.zeros(M - 1)), dict(mocap=None), dict(mocap=np.zeros((M, nm + 1))),
           dict(knot_times=np.zeros((M, P + 1))), dict(state=None), dict(weight=np.ones((M, 2))),
           dict(task_state=np.ones(len(m.task_state))), dict(knots=np.zeros((M, 0, P, m.nu)))]
    for b in bad:
        with pytest.raises(ValueError):
            batched_inputs(m, **{**ok, **b})
    # a model without mocap needs none
    c = get_model("cartpole")
    assert batched_inputs(c, np.zeros((2, 4)), [0.0, 1.0], None, np.zeros((2, 4, 10, 1)), np.zeros((2, 10)))[2] is None
