"""Host-side Predictive Sampling logic around the rollout engine (Python mirror used by tests and bench).

Mirrors mjpc/planners/sampling/planner.cc:
  * UpdateNominalPolicy (non-sliding resample)  :240-323  -> resample_nominal
  * AddNoiseToPolicy                            :326-352  -> candidate_knots (noise injected from Philox4x32-10,
    seed 0x5EED, counter = (iteration, candidate, knot, dof): the reference's absl::BitGen is unseedable,
    SURVEY.md section 0 finding 4)
  * OptimizePolicy / CopyCandidateToPolicy      :197-212, 534-543 -> SamplingPlanner.optimize_policy
The spline itself (mjpc/spline/spline.cc:103-156, 250-287) is restated in sample_spline for the host-side
resampling; the device evaluates the same formula per step.
"""
from __future__ import annotations

import numpy as np

PHILOX_M0, PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
PHILOX_W0, PHILOX_W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)


def philox4x32(counter, key, rounds=10):
    """Vectorised Philox4x32-10. counter: (..., 4) uint32, key: (2,) uint32 -> (..., 4) uint32."""
    c = np.array(counter, dtype=np.uint32, copy=True)
    k0, k1 = np.uint32(key[0]), np.uint32(key[1])
    for _ in range(rounds):
        p0 = PHILOX_M0 * c[..., 0].astype(np.uint64)
        p1 = PHILOX_M1 * c[..., 2].astype(np.uint64)
        hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), p0.astype(np.uint32)
        hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), p1.astype(np.uint32)
        c = np.stack([hi1 ^ c[..., 1] ^ k0, lo1, hi0 ^ c[..., 3] ^ k1, lo0], axis=-1)
        k0 = np.uint32((int(k0) + int(PHILOX_W0)) & 0xFFFFFFFF)
        k1 = np.uint32((int(k1) + int(PHILOX_W1)) & 0xFFFFFFFF)
    return c


def philox_normal(iteration, N, P, nu, seed=0x5EED):
    """Standard normals z[N][P][nu] from counter (iteration, candidate, knot, dof)."""
    cand, knot, dof = np.meshgrid(np.arange(N), np.arange(P), np.arange(nu), indexing="ij")
    ctr = np.stack([np.full_like(cand, iteration), cand, knot, dof], axis=-1).astype(np.uint32)
    r = philox4x32(ctr, (seed, 0))
    u1 = (r[..., 0].astype(np.float64) + 0.5) / 4294967296.0
    u2 = (r[..., 1].astype(np.float64) + 0.5) / 4294967296.0
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


def sample_spline(times, values, interp, t):
    """TimeSpline::Sample (spline.cc:103-156); times [P], values [P][dim]."""
    times = np.asarray(times, float); values = np.asarray(values, float)
    P = len(times)
    if P == 0:
        return np.zeros(values.shape[1])
    upper = int(np.searchsorted(times, t, side="right"))
    if upper == P:
        return values[P - 1].copy()
    if upper == 0:
        return values[0].copy()
    lower = upper - 1
    dt = times[upper] - times[lower]
    s = (t - times[lower]) / dt
    if interp == 0:
        return values[lower].copy()
    if interp == 1:
        return values[lower] * (1 - s) + values[upper] * s

    def slope(node):
        if node == 0:
            return (values[1] - values[0]) / (times[1] - times[0])
        if node == P - 1:
            return (values[node] - values[node - 1]) / (times[node] - times[node - 1])
        return 0.5 * (values[node + 1] - values[node]) / (times[node + 1] - times[node]) + \
            0.5 * (values[node] - values[node - 1]) / (times[node] - times[node - 1])
    c0 = 2 * s ** 3 - 3 * s ** 2 + 1; c1 = (s ** 3 - 2 * s ** 2 + s) * dt
    c2 = -2 * s ** 3 + 3 * s ** 2; c3 = (s ** 3 - s ** 2) * dt
    return c0 * values[lower] + c1 * slope(lower) + c2 * values[upper] + c3 * slope(upper)


def clamp(x, ctrlrange):
    return np.clip(x, ctrlrange[:, 0], ctrlrange[:, 1])


def resample_nominal(times, values, interp, time, horizon, timestep, P, ctrlrange):
    """Non-sliding UpdateNominalPolicy: P knots starting at `time` spanning (horizon-1)*timestep."""
    T = (horizon - 1) * timestep
    shift = max(T / P, 1e-5) if interp == 0 else max(T / (P - 1), 1e-5)
    new_t = time + shift * np.arange(P)
    new_v = np.stack([clamp(sample_spline(times, values, interp, tt), ctrlrange) for tt in new_t])
    return new_t, new_v


def candidate_knots(nominal, sigma, ctrlrange, iteration, N, seed=0x5EED, sigma2=0.0):
    """Candidate 0 = nominal; candidate i>0 = clamp(nominal + std_i * 0.5*(hi-lo) * z), std_i = sigma, or - when
    sigma2 > 0 - sigma2 with probability 0.2 (planner.cc:334-338; the Bernoulli draw is word 2 of the Philox block with
    counter (iteration, candidate, 0xffffffff, 0), as in csrc/host/sampling_planner.cc AddNoiseToPolicy)."""
    P, nu = nominal.shape
    z = philox_normal(iteration, N, P, nu, seed)
    scale = 0.5 * (ctrlrange[:, 1] - ctrlrange[:, 0])
    if sigma2 > 0:
        ctr = np.stack([np.full(N, iteration), np.arange(N), np.full(N, 0xFFFFFFFF), np.zeros(N, np.int64)], -1).astype(np.uint32)
        u = (philox4x32(ctr, (seed, 0))[:, 2].astype(np.float64) + 0.5) / 4294967296.0
        sigma = np.where(u < 0.2, sigma2, sigma)[:, None, None]
    k = nominal[None] + sigma * scale[None, None, :] * z
    k[0] = nominal
    return np.clip(k, ctrlrange[:, 0], ctrlrange[:, 1])


class SamplingPlanner:
    """Predictive Sampling around a rollout backend exposing rollout_spline(state,time,mocap,knots,kt,interp,H)."""

    def __init__(self, model, backend, num_trajectory=None, horizon=None, seed=0x5EED):
        m = self.model = model
        self.backend = backend
        num = m.numeric
        self.num_trajectory = int(num_trajectory or num.get("sampling_trajectories", [10])[0])
        self.P = int(num.get("sampling_spline_points", [3])[0])
        self.sigma = float(num.get("sampling_exploration", [0.1])[0])
        self.sigma2 = 0.0                       # noise_exploration[1] (planner.cc:86): second std, used with p = 0.2
        self.interp = int(num.get("sampling_representation", [2])[0])
        self.timestep = float(m.opt_timestep)
        # steps_ = clamp(horizon/timestep + 1, 1, 512), float truncation (agent.cc:107)
        self.horizon = int(horizon or max(min(num.get("agent_horizon", [0.5])[0] / self.timestep + 1, 512), 1))
        self.ctrlrange = np.asarray(m.actuator_ctrlrange, float).reshape(-1, 2)
        self.seed = seed
        self.iteration = 0
        self.times = np.zeros(1)
        self.values = np.zeros((1, m.nu))
        self.winner = 0
        self.improvement = 0.0

    def reset(self, initial_repeated_action=None):
        self.times = np.zeros(1)
        self.values = np.zeros((1, self.model.nu)) if initial_repeated_action is None else \
            np.asarray(initial_repeated_action, float)[None]
        self.iteration = 0

    def set_state(self, state, time, mocap):
        self.state, self.time, self.mocap = np.asarray(state, float), float(time), np.asarray(mocap, float)

    def make_candidates(self):
        self.times, self.values = resample_nominal(self.times, self.values, self.interp, self.time, self.horizon,
                                                   self.timestep, self.P, self.ctrlrange)
        return candidate_knots(self.values, self.sigma, self.ctrlrange, self.iteration, self.num_trajectory, self.seed,
                               sigma2=self.sigma2)

    def optimize_policy(self):
        knots = self.make_candidates()
        ret, fail, order = self.backend.rollout_spline(self.state, self.time, self.mocap, knots, self.times,
                                                       self.interp, self.horizon)
        self.install_winner(knots, ret, order)
        return ret, fail

    def install_winner(self, knots, ret, order):
        """The rest of OptimizePolicy once the candidates are rolled out: the best one becomes the policy."""
        self.winner = int(order[0]) if order is not None else int(np.argmin(ret))
        self.improvement = max(float(ret[0]) - float(ret[self.winner]), 0.0)
        self.values = knots[self.winner].astype(float)
        self.returns = ret
        self.iteration += 1

    def action_from_policy(self, time):
        return clamp(sample_spline(self.times, self.values, self.interp, time), self.ctrlrange)


_TASK_ATTR = dict(weight="task_weight", parameters="task_parameters", task_state="task_state")   # model attributes


class BatchSamplingPlanner:
    """M independent Predictive Sampling agents of one model, planned together (csrc/host/batch_sampling_planner.cc).

    Each agent is a SamplingPlanner (own policy, seed, iteration, state, time, mocap) with its own task snapshot.  Per
    optimize_policy every agent makes its candidates, then ONE backend.rollout_spline_batched call rolls all of them out
    when the backend has it; otherwise (the CPU oracle) backend.rollout_spline runs per agent, after backend.set_task with
    that agent's snapshot when any agent has one.  Snapshot members an agent never set are the model's values."""

    def __init__(self, model, backend, num_agents, num_trajectory=None, horizon=None, seeds=None):
        self.model, self.backend, self.M = model, backend, int(num_agents)
        seeds = [0x5EED] * self.M if seeds is None else list(seeds)
        if len(seeds) != self.M:
            raise ValueError(f"seeds must have {self.M} entries")
        self.agents = [SamplingPlanner(model, backend, num_trajectory, horizon, sd) for sd in seeds]
        self.tasks = [dict() for _ in range(self.M)]

    def reset(self, agent, initial_repeated_action=None):
        self.agents[agent].reset(initial_repeated_action)

    def set_state(self, agent, state, time, mocap):
        self.agents[agent].set_state(state, time, mocap)

    def set_task(self, agent, weight=None, parameters=None, task_state=None):
        for k, v in (("weight", weight), ("parameters", parameters), ("task_state", task_state)):
            if v is not None:
                self.tasks[agent][k] = np.array(v, float)

    def _task_rows(self, key):
        """[M][...] rows of one snapshot member, or None when no agent set it."""
        if not any(key in t for t in self.tasks):
            return None
        default = np.asarray(getattr(self.model, _TASK_ATTR[key]), float)
        return np.stack([t.get(key, default) for t in self.tasks])

    def optimize_policy(self):
        a0 = self.agents[0]
        knots = np.stack([a.make_candidates() for a in self.agents])
        rows = {k: self._task_rows(k) for k in ("weight", "parameters", "task_state")}
        if hasattr(self.backend, "rollout_spline_batched"):
            ret, fail, order = self.backend.rollout_spline_batched(
                np.stack([a.state for a in self.agents]), np.array([a.time for a in self.agents]),
                np.stack([a.mocap for a in self.agents]), knots, np.stack([a.times for a in self.agents]), a0.interp,
                a0.horizon, **rows)
        else:
            ret, fail, order = [], [], []
            for p, a in enumerate(self.agents):
                if any(r is not None for r in rows.values()):
                    self.backend.set_task(**{k: (getattr(self.model, _TASK_ATTR[k]) if r is None else r[p])
                                             for k, r in rows.items()})
                r, f, o = self.backend.rollout_spline(a.state, a.time, a.mocap, knots[p], a.times, a.interp, a.horizon)
                ret.append(r); fail.append(f); order.append(o)
        for p, a in enumerate(self.agents):
            a.install_winner(knots[p], ret[p], order[p])
        return np.asarray(ret), np.asarray(fail)

    def action_from_policy(self, agent, time):
        return self.agents[agent].action_from_policy(time)


class CrossEntropyPlanner:
    """Cross-Entropy Method planner (mjpc/planners/cross_entropy/planner.cc) on the same rollout backend.

    Per OptimizePolicy (planner.cc:153-292): resample the nominal to the current time (ResamplePolicy, :343-371),
    roll out N noisy candidates + the un-noised nominal (Rollouts, :414-459: ONE launch of N+1 candidates here, the
    nominal is candidate N), rank, then  policy = mean of the n_elite best knot sets, variance = their sample
    variance (/(n_elite-1)).  Noise (AddNoiseToPolicy, :374-411) is N(0, max(sqrt(variance[k]), std)) per
    parameter - not scaled by the control range - with std = sampling_exploration for the first
    explore_fraction*N candidates and std_min for the rest; drawn from the injected Philox stream.
    BestTrajectory() is the NOMINAL trajectory (:462-464).
    """

    def __init__(self, model, backend, num_trajectory=None, horizon=None, n_elite=None, seed=0x5EED):
        m = self.model = model
        self.backend = backend
        num = m.numeric
        self.num_trajectory = int(num_trajectory or num.get("sampling_trajectories", [10])[0])
        self.P = int(num.get("sampling_spline_points", [3])[0])
        self.std_initial = float(num.get("sampling_exploration", [0.1])[0])
        self.std_min = float(num.get("std_min", [0.01])[0])
        self.explore_fraction = float(num.get("explore_fraction", [0.0])[0])
        self.n_elite = int(n_elite or num.get("n_elite", [max(self.num_trajectory // 10, 2)])[0])
        self.interp = int(num.get("sampling_representation", [2])[0])
        self.timestep = float(m.opt_timestep)
        self.horizon = int(horizon or max(min(num.get("agent_horizon", [0.5])[0] / self.timestep + 1, 512), 1))
        self.ctrlrange = np.asarray(m.actuator_ctrlrange, float).reshape(-1, 2)
        self.seed = seed
        self.reset()

    def reset(self, initial_repeated_action=None):
        self.times = np.zeros(1)
        self.values = np.zeros((1, self.model.nu)) if initial_repeated_action is None else \
            np.asarray(initial_repeated_action, float)[None]
        self.variance = np.full((self.P, self.model.nu), self.std_initial ** 2)
        self.iteration = 0
        self.improvement = 0.0

    def set_state(self, state, time, mocap):
        self.state, self.time, self.mocap = np.asarray(state, float), float(time), np.asarray(mocap, float)

    def resample(self):
        """ResamplePolicy (:343-371): always (horizon-1)*dt/(P-1), also for zero-order splines."""
        shift = max((self.horizon - 1) * self.timestep / (self.P - 1), 1e-5)
        new_t = self.time + shift * np.arange(self.P)
        new_v = np.stack([clamp(sample_spline(self.times, self.values, self.interp, tt), self.ctrlrange) for tt in new_t])
        return new_t, new_v

    def make_candidates(self, times, nominal):
        N, P, nu = self.num_trajectory, self.P, self.model.nu
        z = philox_normal(self.iteration, N, P, nu, self.seed)
        std = np.where(np.arange(N) < N * self.explore_fraction, self.std_initial, self.std_min)
        sd = np.maximum(np.sqrt(self.variance)[None], std[:, None, None])
        k = np.clip(nominal[None] + sd * z, self.ctrlrange[:, 0], self.ctrlrange[:, 1])
        return np.concatenate([k, nominal[None]], 0)       # candidate N = the nominal trajectory

    def optimize_policy(self):
        N = self.num_trajectory
        n_elite = self.n_elite = min(self.n_elite, N)
        times, nominal = self.resample()
        knots = self.make_candidates(times, nominal)
        ret, fail, _ = self.backend.rollout_spline(self.state, self.time, self.mocap, knots, times, self.interp, self.horizon)
        ret = np.asarray(ret, float)
        order = np.argsort(ret[:N], kind="stable")
        elite = knots[order[:n_elite]].astype(float)
        mean = elite.mean(0)
        self.variance = ((elite - mean[None]) ** 2).sum(0) / (n_elite - 1)
        self.times, self.values = times, mean
        avg_return = float(ret[order[:n_elite]].mean())
        self.improvement = max(avg_return - float(ret[order[0]]), 0.0)
        self.nominal_index = N
        self.order = order
        self.returns = ret
        self.iteration += 1
        return ret, fail

    def action_from_policy(self, time):
        return clamp(sample_spline(self.times, self.values, self.interp, time), self.ctrlrange)


class RobustPlanner:
    """Robust planner (mjpc/planners/robust/robust_planner.cc:91-157) over a SamplingPlanner delegate.

    OptimizePolicy: the delegate's candidate rollouts -> the best `ncandidates`; each is rolled out `nrepetitions`
    times with NoisyRollout force perturbations (ONE launch of ncandidates*nrepetitions candidates, noise stream =
    launch index, seed + iteration); a candidate's score is the mean of its non-failed noisy returns (its clean
    score only if all failed); the best score is installed.  Defaults: robust_repetitions 5, robust_candidates =
    sampling_trajectories / repetitions, robust_xfrc 0.1, robust_xfrc_rate 0.1 (robust_planner.cc:44-57)."""

    def __init__(self, model, backend, num_trajectory=None, horizon=None, ncandidates=None, nrepetitions=None,
                 xfrc_std=None, xfrc_rate=None, seed=0x5EED):
        num = model.numeric
        self.delegate = SamplingPlanner(model, backend, num_trajectory, horizon, seed)
        self.backend = backend
        self.nrepetitions = int(nrepetitions or num.get("robust_repetitions", [5])[0])
        nc = ncandidates if ncandidates is not None else int(num.get("robust_candidates", [-1])[0])
        self.ncandidates = int(nc if nc != -1 else self.delegate.num_trajectory // self.nrepetitions)
        self.xfrc_std = float(xfrc_std if xfrc_std is not None else num.get("robust_xfrc", [0.1])[0])
        self.xfrc_rate = float(xfrc_rate if xfrc_rate is not None else num.get("robust_xfrc_rate", [0.1])[0])
        self.seed = seed

    def reset(self, initial_repeated_action=None):
        self.delegate.reset(initial_repeated_action)

    def set_state(self, state, time, mocap):
        self.delegate.set_state(state, time, mocap)

    def optimize_policy(self):
        d = self.delegate
        knots = d.make_candidates()                                  # OptimizePolicyCandidates (planner.cc:155-194)
        ret, fail, order = self.backend.rollout_spline(d.state, d.time, d.mocap, knots, d.times, d.interp, d.horizon)
        order = np.asarray(order if order is not None else np.argsort(ret, kind="stable"))
        nc = min(self.ncandidates, d.num_trajectory)
        self.scores = None
        if nc <= 1:
            best = 0
        else:
            top = order[:nc]
            rep = self.nrepetitions
            knots2 = np.repeat(knots[top], rep, axis=0)
            self.backend.set_xfrc_noise(self.xfrc_std, self.xfrc_rate, (self.seed + d.iteration) & 0xFFFFFFFF)
            ret2, fail2, _ = self.backend.rollout_spline(d.state, d.time, d.mocap, knots2, d.times, d.interp, d.horizon)
            self.backend.set_xfrc_noise(0.0, self.xfrc_rate, 0)
            best, best_score, scores = -1, 0.0, []
            for c in range(nc):
                mean, valid = float(ret[top[c]]), 0
                for j in range(rep):
                    if fail2[rep * c + j]:
                        continue
                    mean = (valid * mean + float(ret2[rep * c + j])) / (valid + 1)
                    valid += 1
                scores.append(mean)
                if best == -1 or mean < best_score:
                    best, best_score = c, mean
            self.scores = np.array(scores)
        d.winner = int(order[best])                                   # CopyCandidateToPolicy(best)
        d.improvement = max(float(ret[0]) - float(ret[d.winner]), 0.0)
        d.values = knots[d.winner].astype(float)
        d.returns = ret
        d.iteration += 1
        self.winner = d.winner
        return ret, fail

    def action_from_policy(self, time):
        return self.delegate.action_from_policy(time)
