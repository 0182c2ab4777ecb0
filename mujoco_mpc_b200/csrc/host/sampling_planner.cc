// sampling_planner.cc - see sampling_planner.h.  Compiled into libmjpc_b200.so next to the engine.
#include "sampling_planner.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include <numeric>

namespace mjpc_b200_host {

// ------------------------------------------------------------------------------------------ TimeSpline
void TimeSpline::AddNode(double time, const double* values) {
  times_.push_back(time);
  for (int i = 0; i < dim_; i++) values_.push_back(values ? values[i] : 0.0);
}

double TimeSpline::Slope(int node, int k) const {
  const int P = Size();
  auto v = [&](int n) { return values_[(size_t)n * dim_ + k]; };
  if (node == 0) return (v(1) - v(0)) / (times_[1] - times_[0]);
  if (node == P - 1) return (v(node) - v(node - 1)) / (times_[node] - times_[node - 1]);
  return 0.5 * (v(node + 1) - v(node)) / (times_[node + 1] - times_[node]) +
         0.5 * (v(node) - v(node - 1)) / (times_[node] - times_[node - 1]);
}

void TimeSpline::Sample(double time, double* out) const {
  const int P = Size();
  if (P == 0) { std::fill(out, out + dim_, 0.0); return; }
  const int upper = (int)(std::upper_bound(times_.begin(), times_.end(), time) - times_.begin());
  if (upper == P) { std::copy(NodeValues(P - 1), NodeValues(P - 1) + dim_, out); return; }
  if (upper == 0) { std::copy(NodeValues(0), NodeValues(0) + dim_, out); return; }
  const int lower = upper - 1;
  const double dt = times_[upper] - times_[lower];
  const double t = (time - times_[lower]) / dt;
  const double *lo = NodeValues(lower), *hi = NodeValues(upper);
  switch (interpolation_) {
    case kZeroSpline: std::copy(lo, lo + dim_, out); return;
    case kLinearSpline:
      for (int i = 0; i < dim_; i++) out[i] = lo[i] * (1 - t) + hi[i] * t;
      return;
    case kCubicSpline: {
      const double c0 = 2 * t * t * t - 3 * t * t + 1, c1 = (t * t * t - 2 * t * t + t) * dt,
                   c2 = -2 * t * t * t + 3 * t * t, c3 = (t * t * t - t * t) * dt;
      for (int i = 0; i < dim_; i++) out[i] = c0 * lo[i] + c1 * Slope(lower, i) + c2 * hi[i] + c3 * Slope(upper, i);
      return;
    }
  }
}

void SamplingPolicy::Action(double* action, double time) const {
  plan.Sample(time, action);
  for (int i = 0; i < plan.Dim(); i++) action[i] = std::max(ctrlrange[2 * i], std::min(ctrlrange[2 * i + 1], action[i]));
}

// ------------------------------------------------------------------------------------------ injected noise
void Philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
  uint32_t k0 = key[0], k1 = key[1];
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n[4] = {(uint32_t)(p1 >> 32) ^ c[1] ^ k0, (uint32_t)p1, (uint32_t)(p0 >> 32) ^ c[3] ^ k1, (uint32_t)p0};
    std::memcpy(c, n, sizeof(c));
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  std::memcpy(out, c, sizeof(c));
}

double PhiloxNormal(uint32_t seed, uint32_t iteration, uint32_t candidate, uint32_t knot, uint32_t dof) {
  const uint32_t ctr[4] = {iteration, candidate, knot, dof}, key[2] = {seed, 0};
  uint32_t r[4];
  Philox4x32(ctr, key, r);
  const double u1 = ((double)r[0] + 0.5) / 4294967296.0, u2 = ((double)r[1] + 0.5) / 4294967296.0;
  return std::sqrt(-2.0 * std::log(u1)) * std::cos(2.0 * M_PI * u2);
}

// ------------------------------------------------------------------------------------------ SamplingPlanner
SamplingPlanner::~SamplingPlanner() {
  if (gpu_) mjpc_b200_destroy(gpu_);
}

int SamplingPlanner::Initialize(const mjpc_model_blob* model, int num_trajectory, int num_spline_points, int interpolation,
                                double exploration, double exploration2, double timestep, const double* ctrlrange,
                                uint32_t seed, int max_candidates, int max_horizon, int device) {
  int rc = mjpc_b200_create(model, max_candidates, max_horizon, device, &gpu_);
  if (rc) return rc;
  mjpc_b200_info info;
  mjpc_b200_get_info(gpu_, &info);
  InitializeHost(info, num_trajectory, num_spline_points, interpolation, exploration, exploration2, timestep, ctrlrange, seed,
                 max_candidates);
  return 0;
}

void SamplingPlanner::InitializeHost(const mjpc_b200_info& info, int num_trajectory, int num_spline_points, int interpolation,
                                     double exploration, double exploration2, double timestep, const double* ctrlrange,
                                     uint32_t seed, int max_candidates) {
  info_ = info;
  nu_ = info_.nu;
  num_trajectory_ = num_trajectory;
  interpolation_ = (SplineInterpolation)interpolation;
  noise_exploration_[0] = exploration; noise_exploration_[1] = exploration2;
  timestep_ = timestep; seed_ = seed;
  policy.plan = TimeSpline(nu_, interpolation_);
  policy.num_spline_points = num_spline_points;
  policy.ctrlrange.assign(ctrlrange, ctrlrange + 2 * nu_);
  previous_policy = policy;
  candidate_policy.assign(max_candidates, policy);
  state_.assign(info_.dim_state, 0.0); mocap_.assign(7 * info_.nmocap, 0.0);
  returns_.assign(max_candidates, 0.f); failure_.assign(max_candidates, 0);
  winner = 0;
}

void SamplingPlanner::Reset(int, const double* initial_repeated_action) {
  policy.plan.Clear();
  if (initial_repeated_action) policy.plan.AddNode(0, initial_repeated_action);
  previous_policy = policy;
  for (auto& cp : candidate_policy) cp = policy;
  winner = 0; iteration = 0; improvement = 0;
}

void SamplingPlanner::SetState(const double* state, double time, const double* mocap) {
  std::copy(state, state + state_.size(), state_.begin());
  if (!mocap_.empty()) std::copy(mocap, mocap + mocap_.size(), mocap_.begin());
  time_ = time;
}

void SamplingPlanner::UpdateNominalPolicy(int horizon) {
  const int P = candidate_policy[winner].num_spline_points;
  double nominal_time = time_;
  const double time_horizon = (horizon - 1) * timestep_;
  const double time_shift = interpolation_ == kZeroSpline ? std::max(time_horizon / P, 1.0e-5)
                                                          : std::max(time_horizon / (P - 1), 1.0e-5);
  TimeSpline scratch(nu_, interpolation_);
  std::vector<double> v(nu_);
  for (int t = 0; t < P; t++) {
    candidate_policy[winner].plan.SetInterpolation(interpolation_);
    candidate_policy[winner].Action(v.data(), nominal_time);
    scratch.AddNode(nominal_time, v.data());
    nominal_time += time_shift;
  }
  const std::unique_lock<std::shared_mutex> lock(mtx_);
  policy.plan = scratch;
}

void SamplingPlanner::AddNoiseToPolicy(int i) {
  // fixed std (the optional second std with p = 0.2, planner.cc:334-338, needs a Bernoulli draw: word 2 of the
  // candidate's first Philox block)
  double std = noise_exploration_[0];
  if (noise_exploration_[1] > 0) {
    const uint32_t ctr[4] = {(uint32_t)iteration, (uint32_t)i, 0xffffffffu, 0}, key[2] = {seed_, 0};
    uint32_t r[4];
    Philox4x32(ctr, key, r);
    if (((double)r[2] + 0.5) / 4294967296.0 < 0.2) std = noise_exploration_[1];
  }
  TimeSpline& plan = candidate_policy[i].plan;
  for (int k = 0; k < plan.Size(); k++) {
    double* node = plan.NodeValues(k);
    for (int d = 0; d < nu_; d++) {
      const double lo = policy.ctrlrange[2 * d], hi = policy.ctrlrange[2 * d + 1];
      const double scale = 0.5 * (hi - lo);
      node[d] += scale * std * PhiloxNormal(seed_, (uint32_t)iteration, (uint32_t)i, (uint32_t)k, (uint32_t)d);
      node[d] = std::max(lo, std::min(hi, node[d]));
    }
  }
}

void SamplingPlanner::MakeCandidates(int num_trajectory) {
  const int P = policy.plan.Size();
  knots_.resize((size_t)num_trajectory * P * nu_);
  knot_times_.resize(P);
  for (int i = 0; i < num_trajectory; i++) {
    {
      const std::shared_lock<std::shared_mutex> lock(mtx_);
      candidate_policy[i] = policy;
    }
    if (i != 0) AddNoiseToPolicy(i);
    for (int k = 0; k < P; k++) {
      const double* node = candidate_policy[i].plan.NodeValues(k);
      for (int d = 0; d < nu_; d++) knots_[((size_t)i * P + k) * nu_ + d] = (float)node[d];
    }
  }
  for (int k = 0; k < P; k++) knot_times_[k] = policy.plan.NodeTime(k);
}

int SamplingPlanner::Rollouts(int num_trajectory, int horizon) {
  MakeCandidates(num_trajectory);
  const int P = policy.plan.Size();
  std::vector<float> state_f(state_.begin(), state_.end()), mocap_f(mocap_.begin(), mocap_.end());
  trajectory_order.resize(num_trajectory);
  return mjpc_b200_rollout_spline(gpu_, state_f.data(), time_, mocap_f.empty() ? nullptr : mocap_f.data(), nullptr,
                                  knots_.data(), knot_times_.data(), (int)interpolation_, P, num_trajectory, horizon,
                                  returns_.data(), failure_.data(), trajectory_order.data());
}

int SamplingPlanner::OptimizePolicyCandidates(int ncandidates, int horizon) {
  UpdateNominalPolicy(horizon);
  const int num_trajectory = num_trajectory_;
  ncandidates = std::min(ncandidates, num_trajectory);
  policy.plan.SetInterpolation(interpolation_);
  if (int rc = Rollouts(num_trajectory, horizon)) return -1;   // device ranking replaces partial_sort (:184-188)
  return ncandidates;
}

int SamplingPlanner::OptimizePolicy(int horizon) {
  if (OptimizePolicyCandidates(1, horizon) < 0) return -1;
  InstallWinner();
  return 0;
}

void SamplingPlanner::InstallWinner() {
  CopyCandidateToPolicy(0);
  const double best_return = returns_[0];   // candidate 0 is the un-noised nominal
  improvement = std::max(best_return - (double)returns_[winner], 0.0);
  iteration++;
}

void SamplingPlanner::CopyCandidateToPolicy(int candidate) {
  winner = trajectory_order[candidate];
  const std::unique_lock<std::shared_mutex> lock(mtx_);
  previous_policy = policy;
  policy = candidate_policy[winner];
}

void SamplingPlanner::ActionFromPolicy(double* action, double time, bool use_previous) {
  const std::shared_lock<std::shared_mutex> lock(mtx_);
  (use_previous ? previous_policy : policy).Action(action, time);
}

int SamplingPlanner::FetchTrajectory(int candidate, int horizon, Trajectory* t) {
  const mjpc_b200_info& in = info_;
  const size_t H = horizon;
  t->horizon = horizon; t->dim_state = in.dim_state; t->dim_action = in.nu; t->dim_residual = in.num_residual;
  t->dim_trace = 3 * in.num_trace;
  t->states.resize(H * in.dim_state); t->actions.resize(H * in.nu); t->times.resize(H);
  t->residual.resize(H * in.num_residual); t->costs.resize(H); t->trace.resize(H * t->dim_trace);
  if (mjpc_b200_fetch_trajectory(gpu_, candidate, t->states.data(), t->actions.data(), t->times.data(), t->residual.data(),
                                 t->costs.data(), t->trace.data()))
    return -1;
  t->total_return = returns_[candidate];
  t->failure = failure_[candidate];
  return 0;
}

void SamplingPlanner::SetPolicy(const double* times, const double* parameters, int num_nodes) {
  const std::unique_lock<std::shared_mutex> lock(mtx_);
  policy.plan.Clear();
  for (int t = 0; t < num_nodes; t++) policy.plan.AddNode(times[t], parameters + (size_t)t * nu_);
}

const Trajectory* SamplingPlanner::BestTrajectory() {
  mjpc_b200_info& in = info_;
  const int H = in.max_horizon;
  best_.dim_state = in.dim_state; best_.dim_action = in.nu; best_.dim_residual = in.num_residual;
  best_.dim_trace = 3 * in.num_trace;
  best_.states.resize((size_t)H * in.dim_state); best_.actions.resize((size_t)H * in.nu); best_.times.resize(H);
  best_.residual.resize((size_t)H * in.num_residual); best_.costs.resize(H); best_.trace.resize((size_t)H * best_.dim_trace);
  if (mjpc_b200_fetch_trajectory(gpu_, winner, best_.states.data(), best_.actions.data(), best_.times.data(),
                                 best_.residual.data(), best_.costs.data(), best_.trace.data()))
    return nullptr;
  best_.total_return = returns_[winner];
  best_.failure = failure_[winner];
  return &best_;
}

}  // namespace mjpc_b200_host

// ------------------------------------------------------------------------------------------ C entry points
// (declared in include/mjpc_b200.h; what a ctypes / test harness binds)
using mjpc_b200_host::SamplingPlanner;

extern "C" {

void mjpc_b200_host_spline_sample(const double* times, const double* values, int P, int dim, int interp, double t,
                                  double* out) {
  mjpc_b200_host::TimeSpline s(dim, (mjpc_b200_host::SplineInterpolation)interp);
  for (int i = 0; i < P; i++) s.AddNode(times[i], values + (size_t)i * dim);
  s.Sample(t, out);
}

double mjpc_b200_host_philox_normal(uint32_t seed, uint32_t iteration, uint32_t candidate, uint32_t knot, uint32_t dof) {
  return mjpc_b200_host::PhiloxNormal(seed, iteration, candidate, knot, dof);
}

int mjpc_b200_planner_create(const mjpc_model_blob* model, int num_trajectory, int num_spline_points, int interpolation,
                             double exploration, double timestep, const double* ctrlrange, uint32_t seed, int max_horizon,
                             int device, void** out) {
  if (!model || !ctrlrange || !out) return MJPC_B200_ERR_BAD_ARGUMENT;
  auto* p = new SamplingPlanner;
  int rc = p->Initialize(model, num_trajectory, num_spline_points, interpolation, exploration, 0.0, timestep, ctrlrange,
                         seed, num_trajectory, max_horizon, device);
  if (rc) { delete p; *out = nullptr; return rc; }
  *out = p;
  return 0;
}
void mjpc_b200_planner_destroy(void* p) { delete (SamplingPlanner*)p; }
// noise_exploration[0..1] (sampling/planner.cc:85-88): the second std, when > 0, replaces the first with probability 0.2
void mjpc_b200_planner_set_exploration(void* p, double exploration, double exploration2) {
  ((SamplingPlanner*)p)->SetExploration(exploration, exploration2);
}
void mjpc_b200_planner_reset(void* p, int horizon, const double* initial_repeated_action) {
  ((SamplingPlanner*)p)->Reset(horizon, initial_repeated_action);
}
void mjpc_b200_planner_set_state(void* p, const double* state, double time, const double* mocap) {
  ((SamplingPlanner*)p)->SetState(state, time, mocap);
}
int mjpc_b200_planner_optimize_policy(void* p, int horizon) { return ((SamplingPlanner*)p)->OptimizePolicy(horizon); }
void mjpc_b200_planner_action_from_policy(void* p, double* action, double time, int use_previous) {
  ((SamplingPlanner*)p)->ActionFromPolicy(action, time, use_previous != 0);
}
// winner index, improvement, returns [num_trajectory], policy knots [P][nu] and times [P] of the installed policy
int mjpc_b200_planner_get_result(void* pv, int* winner, double* improvement, float* returns, double* knots, double* knot_times) {
  auto* p = (SamplingPlanner*)pv;
  if (winner) *winner = p->winner;
  if (improvement) *improvement = p->improvement;
  if (returns) std::copy(p->returns().begin(), p->returns().end(), returns);
  const auto& plan = p->policy.plan;
  for (int k = 0; k < plan.Size(); k++) {
    if (knot_times) knot_times[k] = plan.NodeTime(k);
    if (knots) std::copy(plan.NodeValues(k), plan.NodeValues(k) + plan.Dim(), knots + (size_t)k * plan.Dim());
  }
  return plan.Size();
}

}  // extern "C"
