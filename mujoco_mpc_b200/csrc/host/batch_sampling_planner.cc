// batch_sampling_planner.cc - see batch_sampling_planner.h.  Compiled into libmjpc_b200.so next to the engine.
#include "batch_sampling_planner.h"

#include <algorithm>
#include <exception>

#include "../dev_model.h"   // Blob: the model's task weights / parameters / state, every agent's initial snapshot

namespace mjpc_b200_host {

BatchSamplingPlanner::~BatchSamplingPlanner() {
  if (gpu_) mjpc_b200_destroy(gpu_);
}

int BatchSamplingPlanner::Initialize(const mjpc_model_blob* model, int num_agents, const uint32_t* seeds, int num_trajectory,
                                     int num_spline_points, int interpolation, double exploration, double timestep,
                                     const double* ctrlrange, int max_horizon, int device) {
  if (num_agents < 1 || num_trajectory < 1 || !seeds) return MJPC_B200_ERR_BAD_ARGUMENT;
  std::vector<double> w, prm, ts;
  try {
    mjpc_dev::Blob b(model->data, model->nbytes);
    w = b.reals("task_weight"); prm = b.reals("task_parameters"); ts = b.reals("task_state");
  } catch (const std::exception&) {
    return MJPC_B200_ERR_BAD_BLOB;
  }
  const long long total = (long long)num_agents * num_trajectory;
  if (total > (1 << 30)) return MJPC_B200_ERR_CAPACITY;
  if (int rc = mjpc_b200_create(model, (int)total, max_horizon, device, &gpu_)) return rc;
  mjpc_b200_get_info(gpu_, &info_);
  num_trajectory_ = num_trajectory;
  for (int p = 0; p < num_agents; p++) {
    agents_.emplace_back(new SamplingPlanner);
    agents_.back()->InitializeHost(info_, num_trajectory, num_spline_points, interpolation, exploration, 0.0, timestep,
                                   ctrlrange, seeds[p], num_trajectory);
    weight_.insert(weight_.end(), w.begin(), w.end());
    parameters_.insert(parameters_.end(), prm.begin(), prm.end());
    task_state_.insert(task_state_.end(), ts.begin(), ts.end());
  }
  return 0;
}

void BatchSamplingPlanner::Reset(int agent, int horizon, const double* initial_repeated_action) {
  agents_[agent]->Reset(horizon, initial_repeated_action);
}

void BatchSamplingPlanner::SetState(int agent, const double* state, double time, const double* mocap) {
  agents_[agent]->SetState(state, time, mocap);
}

int BatchSamplingPlanner::SetTask(int agent, const mjpc_task_desc* task) {
  const size_t nw = info_.num_term, np = info_.num_parameters, nts = info_.task_state_size;
  if (task->weight) std::copy(task->weight, task->weight + nw, weight_.begin() + agent * nw);
  if (task->parameters) std::copy(task->parameters, task->parameters + np, parameters_.begin() + agent * np);
  if (task->task_state) std::copy(task->task_state, task->task_state + nts, task_state_.begin() + agent * nts);
  const mjpc_task_desc risk_only{nullptr, nullptr, nullptr, task->risk};
  return mjpc_b200_set_task(gpu_, &risk_only);
}

// per agent: SamplingPlanner::OptimizePolicyCandidates up to the device call, then ONE batched launch, then per agent
// what SamplingPlanner::OptimizePolicy does after its own launch
int BatchSamplingPlanner::OptimizePolicy(int horizon) {
  const int M = num_agents(), N = num_trajectory_, nu = info_.nu, ds = info_.dim_state, nm = 7 * info_.nmocap;
  for (auto& a : agents_) {
    a->UpdateNominalPolicy(horizon);
    a->policy.plan.SetInterpolation(a->interpolation_);
    a->MakeCandidates(N);
  }
  const int P = agents_[0]->policy.plan.Size();
  state_.resize((size_t)M * ds); mocap_.resize((size_t)M * nm); time_.resize(M);
  knots_.resize((size_t)M * N * P * nu); knot_times_.resize((size_t)M * P);
  returns_.resize((size_t)M * N); failure_.resize((size_t)M * N); order_.resize((size_t)M * N);
  for (int p = 0; p < M; p++) {
    const SamplingPlanner& a = *agents_[p];
    std::copy(a.state_.begin(), a.state_.end(), state_.begin() + (size_t)p * ds);   // double -> float, as Rollouts does
    std::copy(a.mocap_.begin(), a.mocap_.end(), mocap_.begin() + (size_t)p * nm);
    time_[p] = a.time_;
    std::copy(a.knots_.begin(), a.knots_.end(), knots_.begin() + (size_t)p * N * P * nu);
    std::copy(a.knot_times_.begin(), a.knot_times_.end(), knot_times_.begin() + (size_t)p * P);
  }
  const mjpc_task_batch task{weight_.data(), parameters_.data(), task_state_.data()};
  if (mjpc_b200_rollout_spline_batched(gpu_, M, state_.data(), time_.data(), nm ? mocap_.data() : nullptr, &task,
                                       knots_.data(), knot_times_.data(), (int)agents_[0]->interpolation_, P, N, horizon,
                                       returns_.data(), failure_.data(), order_.data()))
    return -1;
  for (int p = 0; p < M; p++) {
    SamplingPlanner& a = *agents_[p];
    std::copy(returns_.begin() + (size_t)p * N, returns_.begin() + (size_t)(p + 1) * N, a.returns_.begin());
    std::copy(failure_.begin() + (size_t)p * N, failure_.begin() + (size_t)(p + 1) * N, a.failure_.begin());
    a.trajectory_order.assign(order_.begin() + (size_t)p * N, order_.begin() + (size_t)(p + 1) * N);
    a.InstallWinner();
  }
  return 0;
}

}  // namespace mjpc_b200_host

// ------------------------------------------------------------------------------------------ C entry points
using mjpc_b200_host::BatchSamplingPlanner;

extern "C" {

int mjpc_b200_batch_planner_create(const mjpc_model_blob* model, int num_agents, const uint32_t* seeds, int num_trajectory,
                                   int num_spline_points, int interpolation, double exploration, double timestep,
                                   const double* ctrlrange, int max_horizon, int device, void** out) {
  if (!model || !seeds || !ctrlrange || !out) return MJPC_B200_ERR_BAD_ARGUMENT;
  auto* p = new BatchSamplingPlanner;
  int rc = p->Initialize(model, num_agents, seeds, num_trajectory, num_spline_points, interpolation, exploration, timestep,
                         ctrlrange, max_horizon, device);
  if (rc) { delete p; *out = nullptr; return rc; }
  *out = p;
  return 0;
}
void mjpc_b200_batch_planner_destroy(void* p) { delete (BatchSamplingPlanner*)p; }
void mjpc_b200_batch_planner_reset(void* p, int agent, int horizon, const double* initial_repeated_action) {
  ((BatchSamplingPlanner*)p)->Reset(agent, horizon, initial_repeated_action);
}
void mjpc_b200_batch_planner_set_state(void* p, int agent, const double* state, double time, const double* mocap) {
  ((BatchSamplingPlanner*)p)->SetState(agent, state, time, mocap);
}
int mjpc_b200_batch_planner_set_task(void* p, int agent, const mjpc_task_desc* task) {
  if (!p || !task) return MJPC_B200_ERR_BAD_ARGUMENT;
  return ((BatchSamplingPlanner*)p)->SetTask(agent, task);
}
int mjpc_b200_batch_planner_optimize_policy(void* p, int horizon) { return ((BatchSamplingPlanner*)p)->OptimizePolicy(horizon); }
void mjpc_b200_batch_planner_action_from_policy(void* p, int agent, double* action, double time, int use_previous) {
  ((BatchSamplingPlanner*)p)->agent(agent).ActionFromPolicy(action, time, use_previous != 0);
}
int mjpc_b200_batch_planner_get_result(void* pv, int agent, int* winner, double* improvement, float* returns, double* knots,
                                       double* knot_times) {
  auto& a = ((BatchSamplingPlanner*)pv)->agent(agent);
  if (winner) *winner = a.winner;
  if (improvement) *improvement = a.improvement;
  if (returns) std::copy(a.returns().begin(), a.returns().end(), returns);
  const auto& plan = a.policy.plan;
  for (int k = 0; k < plan.Size(); k++) {
    if (knot_times) knot_times[k] = plan.NodeTime(k);
    if (knots) std::copy(plan.NodeValues(k), plan.NodeValues(k) + plan.Dim(), knots + (size_t)k * plan.Dim());
  }
  return plan.Size();
}

}  // extern "C"
