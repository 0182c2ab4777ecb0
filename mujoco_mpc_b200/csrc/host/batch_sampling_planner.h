// batch_sampling_planner.h - Predictive Sampling for M independent agents of the same model on ONE engine handle.
// Each agent is a SamplingPlanner without a handle of its own (policy, previous policy, seed, iteration, state, time,
// mocap) plus its own task snapshot; OptimizePolicy makes every agent's candidates with the single planner's code, rolls
// all of them out with ONE mjpc_b200_rollout_spline_batched call and installs each agent's winner.  Agent p's policy
// after any number of iterations is bit for bit that of a SamplingPlanner with the same seed and inputs.
#pragma once
#include <memory>
#include <vector>

#include "sampling_planner.h"

namespace mjpc_b200_host {

class BatchSamplingPlanner {
 public:
  ~BatchSamplingPlanner();
  int Initialize(const mjpc_model_blob* model, int num_agents, const uint32_t* seeds, int num_trajectory,
                 int num_spline_points, int interpolation, double exploration, double timestep, const double* ctrlrange,
                 int max_horizon, int device);
  int num_agents() const { return (int)agents_.size(); }
  SamplingPlanner& agent(int p) { return *agents_[p]; }
  void Reset(int agent, int horizon, const double* initial_repeated_action);
  void SetState(int agent, const double* state, double time, const double* mocap);
  // the agent's task snapshot (NULL members keep its current value; every agent starts from the model's); the risk is
  // shared by all agents: the last call's value applies
  int SetTask(int agent, const mjpc_task_desc* task);
  int OptimizePolicy(int horizon);                    // one batched launch for all agents
  mjpc_b200_t* gpu() { return gpu_; }

 private:
  mjpc_b200_t* gpu_ = nullptr;
  mjpc_b200_info info_{};
  int num_trajectory_ = 0;
  std::vector<std::unique_ptr<SamplingPlanner>> agents_;
  std::vector<double> weight_, parameters_, task_state_;   // [M][num_term], [M][num_parameters], [M][task_state_size]
  // launch staging
  std::vector<float> state_, mocap_, knots_, returns_;
  std::vector<double> time_, knot_times_;
  std::vector<uint8_t> failure_;
  std::vector<int> order_;
};

}  // namespace mjpc_b200_host
