// sampling_planner.h - C++ host side above the C ABI: the Predictive Sampling planner with the reference's
// method names (mjpc/planners/sampling/planner.h:40-160, planner.cc:40-560), TimeSpline (mjpc/spline/spline.h)
// and SamplingPolicy (mjpc/planners/sampling/policy.cc:52-59).  Only Rollouts() differs from the reference: it
// makes ONE mjpc_b200_rollout_spline call instead of scheduling N closures on a ThreadPool.
//
// The reference's absl::BitGen cannot be seeded (planner.cc:331), so the noise source is injected:
// Philox4x32-10, key (seed, 0), counter (iteration, candidate, knot, dof), Box-Muller on the first two words.
#pragma once
#include <array>
#include <cstdint>
#include <shared_mutex>
#include <vector>

#include "../../../include/mjpc_b200.h"

namespace mjpc_b200_host {

enum SplineInterpolation : int { kZeroSpline = 0, kLinearSpline = 1, kCubicSpline = 2 };

// time-indexed knots, values row-major [node][dim]
class TimeSpline {
 public:
  explicit TimeSpline(int dim = 0, SplineInterpolation interp = kZeroSpline) : dim_(dim), interpolation_(interp) {}
  int Dim() const { return dim_; }
  int Size() const { return (int)times_.size(); }
  void Clear() { times_.clear(); values_.clear(); }
  void SetInterpolation(SplineInterpolation i) { interpolation_ = i; }
  SplineInterpolation Interpolation() const { return interpolation_; }
  void AddNode(double time, const double* values);   // values == nullptr -> zeros
  double NodeTime(int i) const { return times_[i]; }
  double* NodeValues(int i) { return values_.data() + (size_t)i * dim_; }
  const double* NodeValues(int i) const { return values_.data() + (size_t)i * dim_; }
  void Sample(double time, double* out) const;       // spline.cc:103-156
 private:
  double Slope(int node, int k) const;               // spline.cc:269-287
  int dim_;
  SplineInterpolation interpolation_;
  std::vector<double> times_, values_;
};

struct SamplingPolicy {
  TimeSpline plan;
  std::vector<double> ctrlrange;  // [nu][2]
  int num_spline_points = 3;
  void Action(double* action, double time) const;    // Sample + Clamp
};

void Philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
double PhiloxNormal(uint32_t seed, uint32_t iteration, uint32_t candidate, uint32_t knot, uint32_t dof);

struct Trajectory {                                   // mjpc/trajectory.h:74-86 (device arithmetic: float)
  int horizon = 0, dim_state = 0, dim_action = 0, dim_residual = 0, dim_trace = 0;
  std::vector<float> states, actions, residual, costs, trace;
  std::vector<double> times;
  double total_return = 0;
  bool failure = false;
};

class SamplingPlanner {
 public:
  ~SamplingPlanner();
  // model blob + settings that the reference reads from <custom> numerics (planner.cc:54-68)
  int Initialize(const mjpc_model_blob* model, int num_trajectory, int num_spline_points, int interpolation,
                 double exploration, double exploration2, double timestep, const double* ctrlrange, uint32_t seed,
                 int max_candidates, int max_horizon, int device);
  // the same without an engine handle: a planner whose rollouts another object launches (BatchSamplingPlanner)
  void InitializeHost(const mjpc_b200_info& info, int num_trajectory, int num_spline_points, int interpolation,
                      double exploration, double exploration2, double timestep, const double* ctrlrange, uint32_t seed,
                      int max_candidates);
  void Reset(int horizon, const double* initial_repeated_action);
  void SetState(const double* state, double time, const double* mocap);
  int OptimizePolicy(int horizon);                    // planner.cc:197-212
  int OptimizePolicyCandidates(int ncandidates, int horizon);   // :155-194
  void UpdateNominalPolicy(int horizon);              // :240-323 (non-sliding resample)
  void AddNoiseToPolicy(int i);                       // :326-352
  int Rollouts(int num_trajectory, int horizon);      // :355-393 -> MakeCandidates + one C-ABI call
  void MakeCandidates(int num_trajectory);            // candidate policies (nominal + noise) and their knots
  void InstallWinner();                               // OptimizePolicy after the rollouts: best candidate -> policy
  void ActionFromPolicy(double* action, double time, bool use_previous = false);   // :229-237
  void CopyCandidateToPolicy(int candidate);          // :534-543
  const Trajectory* BestTrajectory();
  int FetchTrajectory(int candidate, int horizon, Trajectory* out);   // trajectory[candidate] of the last Rollouts
  void SetPolicy(const double* times, const double* parameters, int num_nodes);   // policy.plan = nodes (ilqs/planner.cc:160-172)
  double time() const { return time_; }
  double timestep() const { return timestep_; }
  SplineInterpolation interpolation() const { return interpolation_; }
  double CandidateScore(int candidate) const { return returns_[trajectory_order[candidate]]; }
  int NumParameters() const { return nu_ * policy.num_spline_points; }

  SamplingPolicy policy, previous_policy;
  std::vector<SamplingPolicy> candidate_policy;
  std::vector<int> trajectory_order;
  int winner = 0;
  double improvement = 0;
  int iteration = 0;
  mjpc_b200_t* gpu() { return gpu_; }
  const std::vector<float>& returns() const { return returns_; }
  // noise_exploration[0..1] (sampling/planner.cc:85-88)
  void SetExploration(double e0, double e1) { noise_exploration_[0] = e0; noise_exploration_[1] = e1; }

 private:
  friend class BatchSamplingPlanner;                  // launches the rollouts of many planners at once
  mjpc_b200_t* gpu_ = nullptr;
  mjpc_b200_info info_{};
  int num_trajectory_ = 0, nu_ = 0;
  SplineInterpolation interpolation_ = kCubicSpline;
  double noise_exploration_[2] = {0.1, 0.0};
  double timestep_ = 0.01;
  uint32_t seed_ = 0x5EED;
  std::vector<double> state_, mocap_;
  double time_ = 0;
  std::vector<float> knots_, returns_;
  std::vector<double> knot_times_;
  std::vector<uint8_t> failure_;
  Trajectory best_;
  mutable std::shared_mutex mtx_;
};

}  // namespace mjpc_b200_host
