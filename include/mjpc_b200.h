/* mjpc_b200.h - C ABI of the B200 rollout engine (libmjpc_b200.so).
 *
 * The engine replaces the data-parallel hot path of MJPC and nothing else.  std::function policies and
 * virtual ResidualFn objects cannot cross to the device, so every entry point takes *data* and sits exactly
 * where the reference fans work out over its ThreadPool:
 *
 *   mjpc_b200_rollout_spline    <- SamplingPlanner::Rollouts            mjpc/planners/sampling/planner.cc:355-393
 *                                  (+ Trajectory::Rollout/NoisyRollout  mjpc/trajectory.cc:92-210,
 *                                     SamplingPolicy::Action            mjpc/planners/sampling/policy.cc:52-59,
 *                                     UpdateReturn                      mjpc/trajectory.cc:312-326,
 *                                     partial_sort by return            mjpc/planners/sampling/planner.cc:184-188)
 *   mjpc_b200_rollout_feedback  <- iLQGPlanner::FeedbackRollouts / ActionRollouts
 *                                                                       mjpc/planners/ilqg/planner.cc:630-724
 *                                  (+ iLQGPolicy::Action                mjpc/planners/ilqg/policy.cc:82-161,
 *                                     Trajectory::RolloutDiscrete       mjpc/trajectory.cc:213-309)
 *   mjpc_b200_model_derivatives <- ModelDerivatives::Compute            mjpc/planners/model_derivatives.cc:45-165
 *   mjpc_b200_cost_derivatives  <- CostDerivatives::Compute             mjpc/planners/cost_derivatives.cc:112-230
 *   mjpc_b200_backward_pass     <- RiccatiStep recursion                mjpc/planners/ilqg/planner.cc:429-520,
 *                                                                       mjpc/planners/ilqg/backward_pass.cc:65-250
 *   mjpc_b200_set_task          <- residual_fn_ snapshot per PlanIteration  mjpc/agent.cc:316-319, task.cc:112-128
 *   mjpc_b200_fetch_trajectory  <- fills a mjpc::Trajectory             mjpc/trajectory.h:74-86
 *   create / destroy            <- Planner::Initialize/Allocate + ResizeMjData  mjpc/planners/planner.cc:23-33;
 *                                  precedent for a C surface: mjpc/interface.h:44-49
 *
 * Conventions: all pointers are HOST memory owned by the caller; the handle owns every device buffer and
 * stream.  All calls come from the single plan thread (as Agent::PlanIteration does today).  Functions return
 * 0 on success or a negative mjpc_b200_error; they never throw or abort.  Per-candidate divergence is
 * reported through failure[i] (= Trajectory::failure) with returns[i] = 1e6 (mjpc/trajectory.cc:29,169-173).
 * Arithmetic on the device is fp32; time is carried relative to the rollout start and returned as double.
 */
#ifndef MJPC_B200_H_
#define MJPC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mjpc_b200 mjpc_b200_t;

typedef enum {
  MJPC_B200_OK = 0,
  MJPC_B200_ERR_BAD_ARGUMENT = -1,
  MJPC_B200_ERR_BAD_BLOB = -2,
  MJPC_B200_ERR_CAPACITY = -3,   /* N / H above what create() reserved, or model too large for shared memory */
  MJPC_B200_ERR_CUDA = -4,       /* no device, launch or copy failure: the engine has NO CPU fallback */
  MJPC_B200_ERR_UNSUPPORTED = -5 /* model feature outside the implemented subset */
} mjpc_b200_error;

/* Flat model + task description (field names = mjModel's); written by mujoco_mpc_b200/blob.py, or by a
 * maintainer from an mjModel* (INTEGRATION.md).  The engine copies what it needs during create(). */
typedef struct {
  const void* data;
  size_t nbytes;
} mjpc_model_blob;

/* Live task snapshot (BaseResidualFn::Update, mjpc/task.cc:112-123). NULL members keep the current value. */
typedef struct {
  const double* weight;      /* [num_term]                         Task::weight        */
  const double* parameters;  /* [num_parameters]                   Task::parameters    */
  const double* task_state;  /* residual-specific state block (e.g. quadruped mode/gait/phase), see DESIGN.md */
  double risk;               /* Task::risk                                              */
} mjpc_task_desc;

typedef struct {
  int nq, nv, nu, na, nmocap, nuserdata;
  int dim_state;        /* nq + nv + na   */
  int dim_dstate;       /* 2*nv + na      */
  int num_residual, num_term, num_trace, num_parameters, task_state_size;
  int max_candidates, max_horizon;
  int device;           /* CUDA device ordinal in use */
  int smem_bytes_per_warp;
} mjpc_b200_info;

/* interp: 0 zero-order, 1 linear, 2 cubic (mjpc/spline/spline.h SplineInterpolation) */
/* feedback mode: 0/1/2 time-indexed with that interpolation (iLQGPolicy::representation), 3 step-indexed */

const char* mjpc_b200_version(void);
const char* mjpc_b200_last_error(void);

int mjpc_b200_create(const mjpc_model_blob* model, int max_candidates, int max_horizon, int device,
                     mjpc_b200_t** out);
void mjpc_b200_destroy(mjpc_b200_t* h);
int mjpc_b200_get_info(const mjpc_b200_t* h, mjpc_b200_info* info);

int mjpc_b200_set_task(mjpc_b200_t* h, const mjpc_task_desc* task);

/* Planning-model overrides of Agent::PlanIteration (agent.cc:288-289): opt.timestep = agent_timestep, opt.integrator =
 * agent_integrator, for the following calls of this handle.  Only the Euler integrator (0) is implemented: any other value
 * returns MJPC_B200_ERR_UNSUPPORTED. */
int mjpc_b200_set_options(mjpc_b200_t* h, double timestep, int integrator);

/* MakeDifferentiable (mjpc/utilities.cc:60-75) for the following calls of this handle: on != 0 zeroes solimp[0] of every
 * joint and geom in the model the kernels read, 0 restores the model's values - what Agent::PlanIteration does around
 * OptimizePolicy for gradient-based planners (agent.cc:296-309,346-356; default on for iLQG / iLQS / Gradient,
 * agent.cc:158-164).  The C++ iLQG planner switches it on unless iLQGSettings::differentiable is cleared. */
int mjpc_b200_set_differentiable(mjpc_b200_t* h, int on);

/* N candidate splines -> N rollouts of H steps. knots [N][P][nu]; knot_times [P] (absolute seconds).
 * candidate_offset: global index of this handle's first candidate (multi-GPU sharding; only used for bookkeeping).
 * returns [N], failure [N]; order [N] = candidate indices sorted by return (ties: lower index first), may be NULL. */
int mjpc_b200_rollout_spline(mjpc_b200_t* h, const float* state, double time, const float* mocap,
                             const float* userdata, const float* knots, const double* knot_times, int interp,
                             int P, int N, int H, float* returns, uint8_t* failure, int* order);

/* Per-problem task snapshot of a batched rollout; a NULL member = the handle's current value for every problem. */
typedef struct {
  const double* weight;      /* [M][num_term]                                                             */
  const double* parameters;  /* [M][num_parameters]                                                       */
  const double* task_state;  /* [M][task_state_size] (absolute times; rebased per problem like set_task's) */
} mjpc_task_batch;

/* M independent planning problems of this handle's model in ONE launch: problem p is (state [p], time [p], mocap [p],
 * task rows p, knots [p][N][P][nu], knot_times [p][P]); all share N, P, H, interp and the handle's risk, timestep,
 * differentiable flag and xfrc noise settings.  Problem p's returns [p][N], failure [p][N] and order [p][N] (problem-local
 * indices, ascending return, ties: lower index first; may be NULL) are bit for bit what mjpc_b200_rollout_spline returns
 * for that problem alone, and so are its trajectories: fetch_trajectory / fetch_all / fetch_stats see the M*N candidates
 * problem-major (candidate i of problem p is p*N + i).  M*N above max_candidates returns MJPC_B200_ERR_CAPACITY; mocap
 * [M][7 nmocap] is required when nmocap > 0; userdata is not accepted.  Never uses a communicator (comm_init). */
int mjpc_b200_rollout_spline_batched(mjpc_b200_t* h, int M, const float* state, const double* time, const float* mocap,
                                     const mjpc_task_batch* task, const float* knots, const double* knot_times, int interp,
                                     int P, int N, int H, float* returns, uint8_t* failure, int* order);

/* NoisyRollout (mjpc/trajectory.cc:100-210, used by the Robust planner): the following rollouts of this handle add
 * Ornstein-Uhlenbeck noise to xfrc_applied of every body (stationary std xfrc_std, correlation time xfrc_rate
 * seconds), drawn from Philox4x32-10 with key (seed, 1) and counter (step, candidate, element, 'XFRC') - the
 * reference's absl::BitGen cannot be seeded.  xfrc_std = 0 switches the noise off (the default). */
int mjpc_b200_set_xfrc_noise(mjpc_b200_t* h, double xfrc_std, double xfrc_rate, uint32_t seed);

/* K line-search rollouts of the iLQG policy. u_nom [H][nu], x_nom [H][dim_state], t_nom [H] (absolute),
 * gains [H][nu][dim_dstate], du [H][nu] (may be NULL), step_sizes [K]. */
int mjpc_b200_rollout_feedback(mjpc_b200_t* h, const float* state, double time, const float* mocap,
                               const float* userdata, const float* u_nom, const float* x_nom, const double* t_nom,
                               const float* gains, const float* du, const float* step_sizes, int mode, int K, int H,
                               float* returns, uint8_t* failure, int* order);

/* Copy candidate i of the last rollout into Trajectory-shaped host arrays (any pointer may be NULL):
 * states [H][dim_state], actions [H][nu], times [H], residual [H][num_residual], costs [H], trace [H][3*num_trace] */
int mjpc_b200_fetch_trajectory(mjpc_b200_t* h, int candidate, float* states, float* actions, double* times,
                               float* residual, float* costs, float* trace);
/* Bulk variant: every candidate of the last rollout ([N] leading dimension). */
int mjpc_b200_fetch_all(mjpc_b200_t* h, float* states, float* actions, double* times, float* residual,
                        float* costs, float* trace);

/* Finite-difference transition / residual Jacobians along a trajectory (ModelDerivatives::Compute,
 * model_derivatives.cc:45-165).  x [H][dim_state], u [H][nu], t [H]; A [H][n][n], B [H][n][nu], C [H][nr][n],
 * D [H][nr][nu], n = dim_dstate, nr = num_residual (the rows CostDerivatives reads).
 *   skip  derivative_skip: only every (skip+1)-th step plus H-2 and H-1 is differentiated, the rest is linearly
 *         interpolated between its evaluated neighbours (model_derivatives.cc:56-72,109-164); 0 = every step
 *   tol   finite-difference step (ilqg/settings.h:23, reference default 1e-6 in double; fp32 wants ~1e-3)
 *   mode  0 one-sided, 1 centred (ilqg/settings.h:24 fd_mode -> mjd_transitionFD flg_centered)
 * Row H-1 of A, B, D is left zero (model_derivatives.cc:89-93). */
int mjpc_b200_model_derivatives(mjpc_b200_t* h, const float* x, const float* u, const double* t,
                                const float* mocap, int H, int skip, float tol, int mode, float* A, float* B,
                                float* C, float* D);

/* Gauss-Newton cost derivatives. residual [H][nr], C, D as above -> cx [H][n], cu [H][nu], cxx [H][n][n],
 * cuu [H][nu][nu], cxu [H][n][nu]. */
int mjpc_b200_cost_derivatives(mjpc_b200_t* h, const float* residual, const float* C, const float* D, int H,
                               float* cx, float* cu, float* cxx, float* cuu, float* cxu);

/* One Riccati sweep at fixed regularisation. status_out: 1 success, 0 failure (caller scales mu and retries).
 * reg_type 0 control, 1 state-control, 2 value, 3 none; limits 1 = box-QP within ctrlrange - action.
 * Outputs: K [H][nu][n], du [H][nu], dV[2], and (optional, may be NULL) Vx [H][n], Vxx [H][n][n]. */
int mjpc_b200_backward_pass(mjpc_b200_t* h, const float* A, const float* B, const float* cx, const float* cu,
                            const float* cxx, const float* cxu, const float* cuu, const float* actions, int H,
                            float mu, int reg_type, int limits, float* K, float* du, float* dV, float* Vx,
                            float* Vxx, int* status_out);

/* Debug / parity hook: one forward-dynamics evaluation + Euler step for a single state through the same
 * device code the rollout kernel runs. qacc[nv], residual[nr], next_qpos[nq], next_qvel[nv], counts[4] =
 * {ncon, nefc, solver iterations, warning}. */
int mjpc_b200_step_debug(mjpc_b200_t* h, const float* qpos, const float* qvel, const float* ctrl,
                         const float* mocap, double time, const float* warmstart, float* qacc, float* residual,
                         float* next_qpos, float* next_qvel, float* qM, float* efc_force, int* counts);

/* Batched variant for teacher-forced per-step parity at full planner sizes: B independent (qpos, qvel, ctrl, warm start,
 * absolute time) tuples are each advanced by one mj_step (mjpc/trajectory.cc:158) through the same kernel instance the
 * rollout uses.  The task state is rebased to time0 as for a rollout starting there.  warmstart may be NULL (zeros).
 * Outputs (any may be NULL): qacc [B][nv], next_qpos [B][nq], next_qvel [B][nv], residual [B][nr], cost [B],
 * counts [B][4] = {ncon, nefc, solver iterations, warning}. */
int mjpc_b200_step_batch(mjpc_b200_t* h, int B, const float* qpos, const float* qvel, const float* ctrl,
                         const float* warmstart, const float* mocap, double time0, const double* times, float* qacc,
                         float* next_qpos, float* next_qvel, float* residual, float* cost, int* counts);

/* Per-candidate execution statistics of the last rollout, stats [N][12] = {SM cycles, Newton iterations, contacts,
 * constraint rows (summed over steps), 8 per-phase cycle counters (zero unless built with -DMJPC_PHASE_TIMING)}. */
int mjpc_b200_fetch_stats(mjpc_b200_t* h, int64_t* stats);

/* Number of CUDA kernels this handle has launched so far (bench.py reports it as gpu_launches). */
int64_t mjpc_b200_launch_count(const mjpc_b200_t* h);
/* Device time (ms, CUDA events on the engine's stream) of the kernels of the last call. */
float mjpc_b200_last_kernel_ms(const mjpc_b200_t* h);
/* Non-zero if the last rollout launch used a statically specialised kernel instance (model == a shipped task model,
 * csrc/spec_*.h): 1 = the shipped instance (one CTA per candidate: main warp + Hessian helper warps + task warp),
 * 2 = its one-warp-per-candidate twin (same source, selected only by MJPC_B200_SHAPE=plain: the bitwise reference of
 * the tests and the baseline of the profiles); 0 = the generic kernel (MJPC_B200_NO_STATIC=1 forces it).
 * MJPC_B200_PAIR_SYNC=0 disables the step-by-step synchronisation of the two candidates that share an SM when
 * #SMs < N <= 2 #SMs (a scheduling aid: it never changes a result). */
int mjpc_b200_last_kernel_static(const mjpc_b200_t* h);
/* Host-only: header + state-layout words of a model ({n_model, n_layout, model words, layout offsets}); what
 * mujoco_mpc_b200/gen_spec.py writes into csrc/spec_*.h.  Returns the number of ints written or <0. */
int mjpc_b200_spec_words(const mjpc_model_blob* model, int* out, int capacity);

/* Resident-input path used for the device-timed bench value: upload once, then launch repeatedly. */
int mjpc_b200_upload_spline_inputs(mjpc_b200_t* h, const float* state, double time, const float* mocap,
                                   const float* userdata, const float* knots, const double* knot_times, int interp,
                                   int P, int N, int H);
int mjpc_b200_launch_resident(mjpc_b200_t* h);          /* async on the engine stream */
int mjpc_b200_sync(mjpc_b200_t* h);
int mjpc_b200_read_returns(mjpc_b200_t* h, float* returns, uint8_t* failure, int* order);
/* ---- Multi-GPU: ONE planning problem, its candidates sharded over the ranks of an NCCL communicator owned by the
 * handle (one process per GPU).  Rank g owns the contiguous candidate range [g*N/G, (g+1)*N/G) (the first N % G ranks
 * one more); candidate 0, the un-noised nominal (sampling/planner.cc:374), lives on rank 0.  The single exchange per
 * planning iteration - per-candidate returns + failure flags - is one ncclAllGather enqueued on the engine stream
 * behind the rollout kernel; ranking runs on the device on the gathered vector, so every rank sees the same
 * returns / failure / order for all N candidates (north_star: "a single NCCL all-reduce of per-candidate returns").
 * NCCL is bound with dlopen("libnccl.so.2") at the first call; without it these return MJPC_B200_ERR_UNSUPPORTED.
 *   comm_unique_id: rank 0 generates the 128-byte ncclUniqueId, the caller distributes it (MPI / torch.distributed / file)
 *   comm_init:      collective over all ranks (ncclCommInitRank)                                                     */
int mjpc_b200_comm_unique_id(void* out, size_t nbytes);
int mjpc_b200_comm_init(mjpc_b200_t* h, int nranks, int rank, const void* unique_id, size_t nbytes);
int mjpc_b200_comm_info(const mjpc_b200_t* h, int* nranks, int* rank);
/* Same arguments on every rank (knots [N][P][nu] for ALL candidates; inputs are replicated, a few KB).  N may be up to
 * nranks * max_candidates.  returns [N], failure [N], order [N] are global and identical on every rank. */
int mjpc_b200_rollout_spline_sharded(mjpc_b200_t* h, const float* state, double time, const float* mocap,
                                     const float* userdata, const float* knots, const double* knot_times, int interp,
                                     int P, int N, int H, float* returns, uint8_t* failure, int* order);
/* Trajectory of GLOBAL candidate index on every rank (ncclBroadcast from its owner); collective. */
int mjpc_b200_fetch_trajectory_sharded(mjpc_b200_t* h, int candidate, float* states, float* actions, double* times,
                                       float* residual, float* costs, float* trace);

/* Raw stream / device pointers for multi-GPU plumbing (NCCL all-gather of returns runs on this stream). */
void* mjpc_b200_stream(mjpc_b200_t* h);
float* mjpc_b200_device_returns(mjpc_b200_t* h);

/* ---- C++ host layer above the ABI (csrc/host/sampling_planner.{h,cc}): SamplingPlanner with the reference's
 * method names (mjpc/planners/sampling/planner.h:40-160); these C wrappers are what ctypes / a test harness binds.
 * mjpc_b200_host_spline_sample = TimeSpline::Sample (mjpc/spline/spline.cc:103-156), usable without a GPU. */
void mjpc_b200_host_spline_sample(const double* times, const double* values, int P, int dim, int interp, double t,
                                  double* out);
double mjpc_b200_host_philox_normal(uint32_t seed, uint32_t iteration, uint32_t candidate, uint32_t knot, uint32_t dof);
int mjpc_b200_planner_create(const mjpc_model_blob* model, int num_trajectory, int num_spline_points, int interpolation,
                             double exploration, double timestep, const double* ctrlrange, uint32_t seed,
                             int max_horizon, int device, void** out);
void mjpc_b200_planner_destroy(void* planner);
/* noise_exploration[0..1] (sampling/planner.cc:85-88, 334-338): exploration2 > 0 replaces the std with probability 0.2 */
void mjpc_b200_planner_set_exploration(void* planner, double exploration, double exploration2);
void mjpc_b200_planner_reset(void* planner, int horizon, const double* initial_repeated_action);
void mjpc_b200_planner_set_state(void* planner, const double* state, double time, const double* mocap);
int mjpc_b200_planner_optimize_policy(void* planner, int horizon);          /* SamplingPlanner::OptimizePolicy */
void mjpc_b200_planner_action_from_policy(void* planner, double* action, double time, int use_previous);
int mjpc_b200_planner_get_result(void* planner, int* winner, double* improvement, float* returns, double* knots,
                                 double* knot_times);

/* ---- Batched Predictive Sampling (csrc/host/batch_sampling_planner.{h,cc}): num_agents independent SamplingPlanners
 * (agent p seeded with seeds[p]) on ONE engine handle.  Every agent has its own policy, previous policy, iteration
 * counter, state, time, mocap and task snapshot (initially the model's; set_task's NULL members keep the agent's value,
 * its risk applies to all agents).  optimize_policy makes each agent's candidates as the single planner does, rolls all
 * of them out with ONE mjpc_b200_rollout_spline_batched launch and installs each agent's winner: agent p's results are
 * bit for bit those of a single planner with seed seeds[p] and the same inputs.  The per-agent calls take an agent index
 * in [0, num_agents). */
int mjpc_b200_batch_planner_create(const mjpc_model_blob* model, int num_agents, const uint32_t* seeds, int num_trajectory,
                                   int num_spline_points, int interpolation, double exploration, double timestep,
                                   const double* ctrlrange, int max_horizon, int device, void** out);
void mjpc_b200_batch_planner_destroy(void* planner);
void mjpc_b200_batch_planner_reset(void* planner, int agent, int horizon, const double* initial_repeated_action);
void mjpc_b200_batch_planner_set_state(void* planner, int agent, const double* state, double time, const double* mocap);
int mjpc_b200_batch_planner_set_task(void* planner, int agent, const mjpc_task_desc* task);
int mjpc_b200_batch_planner_optimize_policy(void* planner, int horizon);    /* all agents, one launch; 0 or -1 */
void mjpc_b200_batch_planner_action_from_policy(void* planner, int agent, double* action, double time, int use_previous);
/* as mjpc_b200_planner_get_result, for one agent */
int mjpc_b200_batch_planner_get_result(void* planner, int agent, int* winner, double* improvement, float* returns,
                                       double* knots, double* knot_times);

/* ---- Cross-Entropy planner (csrc/host/cross_entropy_planner.{h,cc}; mjpc/planners/cross_entropy/planner.h:35-146).
 * One rollout launch covers the N noisy candidates and the un-noised nominal (candidate N); the elite mean and
 * variance are host arithmetic in double, as in the reference (planner.cc:201-262).  n_elite <= 0 selects the
 * reference default max(N/10, 2). */
int mjpc_b200_ce_planner_create(const mjpc_model_blob* model, int num_trajectory, int n_elite, int num_spline_points,
                                int interpolation, double std_initial, double std_min, double explore_fraction,
                                double timestep, const double* ctrlrange, uint32_t seed, int max_horizon, int device,
                                void** out);
void mjpc_b200_ce_planner_destroy(void* planner);
void mjpc_b200_ce_planner_reset(void* planner, int horizon, const double* initial_repeated_action);
void mjpc_b200_ce_planner_set_state(void* planner, const double* state, double time, const double* mocap);
int mjpc_b200_ce_planner_optimize_policy(void* planner, int horizon);       /* CrossEntropyPlanner::OptimizePolicy */
void mjpc_b200_ce_planner_action_from_policy(void* planner, double* action, double time, int use_previous);
/* improvement, returns [N+1] (last = nominal), elite order [N], installed knots [P][nu] / times [P], variance [P][nu];
 * returns the number of spline points */
int mjpc_b200_ce_planner_get_result(void* planner, double* improvement, float* returns, int* order, double* knots,
                                    double* knot_times, double* variance);

/* ---- Robust planner (csrc/host/robust_planner.{h,cc}; mjpc/planners/robust/robust_planner.cc:40-160) over the
 * sampling planner: the best `ncandidates` of the clean launch are re-rolled `nrepetitions` times each with
 * NoisyRollout force perturbations (one launch on a second handle) and the best mean score is installed.
 * ncandidates = -1 -> num_trajectory / nrepetitions, nrepetitions <= 0 -> 5 (the reference's defaults). */
int mjpc_b200_robust_planner_create(const mjpc_model_blob* model, int num_trajectory, int num_spline_points,
                                    int interpolation, double exploration, double timestep, const double* ctrlrange,
                                    uint32_t seed, int ncandidates, int nrepetitions, double xfrc_std, double xfrc_rate,
                                    int max_horizon, int device, void** out);
void mjpc_b200_robust_planner_destroy(void* planner);
void mjpc_b200_robust_planner_reset(void* planner, int horizon, const double* initial_repeated_action);
void mjpc_b200_robust_planner_set_state(void* planner, const double* state, double time, const double* mocap);
int mjpc_b200_robust_planner_optimize_policy(void* planner, int horizon);
void mjpc_b200_robust_planner_action_from_policy(void* planner, double* action, double time, int use_previous);
/* winner, robust scores [ncandidates], clean returns [num_trajectory], installed knots/times; returns #scores */
int mjpc_b200_robust_planner_get_result(void* planner, int* winner, double* scores, float* returns, double* knots,
                                        double* knot_times);

/* ---- Task::Transition of the config tasks on the host (csrc/host/task_transition.{h,cc}): the state machines that
 * produce the task-state block the kernels consume (QuadrupedFlat::TransitionLocked quadruped.cc:228-395,
 * Tracking::TransitionLocked tracking.cc:218-267).  Host only - no device, no handle.
 * quadruped ids[14] = {p_gait, p_gait_switch, p_cadence, p_amplitude, p_duty, p_walk_speed, p_walk_turn,
 *                      w_upright, w_height, w_position, w_gait, w_balance, w_effort, w_posture};
 * view[24] = {time, torso_subtreelinvel[3], torso_xmat[9], torso_xpos[3], torso_xquat[4], head_site_xpos[3],
 *             ground height under the torso subtree com (read when the Flip mode starts)}. */
void* mjpc_b200_quadruped_transition_create(const int* ids, const double* parameters, int nparam, const double* weight,
                                            int nweight, const double* task_state, int nstate, const double* goal_pos);
void mjpc_b200_quadruped_transition_destroy(void* transition);
/* caller / GUI edits of Task::parameters and Task::weight between transitions (either may be NULL) */
void mjpc_b200_quadruped_transition_set(void* transition, const double* parameters, const double* weight);
void mjpc_b200_quadruped_transition_step(void* transition, int* mode_inout, const double* view, double* parameters,
                                         double* weight, double* task_state, double* goal_pos);
void* mjpc_b200_track_transition_create(int nq, int nv, int nmocap, int nkey, const double* key_qpos,
                                        const double* key_qvel, const double* key_mpos);
void mjpc_b200_track_transition_destroy(void* transition);
void mjpc_b200_track_transition_step(void* transition, int mode, double time, double* qpos, double* qvel,
                                     double* mocap_pos, double* task_state);

/* ShadowReorient::TransitionLocked (hand.cc:90-119): cube at rest on the floor -> back into the hand.  Returns 1 on a reset. */
void* mjpc_b200_shadow_transition_create(int cube_qposadr, int cube_dofadr, const double* qpos0_cube /*[7]*/);
void mjpc_b200_shadow_transition_destroy(void* transition);
int mjpc_b200_shadow_transition_step(void* transition, double* qpos, double* qvel, int on_floor, const double* cube_linvel);

/* ---- iLQG planner (csrc/host/ilqg_planner.{h,cc}; mjpc/planners/ilqg/planner.h, planner.cc:156-740).
 * OptimizePolicy = NominalTrajectory (feedback-scaling line search) + Iteration (model derivatives, cost derivatives,
 * backward pass with the regularisation retry loop, K action rollouts, winner, regularisation update); each sweep is
 * one call of the ABI above.  Returns 1 when the policy was updated, 0 when the iteration was rejected, <0 on error. */
int mjpc_b200_ilqg_planner_create(const mjpc_model_blob* model, int num_rollouts, int representation, double fd_tolerance,
                                  int max_horizon, int device, void** out);
void mjpc_b200_ilqg_planner_destroy(void* planner);
/* finite-difference settings (ilqg/settings.h:23-24, iLQGPlanner::derivative_skip_): tolerance <= 0 / mode < 0 / skip < 0 keep
 * the current value.  Defaults here: 3e-4, centred, 0 - the reference's 1e-6 one-sided is an fp64 setting (ilqg_planner.h). */
void mjpc_b200_ilqg_planner_set_fd(void* planner, double tolerance, int mode, int derivative_skip);
void mjpc_b200_ilqg_planner_reset(void* planner, int horizon, const double* initial_repeated_action);
void mjpc_b200_ilqg_planner_set_state(void* planner, const double* state, double time, const double* mocap);
int mjpc_b200_ilqg_planner_nominal_trajectory(void* planner, int horizon);
int mjpc_b200_ilqg_planner_optimize_policy(void* planner, int horizon);
/* iLQGPolicy::Action (ilqg/policy.cc:82-161): state may be NULL (open loop), otherwise the time-varying feedback
 * feedback_scaling * K (state (-) x_nominal) is added before clamping */
void mjpc_b200_ilqg_planner_action_from_policy(void* planner, double* action, const double* state, double time);
/* the same, stateless and host only: u_nom [H][nu], x_nom [H][dim_state], t_nom [H], gains [H][nu][2 nv] */
int mjpc_b200_host_ilqg_policy_action(const mjpc_model_blob* model, const float* u_nom, const float* x_nom,
                                      const double* t_nom, const float* gains, int horizon, int representation,
                                      double feedback_scaling, const double* state, double time, double* action);
/* scalars[6] = {total_return, regularization, improvement, expected, surprise, winner}; nominal states [H][dim_state],
 * actions [H][nu], times [H] (any pointer may be NULL); returns H */
int mjpc_b200_ilqg_planner_get_result(void* planner, double* scalars, float* states, float* actions, double* times);

/* ---- Gradient planner (csrc/host/gradient_planner.{h,cc}; mjpc/planners/gradient/planner.cc:159-383, gradient.cc:44-107,
 * spline_mapping.cc): ResamplePolicy, nominal rollout, {model derivatives, cost derivatives, gradient sweep, total derivative
 * through the spline mapping, K line-search rollouts (ONE mjpc_b200_rollout_spline launch)} x max_rollout.
 * optimize_policy returns 1 when the return improved, 0 when the nominal was kept, <0 on error. */
int mjpc_b200_gradient_planner_create(const mjpc_model_blob* model, int num_trajectory, int num_spline_points, int representation,
                                      double fd_tolerance, double timestep, const double* ctrlrange, int max_horizon, int device,
                                      void** out);
void mjpc_b200_gradient_planner_destroy(void* planner);
void mjpc_b200_gradient_planner_set_fd(void* planner, double tolerance, int mode, int derivative_skip);   /* as for the iLQG planner */
void mjpc_b200_gradient_planner_reset(void* planner, int horizon, const double* initial_repeated_action);
void mjpc_b200_gradient_planner_set_state(void* planner, const double* state, double time, const double* mocap);
int mjpc_b200_gradient_planner_optimize_policy(void* planner, int horizon);
void mjpc_b200_gradient_planner_action_from_policy(void* planner, double* action, double time, int use_previous);
/* scalars[6] = {total_return, winner, action_step, expected, improvement, surprise}; parameters [P][nu], times [P] */
int mjpc_b200_gradient_planner_get_result(void* planner, double* scalars, double* parameters, double* times);
/* SplineMapping::Compute (gradient/spline_mapping.cc) as scalar weights W [num_output][num_input]; host only */
void mjpc_b200_host_spline_mapping(int representation, const double* input_times, int num_input, const double* output_times,
                                   int num_output, double* W);

/* ---- iLQS planner (csrc/host/gradient_planner.{h,cc}; mjpc/planners/ilqs/planner.cc:87-215): Predictive Sampling first;
 * when it does not improve, one iLQG iteration seeded with the sampling nominal; when sampling follows iLQG the trajectory
 * policy is converted to spline parameters through the least-squares inverse of the spline mapping. */
int mjpc_b200_ilqs_planner_create(const mjpc_model_blob* model, int num_trajectory, int num_spline_points, int interpolation,
                                  double exploration, double timestep, const double* ctrlrange, uint32_t seed,
                                  int ilqg_num_rollouts, int ilqg_representation, double fd_tolerance, int max_horizon, int device,
                                  void** out);
void mjpc_b200_ilqs_planner_destroy(void* planner);
void mjpc_b200_ilqs_planner_set_fd(void* planner, double tolerance, int mode, int derivative_skip);       /* its iLQG half */
void mjpc_b200_ilqs_planner_reset(void* planner, int horizon, const double* initial_repeated_action);
void mjpc_b200_ilqs_planner_set_state(void* planner, const double* state, double time, const double* mocap);
void mjpc_b200_ilqs_planner_set_exploration(void* planner, double exploration);
int mjpc_b200_ilqs_planner_optimize_policy(void* planner, int horizon);
void mjpc_b200_ilqs_planner_action_from_policy(void* planner, double* action, const double* state, double time, int use_previous);
/* scalars[4] = {active_policy (0 sampling, 1 iLQG), sampling winner return, iLQG total_return, sampling winner}; returns active_policy */
int mjpc_b200_ilqs_planner_get_result(void* planner, double* scalars);

/* ---- Agent::PlanIteration glue (csrc/host/agent.{h,cc}; mjpc/agent.cc:85-107,150-164,283-357): owns the planner selected
 * by agent_planner (0 Sampling, 1 Gradient, 2 iLQG, 3 iLQS, 4 Robust, 5 Cross-Entropy; mjpc/planners/include.h:26-34) and does
 * per iteration what the reference does around OptimizePolicy: steps_ = int(max(min(horizon / timestep + 1, 512), 1)),
 * timestep / integrator override, MakeDifferentiable for gradient-based planners (restored afterwards), SetState, the
 * residual snapshot (set_task on every engine handle of the planner), OptimizePolicy(steps_) - or NominalTrajectory when
 * planning is disabled.
 * settings[20] = {planner, horizon, timestep, integrator, differentiable (-1 = the reference default), num_trajectory,
 *   num_spline_points, representation, exploration, ilqg_num_rollouts, ilqg_representation, fd_tolerance, n_elite, std_min,
 *   explore_fraction, robust_candidates, robust_repetitions, robust_xfrc, robust_xfrc_rate, seed} */
int mjpc_b200_agent_steps(double horizon, double timestep);
int mjpc_b200_agent_create(const mjpc_model_blob* model, const double* settings, const double* ctrlrange, int device, void** out);
void mjpc_b200_agent_destroy(void* agent);
void mjpc_b200_agent_reset(void* agent, const double* initial_repeated_action);
void mjpc_b200_agent_set_state(void* agent, const double* state, double time, const double* mocap);
void mjpc_b200_agent_set_task(void* agent, const mjpc_task_desc* task);
void mjpc_b200_agent_set_plan_enabled(void* agent, int on);
int mjpc_b200_agent_plan_iteration(void* agent);
int mjpc_b200_agent_get_steps(void* agent);
void mjpc_b200_agent_action_from_policy(void* agent, double* action, const double* state, double time, int use_previous);

#ifdef __cplusplus
}
#endif
#endif /* MJPC_B200_H_ */
