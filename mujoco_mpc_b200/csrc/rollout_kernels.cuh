// rollout_kernels.cuh - the CUDA kernels of the hot path (sm_100a).
//
//   rollout_kernel      one candidate trajectory per warp (generic) or per CTA of main + helper warps (static instances)
//                       (Trajectory::Rollout / RolloutDiscrete,
//                       mjpc/trajectory.cc:92-309) incl. policy, mj_step restatement, residual, cost, return
//   rank_kernel         order of candidates by return (partial_sort, sampling/planner.cc:184-188)
//   *_batched           the rollout instances for M independent problems in one launch (rollout_body<SP, true>),
//   rank_batched_kernel   ranked per problem (DESIGN.md section 6a)
//   step_debug_kernel   a single forward+Euler step through the same device functions (parity hook)
//   fd_*_kernel         finite-difference transition/residual Jacobians (model_derivatives.cc:45-165)
//
// Shared memory per CTA: [model pack (floats | ints)] [warp 0 data] [warp 1 data] ...
// The model pack is staged with ONE 1-D TMA bulk copy (cp.async.bulk -> SASS UBLKCP) signalled on an mbarrier.
// Trajectory outputs are written time-major per candidate with lane-strided (coalesced) stores.
#pragma once
#include "dev_physics.cuh"
#include "dev_task.cuh"
#include "spec_quadruped.h"
#include "spec_humanoid_track.h"

namespace mjpc_dev {

struct RolloutArgs {
  DevModel M;
  DevLayout L;
  const float* pack;        // device: nf floats followed by ni ints
  const float* state;       // [dim_state]
  const float* mocap;       // [7*nmocap]
  const float* task_state;  // [task_state_size] (times rebased to the rollout start) or nullptr
  const float* knots;       // [N][P][nu]
  const float* knot_times;  // [P], relative
  FeedbackArgs fb;
  const float* step_sizes;  // [N] for the feedback policy
  int policy_kind;          // 0 spline, 1 feedback
  float xfrc_std, xfrc_rate;   // NoisyRollout (trajectory.cc:100-210): OU force noise, std 0 = off
  unsigned noise_seed;
  int cand0;                // global index of this launch's first candidate (multi-GPU shards): noise stream = cand0 + local index
  int P, interp, N, H;
  double time0;
  float* states; float* actions; double* times; float* residual; float* costs; float* trace;
  float* returns; unsigned char* failure;
  int pair_sync_mode;       // bit 0: meet at every time step, bit 1: also before every constraint solve
  unsigned* pair_sync;      // HBM [256][32] zeroed before the launch, or nullptr: co-resident pair synchronisation (dev_data.cuh)
  long long* stats;         // [N][12]: cycles, Newton iterations, contacts, constraint rows (summed over steps), 8 phase timers
  // batched instances only (rollout_body<SP, true>): `nprob` problems of N candidates each, candidate p*N + i of the launch
  // is candidate i of problem p; state, mocap, task_state and knot_times above then hold one row per problem
  int nprob;
  const double* time0s;          // [nprob] absolute start time of each problem
  const float* task_weight;      // [nprob][num_term]
  const float* task_parameters;  // [nprob][num_parameters]
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// Stage the model pack into shared memory with a TMA bulk copy; all threads of the CTA must call.
__device__ __forceinline__ void stage_model_pack(float* dst, const float* src, unsigned bytes) {
  __shared__ __align__(8) unsigned long long bar;
  const unsigned bar_a = smem_u32(&bar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_a), "r"(1) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(bar_a) : "memory");
  }
  unsigned done = 0;
  while (!done) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done) : "r"(bar_a), "r"(0) : "memory");
  }
  __syncthreads();
}

// shared-memory words taken by the pack + header copies (must match engine.cu smem_bytes)
__host__ __device__ inline int smem_header_words(const DevModel& M) {
  return M.nf + M.ni + (int)((sizeof(DevModel) + 15) / 16) * 4 + (int)((sizeof(DevLayout) + 15) / 16) * 4;
}

// copy the DevModel / DevLayout kernel parameters behind the pack and set up this warp's context
__device__ __forceinline__ void init_ctx(Ctx& c, const DevModel* M, const DevLayout* L, float* smem, int warp, int lane,
                                         const float* pack) {
  const int hdr = M->nf + M->ni;
  const int lay = hdr + (int)((sizeof(DevModel) + 15) / 16) * 4;
  const int data0 = lay + (int)((sizeof(DevLayout) + 15) / 16) * 4;
  {
    const int* srcM = reinterpret_cast<const int*>(M);
    const int* srcL = reinterpret_cast<const int*>(L);
    int* dst = reinterpret_cast<int*>(smem);
    for (int i = threadIdx.x; i < (int)(sizeof(DevModel) / 4); i += blockDim.x) dst[hdr + i] = srcM[i];
    for (int i = threadIdx.x; i < (int)(sizeof(DevLayout) / 4); i += blockDim.x) dst[lay + i] = srcL[i];
  }
  __syncthreads();
  c.hdr = hdr; c.lay = lay; c.ibase = M->nf;
  c.dbase = data0 + warp * L->total;
  c.lane = lane;
  c.gkey = pack + M->nf + M->ni;   // the keyframe table follows the staged part of the pack in HBM
  c.ncon = 0; c.npseudo = 0; c.xfrc_on = 0; c.nefc = 0; c.ndrow = 0; c.nitem = 0; c.niter = 0; c.nlim = 0; c.warn = 0; c.time = 0.f;
  c.sync = nullptr; c.sync_slot = -1; c.sync_mode = 0;
#ifdef MJPC_PHASE_TIMING
  for (int k = 0; k < 8; k++) c.tph[k] = 0;
  c.tlast = clock64();
#endif
}

// write the trace points (GetTraces, mjpc/utilities.cc:268-285)
template <class SP>
__device__ __forceinline__ void write_traces(Ctx& c, float* out) {
  auto&& M = SP::model(c);
  const int *ty = MI(task_trace_objtype), *id = MI(task_trace_objid);
  for (int w = c.lane; w < 3 * M.num_trace; w += 32) {
    const int k = w / 3, q = w - 3 * k;
    const float* src = ty[k] == OBJ_SITE ? DF(site_xpos) : ty[k] == OBJ_GEOM ? DF(geom_xpos) : ty[k] == OBJ_XBODY ? DF(xpos) : DF(xipos);
    out[w] = src[3 * id[k] + q];
  }
}

// Injected noise of NoisyRollout: Philox4x32-10, key (seed, 1), counter (step, stream, element, 'XFRC'), Box-Muller on
// the first two words - the definition of oracle/rollout.h (xfrc_normal), evaluated in fp32 here.
__device__ __forceinline__ float xfrc_normal(unsigned seed, unsigned step, unsigned stream, unsigned element) {
  unsigned c0 = step, c1 = stream, c2 = element, c3 = 0x58465243u, k0 = seed, k1 = 1u;
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  const float u1 = ((float)c0 + 0.5f) * 2.3283064365386963e-10f, u2 = ((float)c1 + 0.5f) * 2.3283064365386963e-10f;
  return sqrtf(-2.0f * logf(fmaxf(u1, 1e-12f))) * cospif(2.0f * u2);
}

// The task warp of a rollout CTA (StaticSpec<K, W, 1>): per step, between the main warp's fork / join barriers,
//   fork .. join 1 : composite inertia, velocities, smooth forces  (main: collision + constraint rows)
//   join 1 .. join 2: residual, trace, cost, the next step's spline action  (main: reference + Newton solve)
// None of these reads anything the main warp writes in the same interval (the arrays are listed per function in
// DESIGN.md section 5); every value is computed by the same code on the same inputs as in the one-warp order.
template <class SP>
__device__ __noinline__ void task_warp_loop(Ctx& c, const RolloutArgs& A, int cand) {
  auto&& M = SP::model(c);
  const int lane = c.lane, nu = M.nu, nr = M.num_residual, ntr = 3 * M.num_trace, H = A.H;
  (void)nu;
  c.xfrc_on = A.xfrc_std > 0.f ? 1 : 0;
  float* o_res = A.residual + (size_t)cand * H * nr;
  float* o_trace = A.trace + (size_t)cand * H * ntr;
  for (int t = 0; t < H; t++) {
    const bool last = t == H - 1;
    task_bar();   // fork (the main warp has written the state, the action and the poses of step t)
    if (wide_box().task_exit) return;
    k_crb<SP>(c);
    k_com_vel<SP>(c);
    k_smooth_forces<SP>(c);
    task_bar();   // join 1
    k_residual<SP>(c);
    for (int i = lane; i < nr; i += 32) o_res[(size_t)t * nr + i] = DF(residual)[i];
    write_traces<SP>(c, o_trace + (size_t)t * ntr);
    const float cost = k_cost_value<SP>(c);
    if (lane == 0) { wide_box().task_cost = cost; wide_box().task_warn = c.warn; }   // (a residual can raise a warning)
    if (!last) {
      c.time += CM(c).timestep;   // the same sum k_euler forms on the main warp
      if (A.policy_kind == 0 && t + 1 < H - 1) k_policy_spline<SP>(c, A.P, A.interp);
    }
    task_bar();   // join 2
  }
}

// kBatch: A.nprob independent problems in one launch.  A CTA never spans two problems (the grid holds ceil(N / candidates
// per CTA) CTAs per problem), so the per-CTA shared-memory copies of the task weights, parameters and state can be
// overwritten with the problem's rows before the task warp forks.  Outputs are indexed by the launch-wide candidate p*N + i;
// the xfrc noise stream uses the problem-local index i, so every problem computes what a launch of that problem alone does.
template <class SP, bool kBatch = false>
__device__ __forceinline__ void rollout_body(const RolloutArgs& A) {
  float* smem = g_smem;
  stage_model_pack(smem, A.pack, (unsigned)((A.M.nf + A.M.ni) * 4));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // SP::kWide > 1: the whole CTA is ONE candidate (warp 0 runs the pipeline, the others help with the wide phases)
  constexpr bool kCtaPerCand = SP::kWide > 1 || SP::kTask > 0;
  int cand = kCtaPerCand ? (int)blockIdx.x : blockIdx.x * (blockDim.x >> 5) + warp;
  int prob = 0, local = cand;   // problem and problem-local candidate (batched instances)
  if constexpr (kBatch) {
    const int per_cta = kCtaPerCand ? 1 : (int)(blockDim.x >> 5);
    const int ctas = (A.N + per_cta - 1) / per_cta;   // CTAs per problem
    prob = (int)blockIdx.x / ctas;
    local = ((int)blockIdx.x - prob * ctas) * per_cta + (kCtaPerCand ? 0 : warp);
    cand = prob * A.N + local;
  }
  Ctx c;
  init_ctx(c, &A.M, &A.L, smem, kCtaPerCand ? 0 : warp, lane, A.pack);
  if (local >= A.N) return;
  if (SP::kWide > 1 && warp > 0 && warp < SP::kWide) { wide_helper_loop<SP>(c); return; }
  if (SP::kTask > 0 && warp == SP::kWide) { task_warp_loop<SP>(c, A, cand); return; }
  constexpr bool kTask = SP::kTask > 0;
  if (kTask && lane == 0) wide_box().task_exit = 0;
  if constexpr (SP::kWide > 1) pair_sync_init(c, A.pair_sync, A.pair_sync_mode);
  auto&& M = SP::model(c);
  const int nq = M.nq, nv = M.nv, nu = M.nu, ds = nq + nv, nr = M.num_residual, ntr = 3 * M.num_trace, H = A.H;
  // this problem's row of a per-problem input (the single-problem instances read the argument itself at every use)
#define ROW(field, width) (kBatch ? A.field + (size_t)prob * (width) : A.field)
#define TIME0 (kBatch ? A.time0s[prob] : A.time0)
  // per-iteration task state (time-rebased) overrides the packed copy: the pack in shared memory is per CTA,
  // every warp writes the same values
  if (A.task_state) {
    float* ts = const_cast<float*>(MF(task_state));
    for (int i = lane; i < M.task_state_size; i += 32) ts[i] = ROW(task_state, M.task_state_size)[i];
  }
  if constexpr (kBatch) {   // ... and so do the problem's task weights and parameters
    float* w = const_cast<float*>(MF(task_weight));
    float* prm = const_cast<float*>(MF(task_parameters));
    for (int i = lane; i < M.num_term; i += 32) w[i] = A.task_weight[(size_t)prob * M.num_term + i];
    for (int i = lane; i < M.num_parameters; i += 32) prm[i] = A.task_parameters[(size_t)prob * M.num_parameters + i];
  }
  // ---- initial conditions (trajectory.cc:108-137)
  for (int i = lane; i < nq; i += 32) DF(qpos)[i] = ROW(state, ds)[i];
  for (int i = lane; i < nv; i += 32) { DF(qvel)[i] = ROW(state, ds)[nq + i]; DF(qacc_warmstart)[i] = 0; }
  for (int i = lane; i < 7 * M.nmocap; i += 32) {
    const int k = i / 7, q = i - 7 * k;
    if (q < 3) DF(mocap_pos)[3 * k + q] = ROW(mocap, 7 * M.nmocap)[i]; else DF(mocap_quat)[4 * k + q - 3] = ROW(mocap, 7 * M.nmocap)[i];
  }
  for (int i = lane; i < nv * nv; i += 32) DF(qM)[i] = 0;
  const bool noisy = A.xfrc_std > 0.f;
  const float ou_rate = noisy ? expf(-CM(c).timestep / A.xfrc_rate) : 0.f;
  const float ou_scale = noisy ? A.xfrc_std * sqrtf(1.f - ou_rate * ou_rate) : 0.f;
  for (int i = lane; i < 6 * M.nbody; i += 32) DF(xfrc)[i] = 0;
  c.xfrc_on = noisy ? 1 : 0;
  float step_size = 0.f;
  if (A.policy_kind == 0) {
    for (int i = lane; i < A.P * nu; i += 32) DF(knots)[i] = A.knots[(size_t)cand * A.P * nu + i];
    for (int i = lane; i < A.P; i += 32) DF(knot_times)[i] = ROW(knot_times, A.P)[i];
  } else {
    step_size = A.step_sizes[cand];
  }
  __syncwarp();
  float* o_states = A.states + (size_t)cand * H * ds;
  float* o_actions = A.actions + (size_t)cand * H * nu;
  double* o_times = A.times + (size_t)cand * H;
  float* o_res = A.residual + (size_t)cand * H * nr;
  float* o_costs = A.costs + (size_t)cand * H;
  float* o_trace = A.trace + (size_t)cand * H * ntr;
  for (int i = lane; i < ds; i += 32) o_states[i] = ROW(state, ds)[i];
  if (lane == 0) o_times[0] = TIME0;
  float total = 0.f;
  bool failed = false;
  const long long clk0 = clock64();
  long long n_newton = 0, n_con = 0, n_efc = 0;
  for (int t = 0; t < H; t++) {
    const bool last = t == H - 1;
    if ((c.sync_mode & 1) && (t & (c.sync_mode >> 4)) == 0) pair_sync_meet(c, 2 * t);   // bits 4..: step mask (0 = every step)
    // (with a task warp the spline action of step t > 0 was evaluated by it during step t-1's constraint solve)
    if (!last) {
      if (A.policy_kind == 0) { if (!kTask || t == 0) k_policy_spline<SP>(c, A.P, A.interp); }
      else k_policy_feedback<SP>(c, A.fb, step_size, t);
    }
    // action record (the last row repeats the previous action; H == 1 -> zeros; trajectory.cc:190-196)
    for (int i = lane; i < nu; i += 32) {
      if (H == 1) DF(ctrl)[i] = 0;
      o_actions[(size_t)t * nu + i] = DF(ctrl)[i];
    }
    if (!last && (k_bad(c, DF(qpos), nq) || k_bad(c, DF(qvel), nv))) {
      failed = true;
      if (kTask) { if (lane == 0) wide_box().task_exit = 1; task_bar(); }   // the task warp waits at the fork
      break;
    }
    if (noisy && !last) {   // Ornstein-Uhlenbeck perturbation in discrete time (trajectory.cc:147-155)
      float* xf = DF(xfrc);
      for (int i = lane; i < 6 * M.nbody; i += 32)
        xf[i] = ou_rate * xf[i] + ou_scale * xfrc_normal(A.noise_seed, (unsigned)t, (unsigned)(A.cand0 + local), (unsigned)i);
      __syncwarp();
    }
    float cost;
    if constexpr (kTask) {
      // the step as a fork / join graph (the one-warp order is k_forward, dev_physics.cuh):
      //   main: kinematics, com | collision, constraint rows        | reference, Newton solve           | Euler
      //   task:                 | CRB, velocities, smooth forces    | residual, cost, next spline action |
      PHASE(c, 7);
      k_kinematics<SP>(c);
      k_com_pos<SP>(c);
      PHASE(c, 0);
      task_bar();   // fork
      k_collision<SP>(c);
      PHASE(c, 1);
      k_make_constraint<SP>(c);
      PHASE(c, 2);
      task_bar();   // join: qM, qfrc_smooth, qacc_smooth are in place
      k_reference<SP>(c);
      PHASE(c, 3);
      if (c.sync_mode & 2) pair_sync_meet(c, 2 * t + 1);
      k_solve<SP>(c);
      PHASE(c, 4);
      n_newton += c.niter; n_con += c.ncon - c.npseudo; n_efc += c.nefc;
      if (!last && k_bad(c, DF(qacc), nv)) c.warn = 1;
      task_bar();   // join: residual, trace and cost of this step are written, ctrl holds the next action
      cost = wide_box().task_cost;
      if (wide_box().task_warn) c.warn = 1;
    } else {
      k_forward<SP>(c);
      n_newton += c.niter; n_con += c.ncon - c.npseudo; n_efc += c.nefc;
      k_residual<SP>(c);
      if (!last && k_bad(c, DF(qacc), nv)) c.warn = 1;
      for (int i = lane; i < nr; i += 32) o_res[(size_t)t * nr + i] = DF(residual)[i];
      write_traces<SP>(c, o_trace + (size_t)t * ntr);
    }
    if (c.warn) {
      failed = true;
      if (kTask && !last) { if (lane == 0) wide_box().task_exit = 1; task_bar(); }
      break;
    }
    if constexpr (!kTask) cost = k_cost_value<SP>(c);
    if (lane == 0) o_costs[t] = cost;
    total += cost;
    if (last) break;
    for (int i = lane; i < nv; i += 32) DF(qacc_warmstart)[i] = DF(qacc)[i];
    k_euler<SP>(c);
    for (int i = lane; i < nq; i += 32) o_states[(size_t)(t + 1) * ds + i] = DF(qpos)[i];
    for (int i = lane; i < nv; i += 32) o_states[(size_t)(t + 1) * ds + nq + i] = DF(qvel)[i];
    if (lane == 0) o_times[t + 1] = TIME0 + (double)c.time;
  }
  pair_sync_done(c);
  wide_post<SP>(c, WIDE_EXIT);   // releases the helper warps
  if (lane == 0) {
    A.returns[cand] = failed ? 1.0e6f : total / (float)max(H, 1);
    A.failure[cand] = failed ? 1 : 0;
    if (A.stats) {
      A.stats[12 * cand] = clock64() - clk0; A.stats[12 * cand + 1] = n_newton;
      A.stats[12 * cand + 2] = n_con; A.stats[12 * cand + 3] = n_efc;
      for (int k = 0; k < 8; k++) {
#ifdef MJPC_PHASE_TIMING
        A.stats[12 * cand + 4 + k] = c.tph[k];
#else
        A.stats[12 * cand + 4 + k] = 0;
#endif
      }
#ifndef MJPC_PHASE_TIMING
      // placement diagnostics (profiles/placement.py): which SM and which hardware warp slot ran this candidate
      unsigned smid, warpid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      asm volatile("mov.u32 %0, %%warpid;" : "=r"(warpid));
      A.stats[12 * cand + 4] = smid; A.stats[12 * cand + 5] = warpid;
#endif
    }
  }
#undef ROW
#undef TIME0
}

extern "C" __global__ void __launch_bounds__(128) rollout_kernel(const __grid_constant__ RolloutArgs A) {
  rollout_body<DynSpec>(A);
}
// statically specialised instance for the Quadruped (flat) task model (spec_quadruped.h); one warp per CTA
// Static instances: the shipped one holds kRolloutWide + kRolloutTask warps per candidate (main warp, Hessian helper warps,
// task warp: DESIGN.md section 5 "helper warps"; 6 + 1 measured best at 128 and at 256 candidates).  The *_plain instance is
// the same source with ONE warp per candidate: the reference the helper-warp kernel must equal bit for bit
// (tests/test_gpu_parity.py, MJPC_B200_SHAPE=plain) and the baseline of the profiles.
#ifndef MJPC_WIDE
#define MJPC_WIDE 6
#endif
#ifndef MJPC_TASK
#define MJPC_TASK 1
#endif
constexpr int kRolloutWide = MJPC_WIDE, kRolloutTask = MJPC_TASK, kRolloutThreads = 32 * (kRolloutWide + kRolloutTask);
extern "C" __global__ void __launch_bounds__(kRolloutThreads) rollout_kernel_quadruped(const __grid_constant__ RolloutArgs A) {
  rollout_body<StaticSpec<SpecQuadruped, kRolloutWide, kRolloutTask>>(A);
}
extern "C" __global__ void __launch_bounds__(32) rollout_kernel_quadruped_plain(const __grid_constant__ RolloutArgs A) {
  rollout_body<StaticSpec<SpecQuadruped, 1, 0>>(A);
}
// ... and for the Humanoid Track task model (spec_humanoid_track.h)
extern "C" __global__ void __launch_bounds__(kRolloutThreads) rollout_kernel_humanoid_track(const __grid_constant__ RolloutArgs A) {
  rollout_body<StaticSpec<SpecHumanoidTrack, kRolloutWide, kRolloutTask>>(A);
}
extern "C" __global__ void __launch_bounds__(32) rollout_kernel_humanoid_track_plain(const __grid_constant__ RolloutArgs A) {
  rollout_body<StaticSpec<SpecHumanoidTrack, 1, 0>>(A);
}
// Batched twins of the five instances above: A.nprob problems of A.N candidates in one launch (rollout_body<SP, true>).
// Batched<SP> is SP under another name, so the batched kernels get their own copies of the SP-templated non-inlined
// device functions and leave the register allocation of the single-problem kernels' copies exactly as it was.
template <class SP> struct Batched : SP {};
extern "C" __global__ void __launch_bounds__(128) rollout_kernel_batched(const __grid_constant__ RolloutArgs A) {
  rollout_body<Batched<DynSpec>, true>(A);
}
extern "C" __global__ void __launch_bounds__(kRolloutThreads) rollout_kernel_quadruped_batched(const __grid_constant__ RolloutArgs A) {
  rollout_body<Batched<StaticSpec<SpecQuadruped, kRolloutWide, kRolloutTask>>, true>(A);
}
extern "C" __global__ void __launch_bounds__(32) rollout_kernel_quadruped_plain_batched(const __grid_constant__ RolloutArgs A) {
  rollout_body<Batched<StaticSpec<SpecQuadruped, 1, 0>>, true>(A);
}
extern "C" __global__ void __launch_bounds__(kRolloutThreads) rollout_kernel_humanoid_track_batched(const __grid_constant__ RolloutArgs A) {
  rollout_body<Batched<StaticSpec<SpecHumanoidTrack, kRolloutWide, kRolloutTask>>, true>(A);
}
extern "C" __global__ void __launch_bounds__(32) rollout_kernel_humanoid_track_plain_batched(const __grid_constant__ RolloutArgs A) {
  rollout_body<Batched<StaticSpec<SpecHumanoidTrack, 1, 0>>, true>(A);
}

// host: does the live model header / state layout equal the table a static kernel was compiled from?
// (float options are not part of the comparison: static kernels read them from the live header)
template <class K>
inline bool spec_matches(const DevModel& M, const DevLayout& L) {
  if (K::kNumModelWords != (int)(sizeof(DevModel) / 4) || K::kNumLayout != (int)D_COUNT) return false;
  const int* w = K::kModelWords;
#define X(n) if (w[offsetof(DevModel, n) / 4] != M.n) return false;
  MJPC_M_INTS(X)
#undef X
  for (int i = 0; i < F_COUNT; i++) if (w[offsetof(DevModel, fo) / 4 + i] != M.fo[i]) return false;
  for (int i = 0; i < I_COUNT; i++) if (w[offsetof(DevModel, io) / 4 + i] != M.io[i]) return false;
  for (int i = 0; i < D_COUNT; i++) if (K::kLayoutOff[i] != L.off[i]) return false;
  return true;
}

// order[rank] = i, ascending return, ties broken by index
extern "C" __global__ void rank_kernel(const float* __restrict__ ret, int N, int* __restrict__ order) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    const float ri = ret[i];
    int rank = 0;
    for (int j = 0; j < N; j++) {
      const float rj = ret[j];
      rank += (rj < ri) || (rj == ri && j < i) || (ri != ri && rj == rj);
    }
    order[rank] = i;
  }
}

// the same per problem: ret [M][N] -> order [M][N] of problem-local indices (rank_kernel's comparison, NaN last)
extern "C" __global__ void rank_batched_kernel(const float* __restrict__ ret, int M, int N, int* __restrict__ order) {
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < M * N; g += gridDim.x * blockDim.x) {
    const int p = g / N, i = g - p * N;
    const float* r = ret + (size_t)p * N;
    const float ri = r[i];
    int rank = 0;
    for (int j = 0; j < N; j++) {
      const float rj = r[j];
      rank += (rj < ri) || (rj == ri && j < i) || (ri != ri && rj == rj);
    }
    order[(size_t)p * N + rank] = i;
  }
}

struct DebugArgs {
  DevModel M;
  DevLayout L;
  const float* pack;
  const float* qpos; const float* qvel; const float* ctrl; const float* mocap; const float* warmstart;
  const float* task_state;
  float time;
  float* qacc; float* residual; float* next_qpos; float* next_qvel; float* qM; float* efc_force; int* counts;
};

extern "C" __global__ void __launch_bounds__(32) step_debug_kernel(const __grid_constant__ DebugArgs A) {
  using SP = DynSpec;
  extern __shared__ __align__(16) float smem[];
  const DevModel& M = A.M;
  stage_model_pack(smem, A.pack, (unsigned)((M.nf + M.ni) * 4));
  Ctx c;
  init_ctx(c, &A.M, &A.L, smem, 0, threadIdx.x, A.pack);
  const int lane = c.lane, nq = M.nq, nv = M.nv;
  if (A.task_state) {
    float* ts = const_cast<float*>(MF(task_state));
    for (int i = lane; i < M.task_state_size; i += 32) ts[i] = A.task_state[i];
  }
  for (int i = lane; i < nq; i += 32) DF(qpos)[i] = A.qpos[i];
  for (int i = lane; i < nv; i += 32) { DF(qvel)[i] = A.qvel[i]; DF(qacc_warmstart)[i] = A.warmstart ? A.warmstart[i] : 0.f; }
  for (int i = lane; i < M.nu; i += 32) DF(ctrl)[i] = A.ctrl[i];
  for (int i = lane; i < 7 * M.nmocap; i += 32) {
    const int k = i / 7, q = i - 7 * k;
    if (q < 3) DF(mocap_pos)[3 * k + q] = A.mocap[i]; else DF(mocap_quat)[4 * k + q - 3] = A.mocap[i];
  }
  for (int i = lane; i < nv * nv; i += 32) DF(qM)[i] = 0;
  c.time = A.time;
  __syncwarp();
  k_forward<SP>(c);
  k_residual<SP>(c);
  if (k_bad(c, DF(qacc), nv)) c.warn = 1;
  for (int i = lane; i < nv; i += 32) A.qacc[i] = DF(qacc)[i];
  for (int i = lane; i < nv * nv; i += 32) A.qM[i] = DF(qM)[i];
  for (int i = lane; i < M.num_residual; i += 32) A.residual[i] = DF(residual)[i];
  for (int i = lane; i < c.nefc; i += 32) A.efc_force[i] = DF(efc_force)[i];
  if (lane == 0) { A.counts[0] = c.ncon - c.npseudo; A.counts[1] = c.nefc; A.counts[2] = c.niter; A.counts[3] = c.warn; }
  k_euler<SP>(c);
  for (int i = lane; i < nq; i += 32) A.next_qpos[i] = DF(qpos)[i];
  for (int i = lane; i < nv; i += 32) A.next_qvel[i] = DF(qvel)[i];
}


// Batched parity hook: B independent (qpos, qvel, ctrl, warm start, time) tuples, each advanced by ONE mj_step through
// the same device functions - and the same static / generic instances - the rollout kernel runs.  Teacher-forced
// per-step parity tests feed it the oracle's own states, so a mismatch cannot be blamed on trajectory divergence.
struct StepBatchArgs {
  DevModel M;
  DevLayout L;
  const float* pack;
  const float* qpos; const float* qvel; const float* ctrl; const float* warmstart;   // [B][nq|nv|nu|nv]
  const float* mocap; const float* task_state;
  const float* time;    // [B], relative to the rollout start the task state was rebased to
  int B;
  float* qacc; float* next_qpos; float* next_qvel; float* residual; float* cost; int* counts;   // counts [B][4]
};

template <class SP>
__device__ __forceinline__ void step_batch_body(const StepBatchArgs& A) {
  float* smem = g_smem;
  stage_model_pack(smem, A.pack, (unsigned)((A.M.nf + A.M.ni) * 4));
  Ctx c;
  init_ctx(c, &A.M, &A.L, smem, 0, threadIdx.x, A.pack);
  auto&& M = SP::model(c);
  const int lane = c.lane, nq = M.nq, nv = M.nv, nu = M.nu, nr = M.num_residual;
  const int b = blockIdx.x;
  if (b >= A.B) return;
  if (A.task_state) {
    float* ts = const_cast<float*>(MF(task_state));
    for (int i = lane; i < M.task_state_size; i += 32) ts[i] = A.task_state[i];
  }
  for (int i = lane; i < nq; i += 32) DF(qpos)[i] = A.qpos[(size_t)b * nq + i];
  for (int i = lane; i < nv; i += 32) {
    DF(qvel)[i] = A.qvel[(size_t)b * nv + i];
    DF(qacc_warmstart)[i] = A.warmstart ? A.warmstart[(size_t)b * nv + i] : 0.f;
  }
  for (int i = lane; i < nu; i += 32) DF(ctrl)[i] = A.ctrl[(size_t)b * nu + i];
  for (int i = lane; i < 7 * M.nmocap; i += 32) {
    const int k = i / 7, q = i - 7 * k;
    if (q < 3) DF(mocap_pos)[3 * k + q] = A.mocap[i]; else DF(mocap_quat)[4 * k + q - 3] = A.mocap[i];
  }
  for (int i = lane; i < nv * nv; i += 32) DF(qM)[i] = 0;
  for (int i = lane; i < 6 * M.nbody; i += 32) DF(xfrc)[i] = 0;
  c.time = A.time[b];
  __syncwarp();
  k_forward<SP>(c);
  k_residual<SP>(c);
  if (k_bad(c, DF(qacc), nv)) c.warn = 1;
  const float cost = k_cost_value<SP>(c);
  for (int i = lane; i < nv; i += 32) A.qacc[(size_t)b * nv + i] = DF(qacc)[i];
  for (int i = lane; i < nr; i += 32) A.residual[(size_t)b * nr + i] = DF(residual)[i];
  if (lane == 0) {
    A.cost[b] = cost;
    A.counts[4 * b] = c.ncon - c.npseudo; A.counts[4 * b + 1] = c.nefc; A.counts[4 * b + 2] = c.niter; A.counts[4 * b + 3] = c.warn;
  }
  for (int i = lane; i < nv; i += 32) DF(qacc_warmstart)[i] = DF(qacc)[i];
  k_euler<SP>(c);
  for (int i = lane; i < nq; i += 32) A.next_qpos[(size_t)b * nq + i] = DF(qpos)[i];
  for (int i = lane; i < nv; i += 32) A.next_qvel[(size_t)b * nv + i] = DF(qvel)[i];
}
extern "C" __global__ void __launch_bounds__(32) step_batch_kernel(const __grid_constant__ StepBatchArgs A) {
  step_batch_body<DynSpec>(A);
}
extern "C" __global__ void __launch_bounds__(32) step_batch_kernel_quadruped(const __grid_constant__ StepBatchArgs A) {
  step_batch_body<StaticSpec<SpecQuadruped>>(A);
}
extern "C" __global__ void __launch_bounds__(32) step_batch_kernel_humanoid_track(const __grid_constant__ StepBatchArgs A) {
  step_batch_body<StaticSpec<SpecHumanoidTrack>>(A);
}

}  // namespace mjpc_dev
