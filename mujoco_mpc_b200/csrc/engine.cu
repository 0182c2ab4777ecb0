// engine.cu - host side of libmjpc_b200.so: the C ABI declared in include/mjpc_b200.h.
// Owns the device buffers, the stream and the pinned staging areas; validates arguments; launches the
// kernels in rollout_kernels.cuh / ilqg_kernels.cuh.  There is deliberately NO CPU fallback: without a
// usable CUDA device every entry point returns MJPC_B200_ERR_CUDA.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>   // types only: the NCCL entry points are bound with dlopen at comm_init (no link-time dependency)

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/mjpc_b200.h"
#include "ilqg_kernels.cuh"
#include "rollout_kernels.cuh"

using namespace mjpc_dev;

namespace {
thread_local std::string g_last_error;
int fail(int code, const std::string& msg) { g_last_error = msg; return code; }

#define CUDA_TRY(expr)                                                                                     \
  do {                                                                                                     \
    cudaError_t e_ = (expr);                                                                               \
    if (e_ != cudaSuccess)                                                                                 \
      return fail(MJPC_B200_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));                 \
  } while (0)

// indices of task_state entries that hold absolute times (rebased to the rollout start before upload)
std::vector<int> time_like_state(int residual_id) {
  if (residual_id == RESIDUAL_QUADRUPED_FLAT) return {QS_MODE_START_TIME, QS_PHASE_START_TIME};
  if (residual_id == RESIDUAL_HUMANOID_TRACK) return {1};   // reference_time
  return {};
}
}  // namespace

struct mjpc_b200 {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  ModelPack pack;
  int maxN = 0, maxH = 0, maxP = 64;
  int warps_per_cta = 1;
  int num_sms = 148;
  int static_spec = 0;   // 1 / 2: the model equals spec_quadruped.h / spec_humanoid_track.h -> static rollout kernel
  float* d_pack = nullptr;
  // inputs
  float *d_state = nullptr, *d_mocap = nullptr, *d_task_state = nullptr, *d_knots = nullptr, *d_knot_times = nullptr;
  float *d_unom = nullptr, *d_xnom = nullptr, *d_tnom = nullptr, *d_gains = nullptr, *d_du = nullptr, *d_steps = nullptr;
  // outputs
  float *d_states = nullptr, *d_actions = nullptr, *d_residual = nullptr, *d_costs = nullptr, *d_trace = nullptr,
        *d_returns = nullptr;
  double* d_times = nullptr;
  unsigned char* d_failure = nullptr;
  int* d_order = nullptr;
  long long* d_stats = nullptr;
  unsigned* d_pair_sync = nullptr;   // [256][32]: per-SM records of the co-resident pair synchronisation (dev_data.cuh)
  // debug + ilqg scratch
  float* d_dbg = nullptr;
  IlqgBuffers ilqg;
  // pinned staging
  float* h_in = nullptr;
  size_t h_in_floats = 0;
  unsigned char* h_out = nullptr;
  size_t h_out_bytes = 0;
  // host copies of the live task
  std::vector<double> weight, parameters, task_state;
  double risk = 0;
  std::vector<int> time_idx;
  int lastN = 0, lastH = 0;
  int64_t launches = 0;
  float xfrc_std = 0.f, xfrc_rate = 1.f;   // NoisyRollout settings for the following rollouts (0 = off)
  unsigned noise_seed = 0;
  int last_static = 0;
  float last_ms = 0;
  // multi-GPU: one NCCL communicator per handle; the per-iteration exchange (all-gather of returns + failure flags)
  // is enqueued on the engine stream right behind the rollout kernel
  ncclComm_t comm = nullptr;
  int nranks = 1, rank = 0;
  int totalN = 0, shard_lo = 0, shard_hi = 0;   // of the last sharded rollout
  float *d_slot = nullptr, *d_gather = nullptr, *d_returns_all = nullptr;
  unsigned char* d_failure_all = nullptr;
  int* d_order_all = nullptr;
  float* d_bcast = nullptr;
  size_t bcast_floats = 0;
  int maxTotal = 0;
  int nuserdata = 0;
  int differentiable = 0;   // MakeDifferentiable (utilities.cc:60-75) for the following launches (DevModel::differentiable)
  // batched rollouts (mjpc_b200_rollout_spline_batched): per-problem rows for up to max_candidates problems, packed per
  // call as [state | mocap | task_state | weight | parameters | knot_times] and uploaded with one copy; knots use d_knots
  float* d_batch = nullptr;
  double* d_time0s = nullptr;
  float* h_batch = nullptr;
  double* h_time0s = nullptr;
  // resident-input launch description
  RolloutArgs resident;
  bool resident_ok = false;
  size_t smem_bytes(int P, int wpc) const {
    DevLayout L = make_layout(pack.M, P);
    return ((size_t)smem_header_words(pack.M) + (size_t)wpc * L.total) * 4;
  }
};

namespace {

template <class T>
cudaError_t dalloc(T** p, size_t n) { return cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T)); }

int upload_task(mjpc_b200* h) {
  // weights / parameters / task_state live inside the model pack (float section)
  const DevModel& M = h->pack.M;
  std::vector<float>& f = h->pack.f;
  for (size_t i = 0; i < h->weight.size(); i++) f[M.fo[F_task_weight] + i] = (float)h->weight[i];
  for (size_t i = 0; i < h->parameters.size(); i++) f[M.fo[F_task_parameters] + i] = (float)h->parameters[i];
  for (size_t i = 0; i < h->task_state.size(); i++) f[M.fo[F_task_state] + i] = (float)h->task_state[i];
  h->pack.M.risk = (float)h->risk;
  CUDA_TRY(cudaMemcpyAsync(h->d_pack, f.data(), (size_t)(M.nf + M.ni) * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));  // f is pageable
  return 0;
}

// the dynamic shared-memory opt-in is per kernel (process-wide): only ever raise it, several handles may coexist
int set_smem(const void* fn, size_t bytes) {
  CUDA_TRY(mjpc_dev::raise_smem_limit(fn, bytes));
  return 0;
}

// fill the pinned staging buffer with the per-iteration inputs shared by both rollout flavours
struct Staged { size_t state, mocap, tstate, end; };
Staged stage_common(mjpc_b200* h, const float* state, double time, const float* mocap) {
  const DevModel& M = h->pack.M;
  Staged s;
  size_t o = 0;
  s.state = o; std::memcpy(h->h_in + o, state, (M.nq + M.nv) * 4); o += M.nq + M.nv;
  s.mocap = o; if (M.nmocap) std::memcpy(h->h_in + o, mocap, 7 * M.nmocap * 4); o += 7 * M.nmocap;
  s.tstate = o;
  for (int i = 0; i < M.task_state_size; i++) {
    double v = h->task_state[i];
    if (std::find(h->time_idx.begin(), h->time_idx.end(), i) != h->time_idx.end()) v -= time;
    h->h_in[o + i] = (float)v;
  }
  o += M.task_state_size;
  s.end = o;
  return s;
}

int launch_rollout(mjpc_b200* h, const RolloutArgs& A_in) {
  RolloutArgs A = A_in;
  // A.nprob > 0: the batched instances, A.nprob problems of A.N candidates; a CTA never holds two problems' candidates
  const bool batched = A.nprob > 0;
  const int nprob = batched ? A.nprob : 1, total = nprob * A.N;
  const int wpc = h->warps_per_cta;
  const size_t smem = h->smem_bytes(A.P, wpc);
  const int grid = nprob * ((A.N + wpc - 1) / wpc);
  CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
  // static instance: same arguments, same shared-memory image; MJPC_B200_NO_STATIC=1 forces the generic kernel
  const char* ns = std::getenv("MJPC_B200_NO_STATIC");
  const bool use_static = h->static_spec != 0 && wpc == 1 && !(ns && ns[0] == '1');
  // co-resident pair synchronisation: only when at most two candidates can ever be resident per SM and all are resident
  // at once (one wave); MJPC_B200_PAIR_SYNC=0 switches it off (profiling)
  {
    const char* ps = std::getenv("MJPC_B200_PAIR_SYNC");
    const bool on = !(ps && ps[0] == '0') && total > h->num_sms && total <= 2 * h->num_sms;
    A.pair_sync = on ? h->d_pair_sync : nullptr;
    A.pair_sync_mode = (ps && ps[0] >= '1' && ps[0] <= '9') ? std::atoi(ps) : 1;   // 1: meet per step (default), 3: and before the solve; + 16 k: only at steps with (t & k) == 0
    if (on) CUDA_TRY(cudaMemsetAsync(h->d_pair_sync, 0, (size_t)256 * 32 * sizeof(unsigned), h->stream));
  }
  // MJPC_B200_SHAPE=plain selects the one-warp-per-candidate static instance (tests / profiling: the bitwise reference)
  const char* sh = std::getenv("MJPC_B200_SHAPE");
  const bool plain = sh && sh[0] == 'p' && sh[1] == 'l';
  if (use_static && h->static_spec == 1) {
    if (batched && plain) rollout_kernel_quadruped_plain_batched<<<grid, 32, smem, h->stream>>>(A);
    else if (batched) rollout_kernel_quadruped_batched<<<grid, kRolloutThreads, smem, h->stream>>>(A);
    else if (plain) rollout_kernel_quadruped_plain<<<grid, 32, smem, h->stream>>>(A);
    else rollout_kernel_quadruped<<<grid, kRolloutThreads, smem, h->stream>>>(A);
  } else if (use_static && h->static_spec == 2) {
    if (batched && plain) rollout_kernel_humanoid_track_plain_batched<<<grid, 32, smem, h->stream>>>(A);
    else if (batched) rollout_kernel_humanoid_track_batched<<<grid, kRolloutThreads, smem, h->stream>>>(A);
    else if (plain) rollout_kernel_humanoid_track_plain<<<grid, 32, smem, h->stream>>>(A);
    else rollout_kernel_humanoid_track<<<grid, kRolloutThreads, smem, h->stream>>>(A);
  } else if (batched) {
    rollout_kernel_batched<<<grid, 32 * wpc, smem, h->stream>>>(A);
  } else {
    rollout_kernel<<<grid, 32 * wpc, smem, h->stream>>>(A);
  }
  h->last_static = use_static ? (plain ? 2 : 1) : 0;
  if (batched) rank_batched_kernel<<<(total + 255) / 256, 256, 0, h->stream>>>(A.returns, nprob, A.N, h->d_order);
  else rank_kernel<<<(A.N + 255) / 256, 256, 0, h->stream>>>(A.returns, A.N, h->d_order);
  CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
  CUDA_TRY(cudaGetLastError());
  h->launches += 2;
  h->lastN = total; h->lastH = A.H;
  return 0;
}

RolloutArgs base_args(mjpc_b200* h, double time, int N, int H) {
  RolloutArgs A;
  std::memset(&A, 0, sizeof(A));
  A.M = h->pack.M;
  A.pack = h->d_pack;
  A.state = h->d_state; A.mocap = h->d_mocap; A.task_state = h->d_task_state;
  A.N = N; A.H = H; A.time0 = time;
  A.states = h->d_states; A.actions = h->d_actions; A.times = h->d_times; A.residual = h->d_residual;
  A.costs = h->d_costs; A.trace = h->d_trace; A.returns = h->d_returns; A.failure = h->d_failure;
  A.stats = h->d_stats;
  A.xfrc_std = h->xfrc_std; A.xfrc_rate = h->xfrc_rate; A.noise_seed = h->noise_seed;
  return A;
}

int read_back(mjpc_b200* h, int N, float* returns, uint8_t* failure, int* order) {
  float* hr = (float*)h->h_out;
  int* ho = (int*)(h->h_out + (size_t)N * 4);
  unsigned char* hf = h->h_out + (size_t)N * 8;
  CUDA_TRY(cudaMemcpyAsync(hr, h->d_returns, (size_t)N * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaMemcpyAsync(ho, h->d_order, (size_t)N * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaMemcpyAsync(hf, h->d_failure, (size_t)N, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1) != cudaSuccess) cudaGetLastError();
  if (returns) std::memcpy(returns, hr, (size_t)N * 4);
  if (order) std::memcpy(order, ho, (size_t)N * 4);
  if (failure) std::memcpy(failure, hf, (size_t)N);
  return 0;
}

// ---- NCCL, bound at run time (dlopen): a process that already loaded an NCCL (PyTorch's) shares it by SONAME
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};
NcclApi& nccl_api() {
  static NcclApi api;
  if (api.lib) return api;
  api.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!api.lib) api.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!api.lib) return api;
#define BIND(field, name) api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.lib, name))
  BIND(GetUniqueId, "ncclGetUniqueId"); BIND(CommInitRank, "ncclCommInitRank"); BIND(CommDestroy, "ncclCommDestroy");
  BIND(AllGather, "ncclAllGather"); BIND(Broadcast, "ncclBroadcast"); BIND(GetErrorString, "ncclGetErrorString");
#undef BIND
  api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllGather && api.Broadcast && api.GetErrorString;
  return api;
}
#define NCCL_TRY(expr)                                                                                     \
  do {                                                                                                     \
    ncclResult_t r_ = (expr);                                                                              \
    if (r_ != ncclSuccess)                                                                                 \
      return fail(MJPC_B200_ERR_CUDA, std::string(#expr) + ": " + nccl_api().GetErrorString(r_));          \
  } while (0)

// contiguous balanced candidate ranges (SURVEY.md 8e): the first N % G ranks own one candidate more
inline void shard_range(int N, int G, int r, int* lo, int* hi) {
  const int base = N / G, rem = N % G;
  *lo = r * base + std::min(r, rem);
  *hi = *lo + base + (r < rem ? 1 : 0);
}

// gathered [G][width][2] (return, failure flag) -> compact returns[N], failure[N] in global candidate order
__global__ void compact_gather_kernel(const float* __restrict__ gathered, int N, int G, int width, float* __restrict__ ret,
                                      unsigned char* __restrict__ failure) {
  const int base = N / G, rem = N % G;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    // owner of global candidate i under shard_range
    int r = i < rem * (base + 1) ? i / (base + 1) : rem + (base ? (i - rem * (base + 1)) / base : 0);
    const int lo = r * base + min(r, rem);
    const float* src = gathered + ((size_t)r * width + (i - lo)) * 2;
    ret[i] = src[0];
    failure[i] = src[1] != 0.f ? 1 : 0;
  }
}
__global__ void pack_slot_kernel(const float* __restrict__ ret, const unsigned char* __restrict__ failure, int n, int width,
                                 float* __restrict__ slot) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < width; i += gridDim.x * blockDim.x) {
    slot[2 * i] = i < n ? ret[i] : 3.0e38f;
    slot[2 * i + 1] = i < n ? (float)failure[i] : 1.f;
  }
}

}  // namespace

extern "C" {

const char* mjpc_b200_version(void) { return "mjpc_b200 0.1.0 (sm_100a)"; }
const char* mjpc_b200_last_error(void) { return g_last_error.c_str(); }

// inside create(): a failing CUDA call must not leak the half-built handle
#define CREATE_TRY(expr)                                                                                   \
  do {                                                                                                     \
    cudaError_t e_ = (expr);                                                                               \
    if (e_ != cudaSuccess) {                                                                               \
      mjpc_b200_destroy(h);                                                                                \
      return fail(MJPC_B200_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));                 \
    }                                                                                                      \
  } while (0)

int mjpc_b200_create(const mjpc_model_blob* model, int max_candidates, int max_horizon, int device,
                     mjpc_b200_t** out) {
  if (!model || !model->data || !out || max_candidates < 1 || max_horizon < 1)
    return fail(MJPC_B200_ERR_BAD_ARGUMENT, "create: bad argument");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(MJPC_B200_ERR_CUDA, "no CUDA device: the engine has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "create: bad device ordinal");
  mjpc_b200* h = new mjpc_b200;
  try {
    int maxcon = 32, maxefc = 96;
    h->pack = pack_model(model->data, model->nbytes, maxcon, maxefc);
  } catch (const std::exception& e) {
    delete h;
    return fail(MJPC_B200_ERR_BAD_BLOB, std::string("create: ") + e.what());
  }
  h->device = device;
  if (const char* w = std::getenv("MJPC_B200_WARPS_PER_CTA")) {  // tuning knob (profiles/): candidates per CTA
    const int v = std::atoi(w);
    if (v == 1 || v == 2 || v == 4) h->warps_per_cta = v;
  }
  h->maxN = max_candidates; h->maxH = max_horizon;
  const DevModel& M = h->pack.M;
  {
    Blob b(model->data, model->nbytes);
    h->nuserdata = b.i("nuserdata");
    if (h->nuserdata != 0) { delete h; return fail(MJPC_B200_ERR_UNSUPPORTED, "create: mjData::userdata (nuserdata > 0) is not supported"); }
    h->weight = b.reals("task_weight"); h->parameters = b.reals("task_parameters");
    h->task_state = b.reals("task_state"); h->risk = b.r("task_risk");
  }
  h->time_idx = time_like_state(M.residual_id);
  CREATE_TRY(cudaSetDevice(device));
  CREATE_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CREATE_TRY(cudaEventCreate(&h->ev0));
  CREATE_TRY(cudaEventCreate(&h->ev1));
  cudaDeviceProp prop;
  CREATE_TRY(cudaGetDeviceProperties(&prop, device));
  h->num_sms = prop.multiProcessorCount;
  const size_t smem_need = h->smem_bytes(h->maxP, 1);
  if (smem_need > (size_t)prop.sharedMemPerBlockOptin) {
    mjpc_b200_destroy(h);
    return fail(MJPC_B200_ERR_CAPACITY, "model does not fit in shared memory");
  }
  // pack: floats then ints, one buffer (single TMA bulk copy per CTA)
  {
    std::vector<float>& f = h->pack.f;
    const size_t nf = f.size();
    f.resize(nf + h->pack.i.size());
    std::memcpy(f.data() + nf, h->pack.i.data(), h->pack.i.size() * 4);
    // not staged to shared memory: keyframe mocap positions, read from HBM by the tracking residual (Ctx::gkey)
    for (double x : h->pack.key_mpos) f.push_back((float)x);
    CREATE_TRY(dalloc(&h->d_pack, f.size()));
    CREATE_TRY(cudaMemcpy(h->d_pack, f.data(), f.size() * 4, cudaMemcpyHostToDevice));
  }
  const size_t N = max_candidates, H = max_horizon, ds = M.nq + M.nv, n = 2 * M.nv, nu = M.nu, nr = M.num_residual;
  CREATE_TRY(dalloc(&h->d_state, ds)); CREATE_TRY(dalloc(&h->d_mocap, 7 * (size_t)M.nmocap));
  CREATE_TRY(dalloc(&h->d_task_state, (size_t)M.task_state_size));
  CREATE_TRY(dalloc(&h->d_knots, N * h->maxP * nu)); CREATE_TRY(dalloc(&h->d_knot_times, (size_t)h->maxP));
  CREATE_TRY(dalloc(&h->d_unom, H * nu)); CREATE_TRY(dalloc(&h->d_xnom, H * ds)); CREATE_TRY(dalloc(&h->d_tnom, H));
  CREATE_TRY(dalloc(&h->d_gains, H * nu * n)); CREATE_TRY(dalloc(&h->d_du, H * nu)); CREATE_TRY(dalloc(&h->d_steps, N));
  CREATE_TRY(dalloc(&h->d_states, N * H * ds)); CREATE_TRY(dalloc(&h->d_actions, N * H * nu));
  CREATE_TRY(dalloc(&h->d_times, N * H)); CREATE_TRY(dalloc(&h->d_residual, N * H * nr));
  CREATE_TRY(dalloc(&h->d_costs, N * H)); CREATE_TRY(dalloc(&h->d_trace, N * H * 3 * (size_t)M.num_trace));
  CREATE_TRY(dalloc(&h->d_returns, N)); CREATE_TRY(dalloc(&h->d_failure, N)); CREATE_TRY(dalloc(&h->d_order, N)); CREATE_TRY(dalloc(&h->d_stats, 12 * N));
  CREATE_TRY(dalloc(&h->d_pair_sync, (size_t)256 * 32));
  CREATE_TRY(dalloc(&h->d_dbg, 4 * ds + 2 * nu + (size_t)M.nv * M.nv + nr + 256 + 64 + 7 * (size_t)M.nmocap));
  h->h_in_floats = ds + 7 * M.nmocap + M.task_state_size + N * h->maxP * nu + h->maxP + H * (nu + ds + 1 + nu * n + nu) + N + 64;
  CREATE_TRY(cudaMallocHost((void**)&h->h_in, h->h_in_floats * 4));
  h->h_out_bytes = N * 16 + 64;
  CREATE_TRY(cudaMallocHost((void**)&h->h_out, h->h_out_bytes));
  {
    const size_t row = ds + 7 * (size_t)M.nmocap + M.task_state_size + M.num_term + M.num_parameters + h->maxP;
    CREATE_TRY(dalloc(&h->d_batch, N * row)); CREATE_TRY(dalloc(&h->d_time0s, N));
    CREATE_TRY(cudaMallocHost((void**)&h->h_batch, N * row * 4)); CREATE_TRY(cudaMallocHost((void**)&h->h_time0s, N * 8));
  }
  if (int rc = set_smem((const void*)rollout_kernel, h->smem_bytes(h->maxP, h->warps_per_cta))) { mjpc_b200_destroy(h); return rc; }
  if (int rc = set_smem((const void*)rollout_kernel_batched, h->smem_bytes(h->maxP, h->warps_per_cta))) { mjpc_b200_destroy(h); return rc; }
  if (int rc = set_smem((const void*)step_debug_kernel, h->smem_bytes(1, 1))) { mjpc_b200_destroy(h); return rc; }
  if (spec_matches<SpecQuadruped>(M, make_layout(M, 1))) {
    h->static_spec = 1;
    if (int rc = set_smem((const void*)rollout_kernel_quadruped, h->smem_bytes(h->maxP, 1))) { mjpc_b200_destroy(h); return rc; }
    if (int rc = set_smem((const void*)rollout_kernel_quadruped_plain, h->smem_bytes(h->maxP, 1))) { mjpc_b200_destroy(h); return rc; }
    if (int rc = set_smem((const void*)rollout_kernel_quadruped_batched, h->smem_bytes(h->maxP, 1))) { mjpc_b200_destroy(h); return rc; }
    if (int rc = set_smem((const void*)rollout_kernel_quadruped_plain_batched, h->smem_bytes(h->maxP, 1))) { mjpc_b200_destroy(h); return rc; }
  } else if (spec_matches<SpecHumanoidTrack>(M, make_layout(M, 1))) {
    h->static_spec = 2;
    if (int rc = set_smem((const void*)rollout_kernel_humanoid_track, h->smem_bytes(h->maxP, 1))) { mjpc_b200_destroy(h); return rc; }
    if (int rc = set_smem((const void*)rollout_kernel_humanoid_track_plain, h->smem_bytes(h->maxP, 1))) { mjpc_b200_destroy(h); return rc; }
    if (int rc = set_smem((const void*)rollout_kernel_humanoid_track_batched, h->smem_bytes(h->maxP, 1))) { mjpc_b200_destroy(h); return rc; }
    if (int rc = set_smem((const void*)rollout_kernel_humanoid_track_plain_batched, h->smem_bytes(h->maxP, 1))) { mjpc_b200_destroy(h); return rc; }
  }
  if (int rc = ilqg_init(h->ilqg, h->pack.M, (int)H, h->smem_bytes(1, 1))) {
    mjpc_b200_destroy(h);
    return fail(rc, "ilqg buffer allocation failed");
  }
  *out = h;
  return MJPC_B200_OK;
}

void mjpc_b200_destroy(mjpc_b200_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->comm && nccl_api().ok) nccl_api().CommDestroy(h->comm);
  void* mbufs[] = {h->d_slot, h->d_gather, h->d_returns_all, h->d_failure_all, h->d_order_all, h->d_bcast};
  for (void* p : mbufs) if (p) cudaFree(p);
  void* bufs[] = {h->d_pack, h->d_state, h->d_mocap, h->d_task_state, h->d_knots, h->d_knot_times, h->d_unom, h->d_xnom,
                  h->d_tnom, h->d_gains, h->d_du, h->d_steps, h->d_states, h->d_actions, h->d_times, h->d_residual,
                  h->d_costs, h->d_trace, h->d_returns, h->d_failure, h->d_order, h->d_dbg, h->d_stats, h->d_pair_sync,
                  h->d_batch, h->d_time0s};
  for (void* p : bufs) if (p) cudaFree(p);
  ilqg_free(h->ilqg);
  if (h->h_in) cudaFreeHost(h->h_in);
  if (h->h_out) cudaFreeHost(h->h_out);
  if (h->h_batch) cudaFreeHost(h->h_batch);
  if (h->h_time0s) cudaFreeHost(h->h_time0s);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int mjpc_b200_get_info(const mjpc_b200_t* h, mjpc_b200_info* info) {
  if (!h || !info) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "get_info: null");
  const DevModel& M = h->pack.M;
  info->nq = M.nq; info->nv = M.nv; info->nu = M.nu; info->na = 0 /* na > 0 is rejected by create() */; info->nmocap = M.nmocap; info->nuserdata = h->nuserdata;
  info->dim_state = M.nq + M.nv; info->dim_dstate = 2 * M.nv;
  info->num_residual = M.num_residual; info->num_term = M.num_term; info->num_trace = M.num_trace;
  info->num_parameters = M.num_parameters; info->task_state_size = M.task_state_size;
  info->max_candidates = h->maxN; info->max_horizon = h->maxH; info->device = h->device;
  info->smem_bytes_per_warp = make_layout(M, 3).total * 4;
  return 0;
}

int mjpc_b200_set_task(mjpc_b200_t* h, const mjpc_task_desc* task) {
  if (!h || !task) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "set_task: null");
  CUDA_TRY(cudaSetDevice(h->device));
  if (task->weight) h->weight.assign(task->weight, task->weight + h->weight.size());
  if (task->parameters) h->parameters.assign(task->parameters, task->parameters + h->parameters.size());
  if (task->task_state) h->task_state.assign(task->task_state, task->task_state + h->task_state.size());
  h->risk = task->risk;
  return upload_task(h);
}

// Agent::PlanIteration's planning-model overrides (agent.cc:288-289): model_->opt.timestep = agent_timestep,
// model_->opt.integrator = agent_integrator.  The timestep is a live header option (no re-upload); only the Euler
// integrator (mjINT_EULER = 0) is implemented on the device - anything else is refused, never silently replaced.
int mjpc_b200_set_options(mjpc_b200_t* h, double timestep, int integrator) {
  if (!h || !(timestep > 0)) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "set_options: bad argument");
  if (integrator != 0) return fail(MJPC_B200_ERR_UNSUPPORTED, "set_options: only the Euler integrator (0) is implemented");
  h->pack.M.timestep = (float)timestep;
  return 0;
}

// Agent::PlanIteration's MakeDifferentiable (agent.cc:296-309, utilities.cc:60-75): while on, every joint's and geom's
// solimp[0] reads as 0 in the kernels (contact pairs take their solimp from the geoms here); off restores the model's own
// values (agent.cc:346-356).  Gradient-based planners (iLQG, iLQS, Gradient) plan with it on by default.
int mjpc_b200_set_differentiable(mjpc_b200_t* h, int on) {
  if (!h) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "set_differentiable: null");
  h->differentiable = on ? 1 : 0;
  h->pack.M.differentiable = on ? 1.f : 0.f;   // a header option: every launch copies the live header, no re-upload
  return 0;
}

int mjpc_b200_upload_spline_inputs(mjpc_b200_t* h, const float* state, double time, const float* mocap,
                                   const float* userdata, const float* knots, const double* knot_times, int interp,
                                   int P, int N, int H) {
  if (!h || !state || !knots || !knot_times) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_spline: null pointer");
  const DevModel& M = h->pack.M;
  // mjData::userdata: none of the implemented residuals reads it; a model that declares nuserdata > 0 is rejected at
  // create(), so a non-NULL pointer here can only be a caller error - refuse rather than silently ignore it
  if (userdata && h->nuserdata == 0) return fail(MJPC_B200_ERR_UNSUPPORTED, "rollout_spline: the model has nuserdata = 0, userdata must be NULL");
  if (M.nmocap && !mocap) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_spline: mocap required");
  if (N < 1 || H < 1 || P < 1 || interp < 0 || interp > 2) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_spline: bad sizes");
  if (N > h->maxN || H > h->maxH || P > h->maxP) return fail(MJPC_B200_ERR_CAPACITY, "rollout_spline: N/H/P above capacity");
  CUDA_TRY(cudaSetDevice(h->device));
  Staged s = stage_common(h, state, time, mocap);
  size_t o = s.end;
  const size_t ok = o; std::memcpy(h->h_in + o, knots, (size_t)N * P * M.nu * 4); o += (size_t)N * P * M.nu;
  const size_t ot = o;
  for (int i = 0; i < P; i++) h->h_in[o + i] = (float)(knot_times[i] - time);
  o += P;
  CUDA_TRY(cudaMemcpyAsync(h->d_state, h->h_in + s.state, (M.nq + M.nv) * 4, cudaMemcpyHostToDevice, h->stream));
  if (M.nmocap) CUDA_TRY(cudaMemcpyAsync(h->d_mocap, h->h_in + s.mocap, 7 * M.nmocap * 4, cudaMemcpyHostToDevice, h->stream));
  if (M.task_state_size) CUDA_TRY(cudaMemcpyAsync(h->d_task_state, h->h_in + s.tstate, M.task_state_size * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaMemcpyAsync(h->d_knots, h->h_in + ok, (size_t)N * P * M.nu * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaMemcpyAsync(h->d_knot_times, h->h_in + ot, (size_t)P * 4, cudaMemcpyHostToDevice, h->stream));
  RolloutArgs A = base_args(h, time, N, H);
  A.L = make_layout(h->pack.M, P);
  A.knots = h->d_knots; A.knot_times = h->d_knot_times; A.P = P; A.interp = interp; A.policy_kind = 0;
  h->resident = A;
  h->resident_ok = true;
  return 0;
}

int mjpc_b200_launch_resident(mjpc_b200_t* h) {
  if (!h || !h->resident_ok) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "launch_resident: no uploaded inputs");
  CUDA_TRY(cudaSetDevice(h->device));
  h->resident.M = h->pack.M;  // picks up set_task changes (risk)
  return launch_rollout(h, h->resident);
}

int mjpc_b200_sync(mjpc_b200_t* h) {
  if (!h) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "sync: null");
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (h->lastN > 0 && cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1) != cudaSuccess) cudaGetLastError();
  return 0;
}

int mjpc_b200_read_returns(mjpc_b200_t* h, float* returns, uint8_t* failure, int* order) {
  if (!h || h->lastN < 1) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "read_returns: nothing launched");
  CUDA_TRY(cudaSetDevice(h->device));
  return read_back(h, h->lastN, returns, failure, order);
}

int mjpc_b200_rollout_spline(mjpc_b200_t* h, const float* state, double time, const float* mocap,
                             const float* userdata, const float* knots, const double* knot_times, int interp,
                             int P, int N, int H, float* returns, uint8_t* failure, int* order) {
  int rc = mjpc_b200_upload_spline_inputs(h, state, time, mocap, userdata, knots, knot_times, interp, P, N, H);
  if (rc) return rc;
  rc = launch_rollout(h, h->resident);
  if (rc) return rc;
  return read_back(h, N, returns, failure, order);
}

// M independent problems of the same model in one launch.  Every per-problem input is converted exactly as
// upload_spline_inputs / upload_task convert a single problem's (knot and task-state times rebased to the problem's own
// start, weights and parameters rounded to float), so problem p computes bit for bit what rollout_spline computes for it.
int mjpc_b200_rollout_spline_batched(mjpc_b200_t* h, int M, const float* state, const double* time, const float* mocap,
                                     const mjpc_task_batch* task, const float* knots, const double* knot_times, int interp,
                                     int P, int N, int H, float* returns, uint8_t* failure, int* order) {
  if (!h || !state || !time || !knots || !knot_times) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_spline_batched: null pointer");
  const DevModel& D = h->pack.M;
  if (D.nmocap && !mocap) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_spline_batched: mocap required");
  if (M < 1 || N < 1 || H < 1 || P < 1 || interp < 0 || interp > 2)
    return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_spline_batched: bad sizes");
  if ((int64_t)M * N > h->maxN || H > h->maxH || P > h->maxP)
    return fail(MJPC_B200_ERR_CAPACITY, "rollout_spline_batched: M*N/H/P above capacity");
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t ds = D.nq + D.nv, nm = 7 * (size_t)D.nmocap, nts = D.task_state_size, nw = D.num_term,
               np = D.num_parameters, nk = (size_t)N * P * D.nu;
  const size_t o_state = 0, o_mocap = o_state + M * ds, o_ts = o_mocap + M * nm, o_w = o_ts + M * nts, o_p = o_w + M * nw,
               o_kt = o_p + M * np, end = o_kt + (size_t)M * P;
  float* b = h->h_batch;
  std::memcpy(b + o_state, state, M * ds * 4);
  if (nm) std::memcpy(b + o_mocap, mocap, M * nm * 4);
  const double* tw = task ? task->weight : nullptr;
  const double* tp = task ? task->parameters : nullptr;
  const double* tts = task ? task->task_state : nullptr;
  for (int p = 0; p < M; p++) {
    const double t0 = time[p];
    h->h_time0s[p] = t0;
    for (size_t i = 0; i < nts; i++) {
      double v = tts ? tts[p * nts + i] : h->task_state[i];
      if (std::find(h->time_idx.begin(), h->time_idx.end(), (int)i) != h->time_idx.end()) v -= t0;
      b[o_ts + p * nts + i] = (float)v;
    }
    for (size_t i = 0; i < nw; i++) b[o_w + p * nw + i] = (float)(tw ? tw[p * nw + i] : h->weight[i]);
    for (size_t i = 0; i < np; i++) b[o_p + p * np + i] = (float)(tp ? tp[p * np + i] : h->parameters[i]);
    for (int k = 0; k < P; k++) b[o_kt + (size_t)p * P + k] = (float)(knot_times[(size_t)p * P + k] - t0);
  }
  std::memcpy(h->h_in, knots, M * nk * 4);
  CUDA_TRY(cudaMemcpyAsync(h->d_batch, b, end * 4, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaMemcpyAsync(h->d_time0s, h->h_time0s, (size_t)M * 8, cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(cudaMemcpyAsync(h->d_knots, h->h_in, M * nk * 4, cudaMemcpyHostToDevice, h->stream));
  RolloutArgs A = base_args(h, time[0], N, H);
  A.L = make_layout(h->pack.M, P);
  A.state = h->d_batch + o_state; A.mocap = h->d_batch + o_mocap; A.task_state = h->d_batch + o_ts;
  A.task_weight = h->d_batch + o_w; A.task_parameters = h->d_batch + o_p;
  A.knots = h->d_knots; A.knot_times = h->d_batch + o_kt; A.P = P; A.interp = interp; A.policy_kind = 0;
  A.nprob = M; A.time0s = h->d_time0s;
  h->resident_ok = false;   // d_knots now holds the batch
  int rc = launch_rollout(h, A);
  if (rc) return rc;
  return read_back(h, M * N, returns, failure, order);
}

int mjpc_b200_rollout_feedback(mjpc_b200_t* h, const float* state, double time, const float* mocap,
                               const float* userdata, const float* u_nom, const float* x_nom, const double* t_nom,
                               const float* gains, const float* du, const float* step_sizes, int mode, int K, int H,
                               float* returns, uint8_t* failure, int* order) {
  if (!h || !state || !u_nom || !x_nom || !t_nom || !gains || !step_sizes)
    return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_feedback: null pointer");
  if (userdata && h->nuserdata == 0) return fail(MJPC_B200_ERR_UNSUPPORTED, "rollout_feedback: the model has nuserdata = 0, userdata must be NULL");
  const DevModel& M = h->pack.M;
  if (M.nmocap && !mocap) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_feedback: mocap required");
  if (K < 1 || H < 1 || mode < 0 || mode > 3) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_feedback: bad sizes");
  if (K > h->maxN || H > h->maxH) return fail(MJPC_B200_ERR_CAPACITY, "rollout_feedback: K/H above capacity");
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t ds = M.nq + M.nv, n = 2 * M.nv, nu = M.nu;
  Staged s = stage_common(h, state, time, mocap);
  size_t o = s.end;
  auto put = [&](const float* src, size_t cnt) { size_t at = o; if (src) std::memcpy(h->h_in + o, src, cnt * 4); o += cnt; return at; };
  const size_t ou = put(u_nom, H * nu), ox = put(x_nom, H * ds);
  const size_t ot = o;
  for (int i = 0; i < H; i++) h->h_in[o + i] = (float)(t_nom[i] - time);
  o += H;
  const size_t og = put(gains, H * nu * n), od = put(du, H * nu), os = put(step_sizes, K);
  auto up = [&](float* dst, size_t at, size_t cnt) { return cudaMemcpyAsync(dst, h->h_in + at, cnt * 4, cudaMemcpyHostToDevice, h->stream); };
  CUDA_TRY(up(h->d_state, s.state, ds));
  if (M.nmocap) CUDA_TRY(up(h->d_mocap, s.mocap, 7 * M.nmocap));
  if (M.task_state_size) CUDA_TRY(up(h->d_task_state, s.tstate, M.task_state_size));
  CUDA_TRY(up(h->d_unom, ou, H * nu)); CUDA_TRY(up(h->d_xnom, ox, H * ds)); CUDA_TRY(up(h->d_tnom, ot, H));
  CUDA_TRY(up(h->d_gains, og, H * nu * n));
  if (du) CUDA_TRY(up(h->d_du, od, H * nu));
  CUDA_TRY(up(h->d_steps, os, K));
  RolloutArgs A = base_args(h, time, K, H);
  A.L = make_layout(h->pack.M, 1);
  A.P = 1; A.policy_kind = 1;
  A.fb.u_nom = h->d_unom; A.fb.x_nom = h->d_xnom; A.fb.t_nom = h->d_tnom; A.fb.gains = h->d_gains;
  A.fb.du = du ? h->d_du : nullptr; A.fb.mode = mode; A.fb.H = H;
  A.step_sizes = h->d_steps;
  h->resident_ok = false;
  int rc = launch_rollout(h, A);
  if (rc) return rc;
  return read_back(h, K, returns, failure, order);
}

static int fetch_impl(mjpc_b200_t* h, int first, int count, float* states, float* actions, double* times,
                      float* residual, float* costs, float* trace) {
  const DevModel& M = h->pack.M;
  const size_t H = h->lastH, ds = M.nq + M.nv, nu = M.nu, nr = M.num_residual, ntr = 3 * M.num_trace;
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  auto get = [&](void* dst, const void* src, size_t per, size_t elt) {
    return dst ? cudaMemcpy(dst, (const char*)src + (size_t)first * per * elt, (size_t)count * per * elt, cudaMemcpyDeviceToHost) : cudaSuccess;
  };
  CUDA_TRY(get(states, h->d_states, H * ds, 4)); CUDA_TRY(get(actions, h->d_actions, H * nu, 4));
  CUDA_TRY(get(times, h->d_times, H, 8)); CUDA_TRY(get(residual, h->d_residual, H * nr, 4));
  CUDA_TRY(get(costs, h->d_costs, H, 4)); CUDA_TRY(get(trace, h->d_trace, H * ntr, 4));
  return 0;
}

int mjpc_b200_fetch_trajectory(mjpc_b200_t* h, int candidate, float* states, float* actions, double* times,
                               float* residual, float* costs, float* trace) {
  if (!h || h->lastN < 1 || candidate < 0 || candidate >= h->lastN)
    return fail(MJPC_B200_ERR_BAD_ARGUMENT, "fetch_trajectory: bad candidate");
  return fetch_impl(h, candidate, 1, states, actions, times, residual, costs, trace);
}

int mjpc_b200_fetch_all(mjpc_b200_t* h, float* states, float* actions, double* times, float* residual, float* costs,
                        float* trace) {
  if (!h || h->lastN < 1) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "fetch_all: nothing to fetch");
  return fetch_impl(h, 0, h->lastN, states, actions, times, residual, costs, trace);
}

int mjpc_b200_step_debug(mjpc_b200_t* h, const float* qpos, const float* qvel, const float* ctrl,
                         const float* mocap, double time, const float* warmstart, float* qacc, float* residual,
                         float* next_qpos, float* next_qvel, float* qM, float* efc_force, int* counts) {
  if (!h || !qpos || !qvel || !ctrl) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "step_debug: null");
  const DevModel& M = h->pack.M;
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t nq = M.nq, nv = M.nv, nu = M.nu, nr = M.num_residual;
  float* d = h->d_dbg;
  float *d_qpos = d, *d_qvel = d_qpos + nq, *d_ctrl = d_qvel + nv, *d_mocap = d_ctrl + nu, *d_warm = d_mocap + 7 * M.nmocap,
        *d_qacc = d_warm + nv, *d_res = d_qacc + nv, *d_nq = d_res + nr, *d_nv = d_nq + nq, *d_qM = d_nv + nv,
        *d_force = d_qM + nv * nv;
  int* d_counts = (int*)(d_force + 256);
  CUDA_TRY(cudaMemcpy(d_qpos, qpos, nq * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_qvel, qvel, nv * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_ctrl, ctrl, nu * 4, cudaMemcpyHostToDevice));
  if (M.nmocap) CUDA_TRY(cudaMemcpy(d_mocap, mocap, 7 * M.nmocap * 4, cudaMemcpyHostToDevice));
  if (warmstart) CUDA_TRY(cudaMemcpy(d_warm, warmstart, nv * 4, cudaMemcpyHostToDevice));
  std::vector<float> ts(M.task_state_size);
  for (int i = 0; i < M.task_state_size; i++) ts[i] = (float)h->task_state[i];
  if (M.task_state_size) CUDA_TRY(cudaMemcpy(h->d_task_state, ts.data(), ts.size() * 4, cudaMemcpyHostToDevice));
  DebugArgs A;
  std::memset(&A, 0, sizeof(A));
  A.M = h->pack.M; A.L = make_layout(h->pack.M, 1); A.pack = h->d_pack;
  A.qpos = d_qpos; A.qvel = d_qvel; A.ctrl = d_ctrl; A.mocap = d_mocap; A.warmstart = warmstart ? d_warm : nullptr;
  A.task_state = M.task_state_size ? h->d_task_state : nullptr;
  A.time = (float)time;
  A.qacc = d_qacc; A.residual = d_res; A.next_qpos = d_nq; A.next_qvel = d_nv; A.qM = d_qM; A.efc_force = d_force;
  A.counts = d_counts;
  step_debug_kernel<<<1, 32, h->smem_bytes(1, 1), h->stream>>>(A);
  h->launches += 1;
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (qacc) CUDA_TRY(cudaMemcpy(qacc, d_qacc, nv * 4, cudaMemcpyDeviceToHost));
  if (residual) CUDA_TRY(cudaMemcpy(residual, d_res, nr * 4, cudaMemcpyDeviceToHost));
  if (next_qpos) CUDA_TRY(cudaMemcpy(next_qpos, d_nq, nq * 4, cudaMemcpyDeviceToHost));
  if (next_qvel) CUDA_TRY(cudaMemcpy(next_qvel, d_nv, nv * 4, cudaMemcpyDeviceToHost));
  if (qM) CUDA_TRY(cudaMemcpy(qM, d_qM, nv * nv * 4, cudaMemcpyDeviceToHost));
  if (efc_force) CUDA_TRY(cudaMemcpy(efc_force, d_force, 256 * 4, cudaMemcpyDeviceToHost));
  if (counts) CUDA_TRY(cudaMemcpy(counts, d_counts, 16, cudaMemcpyDeviceToHost));
  return 0;
}

// ---- multi-GPU: one planning problem, candidates sharded over the ranks of an NCCL communicator (SURVEY.md 8e)
int mjpc_b200_comm_unique_id(void* out, size_t nbytes) {
  if (!out || nbytes < sizeof(ncclUniqueId)) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "comm_unique_id: need 128 bytes");
  NcclApi& api = nccl_api();
  if (!api.ok) return fail(MJPC_B200_ERR_UNSUPPORTED, "libnccl.so.2 not found");
  ncclUniqueId id;
  NCCL_TRY(api.GetUniqueId(&id));
  std::memcpy(out, &id, sizeof(id));
  return 0;
}

int mjpc_b200_comm_init(mjpc_b200_t* h, int nranks, int rank, const void* unique_id, size_t nbytes) {
  if (!h || nranks < 1 || rank < 0 || rank >= nranks || !unique_id || nbytes < sizeof(ncclUniqueId))
    return fail(MJPC_B200_ERR_BAD_ARGUMENT, "comm_init: bad argument");
  if (h->comm) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "comm_init: communicator already initialised");
  NcclApi& api = nccl_api();
  if (!api.ok) return fail(MJPC_B200_ERR_UNSUPPORTED, "libnccl.so.2 not found");
  CUDA_TRY(cudaSetDevice(h->device));
  ncclUniqueId id;
  std::memcpy(&id, unique_id, sizeof(id));
  NCCL_TRY(api.CommInitRank(&h->comm, nranks, id, rank));
  h->nranks = nranks; h->rank = rank;
  h->maxTotal = nranks * h->maxN;
  const DevModel& M = h->pack.M;
  const size_t width = h->maxN;
  CUDA_TRY(dalloc(&h->d_slot, 2 * width)); CUDA_TRY(dalloc(&h->d_gather, 2 * width * nranks));
  CUDA_TRY(dalloc(&h->d_returns_all, (size_t)h->maxTotal)); CUDA_TRY(dalloc(&h->d_failure_all, (size_t)h->maxTotal));
  CUDA_TRY(dalloc(&h->d_order_all, (size_t)h->maxTotal));
  h->bcast_floats = (size_t)h->maxH * (M.nq + M.nv + M.nu + M.num_residual + 1 + 3 * M.num_trace + 2) + 16;
  CUDA_TRY(dalloc(&h->d_bcast, h->bcast_floats));
  return 0;
}

int mjpc_b200_comm_info(const mjpc_b200_t* h, int* nranks, int* rank) {
  if (!h) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "comm_info: null");
  if (nranks) *nranks = h->nranks;
  if (rank) *rank = h->rank;
  return 0;
}

// SamplingPlanner::Rollouts for ONE planning problem on all ranks: every rank passes the same N candidates (inputs are
// replicated: a few KB), rolls out its contiguous shard, then the per-candidate returns and failure flags are exchanged
// with ONE ncclAllGather enqueued on the engine stream behind the rollout kernel (no host hop), compacted to global
// candidate order and ranked on the device.  returns / failure / order describe all N candidates, identical on every rank.
int mjpc_b200_rollout_spline_sharded(mjpc_b200_t* h, const float* state, double time, const float* mocap,
                                     const float* userdata, const float* knots, const double* knot_times, int interp,
                                     int P, int N, int H, float* returns, uint8_t* failure, int* order) {
  if (!h || !knots) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_spline_sharded: null");
  if (h->nranks > 1 && !h->comm) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "rollout_spline_sharded: comm_init first");
  if (h->nranks == 1) {
    int rc = mjpc_b200_rollout_spline(h, state, time, mocap, userdata, knots, knot_times, interp, P, N, H, returns, failure, order);
    if (rc == 0) { h->totalN = N; h->shard_lo = 0; h->shard_hi = N; }
    return rc;
  }
  if (N < h->nranks || N > h->maxTotal) return fail(MJPC_B200_ERR_CAPACITY, "rollout_spline_sharded: N outside [nranks, nranks * max_candidates]");
  const DevModel& M = h->pack.M;
  int lo, hi;
  shard_range(N, h->nranks, h->rank, &lo, &hi);
  const int n = hi - lo, width = N / h->nranks + (N % h->nranks ? 1 : 0);
  if (n > h->maxN) return fail(MJPC_B200_ERR_CAPACITY, "rollout_spline_sharded: shard above max_candidates");
  int rc = mjpc_b200_upload_spline_inputs(h, state, time, mocap, userdata, knots + (size_t)lo * P * M.nu, knot_times, interp, P, n, H);
  if (rc) return rc;
  h->resident.cand0 = lo;
  rc = launch_rollout(h, h->resident);
  if (rc) return rc;
  NcclApi& api = nccl_api();
  pack_slot_kernel<<<(width + 255) / 256, 256, 0, h->stream>>>(h->d_returns, h->d_failure, n, width, h->d_slot);
  NCCL_TRY(api.AllGather(h->d_slot, h->d_gather, 2 * (size_t)width, ncclFloat, h->comm, h->stream));
  compact_gather_kernel<<<(N + 255) / 256, 256, 0, h->stream>>>(h->d_gather, N, h->nranks, width, h->d_returns_all, h->d_failure_all);
  rank_kernel<<<(N + 255) / 256, 256, 0, h->stream>>>(h->d_returns_all, N, h->d_order_all);
  CUDA_TRY(cudaEventRecord(h->ev1, h->stream));   // the timed span now covers rollout + exchange + ranking
  CUDA_TRY(cudaGetLastError());
  h->launches += 3;
  h->totalN = N; h->shard_lo = lo; h->shard_hi = hi;
  float* hr = (float*)h->h_out;   // h_out holds maxN * 16 bytes: read back in chunks through pageable copies instead
  (void)hr;
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1) != cudaSuccess) cudaGetLastError();
  if (returns) CUDA_TRY(cudaMemcpy(returns, h->d_returns_all, (size_t)N * 4, cudaMemcpyDeviceToHost));
  if (failure) CUDA_TRY(cudaMemcpy(failure, h->d_failure_all, (size_t)N, cudaMemcpyDeviceToHost));
  if (order) CUDA_TRY(cudaMemcpy(order, h->d_order_all, (size_t)N * 4, cudaMemcpyDeviceToHost));
  return 0;
}

// Trajectory of GLOBAL candidate `candidate` of the last sharded rollout on every rank: the owner packs it into one
// buffer, ncclBroadcast on the engine stream, every rank unpacks (BestTrajectory must be available wherever the policy
// is installed).  Any output pointer may be NULL.
int mjpc_b200_fetch_trajectory_sharded(mjpc_b200_t* h, int candidate, float* states, float* actions, double* times,
                                       float* residual, float* costs, float* trace) {
  if (!h || h->totalN < 1 || candidate < 0 || candidate >= h->totalN)
    return fail(MJPC_B200_ERR_BAD_ARGUMENT, "fetch_trajectory_sharded: bad candidate");
  if (h->nranks == 1) return mjpc_b200_fetch_trajectory(h, candidate, states, actions, times, residual, costs, trace);
  const DevModel& M = h->pack.M;
  const size_t H = h->lastH, ds = M.nq + M.nv, nu = M.nu, nr = M.num_residual, ntr = 3 * M.num_trace;
  CUDA_TRY(cudaSetDevice(h->device));
  int owner = 0, lo = 0, hi = 0;
  for (owner = 0; owner < h->nranks; owner++) { shard_range(h->totalN, h->nranks, owner, &lo, &hi); if (candidate < hi) break; }
  float* b = h->d_bcast;
  const size_t o_s = 0, o_a = o_s + H * ds, o_r = o_a + H * nu, o_c = o_r + H * nr, o_tr = o_c + H, o_t = (o_tr + H * ntr + 1) & ~(size_t)1,
               total = o_t + 2 * H;
  if (total > h->bcast_floats) return fail(MJPC_B200_ERR_CAPACITY, "fetch_trajectory_sharded: horizon above capacity");
  if (owner == h->rank) {
    const size_t i = candidate - lo;
    auto cp = [&](size_t off, const void* src, size_t bytes) { return cudaMemcpyAsync(b + off, src, bytes, cudaMemcpyDeviceToDevice, h->stream); };
    CUDA_TRY(cp(o_s, h->d_states + i * H * ds, H * ds * 4)); CUDA_TRY(cp(o_a, h->d_actions + i * H * nu, H * nu * 4));
    CUDA_TRY(cp(o_r, h->d_residual + i * H * nr, H * nr * 4)); CUDA_TRY(cp(o_c, h->d_costs + i * H, H * 4));
    if (ntr) CUDA_TRY(cp(o_tr, h->d_trace + i * H * ntr, H * ntr * 4));
    CUDA_TRY(cp(o_t, h->d_times + i * H, H * 8));
  }
  NCCL_TRY(nccl_api().Broadcast(b, b, total, ncclFloat, owner, h->comm, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  auto get = [&](void* dst, size_t off, size_t bytes) { return dst ? cudaMemcpy(dst, b + off, bytes, cudaMemcpyDeviceToHost) : cudaSuccess; };
  CUDA_TRY(get(states, o_s, H * ds * 4)); CUDA_TRY(get(actions, o_a, H * nu * 4)); CUDA_TRY(get(residual, o_r, H * nr * 4));
  CUDA_TRY(get(costs, o_c, H * 4)); CUDA_TRY(get(trace, o_tr, H * ntr * 4)); CUDA_TRY(get(times, o_t, H * 8));
  return 0;
}

// Batched single-step parity hook (see step_batch_kernel): B tuples -> one mj_step each.  times are absolute; the task
// state is rebased to `time0` exactly as a rollout starting at time0 would (device time = times[b] - time0).
int mjpc_b200_step_batch(mjpc_b200_t* h, int B, const float* qpos, const float* qvel, const float* ctrl,
                         const float* warmstart, const float* mocap, double time0, const double* times, float* qacc,
                         float* next_qpos, float* next_qvel, float* residual, float* cost, int* counts) {
  if (!h || B < 1 || !qpos || !qvel || !ctrl || !times) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "step_batch: bad argument");
  const DevModel& M = h->pack.M;
  if (M.nmocap && !mocap) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "step_batch: mocap required");
  CUDA_TRY(cudaSetDevice(h->device));
  const size_t nq = M.nq, nv = M.nv, nu = M.nu, nr = std::max(M.num_residual, 1), nm = 7 * (size_t)M.nmocap,
               nts = (size_t)M.task_state_size;
  const size_t per = nq + nv + nu + nv + 1 + nv + nq + nv + nr + 1 + 4;
  const size_t words = per * (size_t)B + nm + nts + 16;
  float* d = nullptr;
  CUDA_TRY(dalloc(&d, words));
  struct Guard { float* p; ~Guard() { cudaFree(p); } } guard{d};
  float *d_qpos = d, *d_qvel = d_qpos + B * nq, *d_ctrl = d_qvel + B * nv, *d_warm = d_ctrl + B * nu, *d_time = d_warm + B * nv,
        *d_qacc = d_time + B, *d_nq = d_qacc + B * nv, *d_nv = d_nq + B * nq, *d_res = d_nv + B * nv, *d_cost = d_res + B * nr,
        *d_counts = d_cost + B, *d_mocap = d_counts + 4 * (size_t)B, *d_ts = d_mocap + nm;
  std::vector<float> trel(B), ts(nts);
  for (int i = 0; i < B; i++) trel[i] = (float)(times[i] - time0);
  for (size_t i = 0; i < nts; i++) {
    double v = h->task_state[i];
    if (std::find(h->time_idx.begin(), h->time_idx.end(), (int)i) != h->time_idx.end()) v -= time0;
    ts[i] = (float)v;
  }
  CUDA_TRY(cudaMemcpy(d_qpos, qpos, B * nq * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_qvel, qvel, B * nv * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_ctrl, ctrl, B * nu * 4, cudaMemcpyHostToDevice));
  if (warmstart) CUDA_TRY(cudaMemcpy(d_warm, warmstart, B * nv * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_time, trel.data(), (size_t)B * 4, cudaMemcpyHostToDevice));
  if (nm) CUDA_TRY(cudaMemcpy(d_mocap, mocap, nm * 4, cudaMemcpyHostToDevice));
  if (nts) CUDA_TRY(cudaMemcpy(d_ts, ts.data(), nts * 4, cudaMemcpyHostToDevice));
  StepBatchArgs A;
  std::memset(&A, 0, sizeof(A));
  A.M = h->pack.M; A.L = make_layout(h->pack.M, 1); A.pack = h->d_pack;
  A.qpos = d_qpos; A.qvel = d_qvel; A.ctrl = d_ctrl; A.warmstart = warmstart ? d_warm : nullptr; A.mocap = d_mocap;
  A.task_state = nts ? d_ts : nullptr; A.time = d_time; A.B = B;
  A.qacc = d_qacc; A.next_qpos = d_nq; A.next_qvel = d_nv; A.residual = d_res; A.cost = d_cost; A.counts = (int*)d_counts;
  const size_t smem = h->smem_bytes(1, 1);
  const char* ns = std::getenv("MJPC_B200_NO_STATIC");
  const bool use_static = h->static_spec != 0 && !(ns && ns[0] == '1');
  const void* fn = use_static ? (h->static_spec == 1 ? (const void*)step_batch_kernel_quadruped : (const void*)step_batch_kernel_humanoid_track)
                              : (const void*)step_batch_kernel;
  if (int rc = set_smem(fn, smem)) return rc;
  CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
  if (use_static && h->static_spec == 1) step_batch_kernel_quadruped<<<B, 32, smem, h->stream>>>(A);
  else if (use_static) step_batch_kernel_humanoid_track<<<B, 32, smem, h->stream>>>(A);
  else step_batch_kernel<<<B, 32, smem, h->stream>>>(A);
  CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  h->last_static = use_static ? 1 : 0;
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  if (cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1) != cudaSuccess) cudaGetLastError();
  if (qacc) CUDA_TRY(cudaMemcpy(qacc, d_qacc, B * nv * 4, cudaMemcpyDeviceToHost));
  if (next_qpos) CUDA_TRY(cudaMemcpy(next_qpos, d_nq, B * nq * 4, cudaMemcpyDeviceToHost));
  if (next_qvel) CUDA_TRY(cudaMemcpy(next_qvel, d_nv, B * nv * 4, cudaMemcpyDeviceToHost));
  if (residual) CUDA_TRY(cudaMemcpy(residual, d_res, B * (size_t)M.num_residual * 4, cudaMemcpyDeviceToHost));
  if (cost) CUDA_TRY(cudaMemcpy(cost, d_cost, (size_t)B * 4, cudaMemcpyDeviceToHost));
  if (counts) CUDA_TRY(cudaMemcpy(counts, d_counts, (size_t)B * 16, cudaMemcpyDeviceToHost));
  return 0;
}

int mjpc_b200_fetch_stats(mjpc_b200_t* h, int64_t* stats) {
  if (!h || !stats || h->lastN < 1) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "fetch_stats: nothing to fetch");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaMemcpy(stats, h->d_stats, (size_t)h->lastN * 12 * sizeof(long long), cudaMemcpyDeviceToHost));
  return 0;
}

// NoisyRollout (mjpc/trajectory.cc:100-210) for the following rollouts of this handle: Ornstein-Uhlenbeck
// xfrc_applied noise with stationary std `xfrc_std` [N, N m] and correlation time `xfrc_rate` [s]; 0 switches it off.
int mjpc_b200_set_xfrc_noise(mjpc_b200_t* h, double xfrc_std, double xfrc_rate, uint32_t seed) {
  if (!h || xfrc_std < 0 || !(xfrc_rate > 0)) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "set_xfrc_noise: bad argument");
  h->xfrc_std = (float)xfrc_std; h->xfrc_rate = (float)xfrc_rate; h->noise_seed = seed;
  h->resident_ok = false;
  return MJPC_B200_OK;
}

int64_t mjpc_b200_launch_count(const mjpc_b200_t* h) { return h ? h->launches : 0; }
float mjpc_b200_last_kernel_ms(const mjpc_b200_t* h) { return h ? h->last_ms : 0.f; }
int mjpc_b200_last_kernel_static(const mjpc_b200_t* h) { return h ? h->last_static : 0; }

// Header + state-layout words of a model, as the static kernel tables (spec_*.h) store them.  Host only.
int mjpc_b200_spec_words(const mjpc_model_blob* model, int* out, int capacity) {
  if (!model || !model->data || !out) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "spec_words: null");
  try {
    ModelPack P = pack_model(model->data, model->nbytes, 32, 96);
    const DevLayout L = make_layout(P.M, 1);
    const int nm = (int)(sizeof(DevModel) / 4), nl = (int)D_COUNT;
    if (capacity < 2 + nm + nl) return fail(MJPC_B200_ERR_CAPACITY, "spec_words: buffer too small");
    out[0] = nm; out[1] = nl;
    std::memcpy(out + 2, &P.M, sizeof(DevModel));
    for (int i = 0; i < nl; i++) out[2 + nm + i] = L.off[i];
    return 2 + nm + nl;
  } catch (const std::exception& e) {
    return fail(MJPC_B200_ERR_BAD_BLOB, std::string("spec_words: ") + e.what());
  }
}
void* mjpc_b200_stream(mjpc_b200_t* h) { return h ? (void*)h->stream : nullptr; }
float* mjpc_b200_device_returns(mjpc_b200_t* h) { return h ? h->d_returns : nullptr; }

// ---- iLQG entry points (kernels in ilqg_kernels.cuh)
int mjpc_b200_model_derivatives(mjpc_b200_t* h, const float* x, const float* u, const double* t, const float* mocap,
                                int H, int skip, float tol, int mode, float* A, float* B, float* C, float* D) {
  if (!h || !x || !u || !t || !A || !B || !C || !D) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "model_derivatives: null");
  if (H < 1 || H > h->maxH || !(tol > 0)) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "model_derivatives: bad H or tol");
  if (skip < 0 || mode < 0 || mode > 1) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "model_derivatives: bad skip or mode");
  if (h->pack.M.nmocap && !mocap) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "model_derivatives: mocap required");
  CUDA_TRY(cudaSetDevice(h->device));
  std::vector<float> ts(h->pack.M.task_state_size), trel(H);
  // derivative sweeps use absolute-time task state rebased to t[0]
  for (size_t i = 0; i < ts.size(); i++) {
    double v = h->task_state[i];
    if (std::find(h->time_idx.begin(), h->time_idx.end(), (int)i) != h->time_idx.end()) v -= t[0];
    ts[i] = (float)v;
  }
  for (int i = 0; i < H; i++) trel[i] = (float)(t[i] - t[0]);
  int launches = 0;
  int rc = ilqg_model_derivatives(h->ilqg, h->pack.M, h->d_pack, h->stream, x, u, trel.data(), mocap, ts.data(), H, tol,
                                  A, B, C, D, h->smem_bytes(1, 1), &launches, h->ev0, h->ev1, skip, mode);
  h->launches += launches;
  if (rc == 0 && cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1) != cudaSuccess) cudaGetLastError();
  if (rc) return fail(rc, "model_derivatives: CUDA failure");
  return 0;
}

int mjpc_b200_cost_derivatives(mjpc_b200_t* h, const float* residual, const float* C, const float* D, int H,
                               float* cx, float* cu, float* cxx, float* cuu, float* cxu) {
  if (!h || !residual || !C || !D || !cx || !cu || !cxx || !cuu || !cxu)
    return fail(MJPC_B200_ERR_BAD_ARGUMENT, "cost_derivatives: null");
  if (H < 1 || H > h->maxH) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "cost_derivatives: bad H");
  CUDA_TRY(cudaSetDevice(h->device));
  int launches = 0;
  int rc = ilqg_cost_derivatives(h->ilqg, h->pack.M, h->d_pack, h->stream, residual, C, D, H, cx, cu, cxx, cuu, cxu, &launches, h->ev0, h->ev1);
  h->launches += launches;
  if (rc == 0 && cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1) != cudaSuccess) cudaGetLastError();
  if (rc) return fail(rc, "cost_derivatives: CUDA failure");
  return 0;
}

int mjpc_b200_backward_pass(mjpc_b200_t* h, const float* A, const float* B, const float* cx, const float* cu,
                            const float* cxx, const float* cxu, const float* cuu, const float* actions, int H,
                            float mu, int reg_type, int limits, float* K, float* du, float* dV, float* Vx, float* Vxx,
                            int* status_out) {
  if (!h || !A || !B || !cx || !cu || !cxx || !cxu || !cuu || !actions || !K || !du || !dV || !status_out)
    return fail(MJPC_B200_ERR_BAD_ARGUMENT, "backward_pass: null");
  if (H < 2 || H > h->maxH) return fail(MJPC_B200_ERR_BAD_ARGUMENT, "backward_pass: bad H");
  CUDA_TRY(cudaSetDevice(h->device));
  int launches = 0;
  int rc = ilqg_backward_pass(h->ilqg, h->pack.M, h->d_pack, h->stream, A, B, cx, cu, cxx, cxu, cuu, actions, H, mu,
                              reg_type, limits, K, du, dV, Vx, Vxx, status_out, &launches, h->ev0, h->ev1);
  h->launches += launches;
  if (rc == 0 && cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1) != cudaSuccess) cudaGetLastError();
  if (rc) return fail(rc, "backward_pass: CUDA failure");
  return 0;
}

}  // extern "C"
