// mb200.cu -- the C ABI declared in include/mocca_b200.h over the per-kind kernel tables (csrc/kinds/*.cu).
// One warp per environment, MB_WARPS warps per CTA; per-env working set lives in shared memory (WarpMem).
//
// 14 warps (envs) per CTA, 2 CTAs per SM, and one CTA barrier per substep (MB_SYNC): the barrier keeps the warps of a
// CTA in the same phase of the (large) step code so instruction-cache lines are shared (profiles/README.md).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>

#include "../../include/mocca_b200.h"
#include "mb_kind.cuh"

static thread_local std::string g_err;
static int fail(const std::string& m) { g_err = m; return -1; }
#define CUDA_OK(x)                                                                                       \
  do {                                                                                                   \
    cudaError_t e_ = (x);                                                                                \
    if (e_ != cudaSuccess) return fail(std::string(#x) + ": " + cudaGetErrorString(e_));                 \
  } while (0)

// Every kernel table (csrc/kinds/*.cu).  An env id runs its "" variant; plank_class = Pillar switches a stepper
// batch to its "pillar" variant (the cylinder-stone instantiation).
extern const MbKindOps mb_kind_walker3d_custom, mb_kind_walker3d_stepper, mb_kind_walker3d_stepper_pillar,
    mb_kind_monkey3d_custom, mb_kind_cassie, mb_kind_child3d_custom, mb_kind_walker2d_custom, mb_kind_crab2d_custom,
    mb_kind_mike_stepper, mb_kind_mike_stepper_pillar;
static const MbKindOps* const g_kinds[] = {
    &mb_kind_walker3d_custom, &mb_kind_walker3d_stepper, &mb_kind_walker3d_stepper_pillar, &mb_kind_monkey3d_custom,
    &mb_kind_cassie,          &mb_kind_child3d_custom,   &mb_kind_mike_stepper,            &mb_kind_mike_stepper_pillar,
    &mb_kind_walker2d_custom, &mb_kind_crab2d_custom,
};

static const MbKindOps* find_kind(const char* env_id, const char* variant) {
  if (env_id)
    for (const MbKindOps* k : g_kinds)
      if (strcmp(k->env_id, env_id) == 0 && strcmp(k->variant, variant) == 0) return k;
  return nullptr;
}

struct mb200_env {
  const MbKindOps* ops;  // the kernels this batch launches
  int warps;       // envs per CTA of this kind's kernels
  int rec_stride;  // floats per env in `rec`
  int n, device;
  int obs_dim, act_dim, state_dim, nu;
  MbPhysics phys;
  float* state;     // [n][MB_STATE_STRIDE]
  float* rec;       // [n][MB_REC_STRIDE]
  uint32_t* mt;     // [n][2][MB_MT_STRIDE]
  MbStats* stats;   // device
  float* stage_act; // device staging for the host-buffer entry point
  float* stage_obs;
  float* stage_rew;
  uint8_t* stage_done;
  uint8_t* stage_trunc;
  uint8_t* stage_mask;   // mb200_reset_host
  int* info;             // [n] per-step integer info (steps_reached), written by the step kernel
  float* warm;           // [n_pad][MB_NWARM] warm-start impulses (allocated when phys.warmstart > 0)
  cudaEvent_t host_done; // results of mb200_step_host have reached the host buffers
  // CTA barriers require every warp of a CTA to run: the state arrays are padded to a whole number of CTAs and
  // the pad envs ("tail") step like any other env but write their outputs/statistics to these dummies
  int n_pad;
  float* dummy_obs;    // [MB_WARPS_MAX][obs_dim] x2 (obs, final_obs)
  float* dummy_rew;    // [MB_WARPS_MAX]
  uint8_t* dummy_flag; // [2][MB_WARPS_MAX]
  MbStats* dummy_stats;
  // work-sorted slot -> env map: the warps of a CTA meet at one barrier per substep, so a CTA runs at the pace of
  // its slowest env; grouping envs with similar constraint-row counts (of the previous step) removes most of that
  // wait, and heavy CTAs are scheduled first.  Pure scheduling: every env's arithmetic is unchanged.
  // The step kernel itself classifies: each warp turns the rows of its step into a key (heaviest = 0), stores it and
  // counts it in a 256-bin histogram (global atomics spread over the launch); a small multi-CTA kernel then scans
  // the bins and scatters the env ids (k_order_by_key, ~10 us instead of the 38 us of a single-CTA counting sort).
  int* order;      // [n_pad]
  int* key;        // [n_pad] sort key of the last step
  int* hist;       // [2][256] step t counts into hist[t & 1]; the scatter kernel zeroes the other half
  int* cursor;     // [2][256] scatter cursors, same double buffering
  int sort_every;  // 0 = never re-sort (identity order), otherwise after every step
  float* render_scene;  // [render_cap][MB_RMAX][MB_RSTRIDE] primitive lists of mb200_render's scene pass
  int render_cap;       // cameras the scene buffer holds
  long long steps;
  long long launches;
  size_t smem;
};

// ------------------------------------------------------------------------------------------------ kernels
// Second half of the counting sort (the histogram was filled by the step kernel): every CTA scans the 256 bins into
// bin starts, then places its 256 envs with warp-aggregated global cursors.  Order inside a bin is arbitrary (pure
// scheduling).  CTA 0 also clears the other halves of hist / cursor for the next step.
__global__ void __launch_bounds__(256) k_order_by_key(int n_pad, const int* key, const int* hist, int* cursor,
                                                       int* hist_next, int* cursor_next, int* order) {
  __shared__ int start[256];
  __shared__ int wsum[8];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int h = hist[tid];
  int incl = h;
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) wsum[wid] = incl;
  __syncthreads();
  int base = 0;
  for (int w = 0; w < wid; ++w) base += wsum[w];
  start[tid] = base + incl - h;
  if (blockIdx.x == 0) { hist_next[tid] = 0; cursor_next[tid] = 0; }
  __syncthreads();
  const int e = blockIdx.x * 256 + tid;
  const int k = e < n_pad ? key[e] : 256 + lane;  // out of range: a key nobody shares
  const unsigned peers = __match_any_sync(0xffffffffu, k);
  const int leader = __ffs(peers) - 1;
  int off = 0;
  if (k < 256 && lane == leader) off = atomicAdd(&cursor[k], __popc(peers));
  off = __shfl_sync(0xffffffffu, off, leader);
  if (k < 256) order[start[k] + off + __popc(peers & ((1u << lane) - 1u))] = e;
}

__global__ void k_copy_strided(int n, int width, const float* src, int src_stride, float* dst, int dst_stride) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * width) return;
  const int e = i / width, k = i % width;
  dst[(size_t)e * dst_stride + k] = src[(size_t)e * src_stride + k];
}

// FP32 FMA throughput probe: the roofline denominator for this (CUDA-core bound) path, measured on the same
// device in the same process as the benchmark (MEASURED_PEAKS.json only carries HBM and tensor-core peaks).
__global__ void __launch_bounds__(256) k_fma_probe(float* out, int iters, float b, float c) {
  float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f,
        a6 = a0 + 6.f, a7 = a0 + 7.f;
#pragma unroll 4
  for (int i = 0; i < iters; ++i) {
    a0 = fmaf(a0, b, c); a1 = fmaf(a1, b, c); a2 = fmaf(a2, b, c); a3 = fmaf(a3, b, c);
    a4 = fmaf(a4, b, c); a5 = fmaf(a5, b, c); a6 = fmaf(a6, b, c); a7 = fmaf(a7, b, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

const char* mb200_last_error(void) { return g_err.c_str(); }

void mb200_default_physics(mb200_physics* p) { mb_default_physics(p); }

void mb200_default_physics_for(const char* env_id, mb200_physics* p) {
  mb_default_physics(p);
  if (const MbKindOps* K = find_kind(env_id, "")) K->default_physics(*p);
}

static int grid_for(const mb200_env* e) { return (e->n + e->warps - 1) / e->warps; }

// the device arrays of a new handle, all zeroed (info: -1 = not reported) except the identity launch order
static int alloc_buffers(mb200_env* e) {
  const size_t n = (size_t)e->n_pad;
  CUDA_OK(cudaMalloc(&e->dummy_obs, (size_t)2 * MB_WARPS_MAX * e->obs_dim * sizeof(float)));
  CUDA_OK(cudaMalloc(&e->dummy_rew, MB_WARPS_MAX * sizeof(float)));
  CUDA_OK(cudaMalloc(&e->dummy_flag, 2 * MB_WARPS_MAX));
  CUDA_OK(cudaMalloc(&e->dummy_stats, sizeof(MbStats)));
  CUDA_OK(cudaMemset(e->dummy_stats, 0, sizeof(MbStats)));
  CUDA_OK(cudaMalloc(&e->state, n * MB_STATE_STRIDE * sizeof(float)));
  CUDA_OK(cudaMalloc(&e->rec, n * e->rec_stride * sizeof(float)));
  CUDA_OK(cudaMalloc(&e->mt, n * 2 * MB_MT_STRIDE * sizeof(uint32_t)));
  CUDA_OK(cudaMalloc(&e->stats, sizeof(MbStats)));
  CUDA_OK(cudaMalloc(&e->order, n * sizeof(int)));
  CUDA_OK(cudaMalloc(&e->key, n * sizeof(int)));
  CUDA_OK(cudaMalloc(&e->hist, 2 * 256 * sizeof(int)));
  CUDA_OK(cudaMalloc(&e->cursor, 2 * 256 * sizeof(int)));
  CUDA_OK(cudaMemset(e->key, 0, n * sizeof(int)));
  CUDA_OK(cudaMemset(e->hist, 0, 2 * 256 * sizeof(int)));
  CUDA_OK(cudaMemset(e->cursor, 0, 2 * 256 * sizeof(int)));
  {
    int* ident = (int*)malloc(n * sizeof(int));
    if (!ident) return fail("mb200_create: host allocation failed");
    for (size_t i = 0; i < n; ++i) ident[i] = (int)i;
    cudaError_t ce = cudaMemcpy(e->order, ident, n * sizeof(int), cudaMemcpyHostToDevice);
    free(ident);
    CUDA_OK(ce);
  }
  CUDA_OK(cudaMalloc(&e->stage_act, n * e->act_dim * sizeof(float)));
  CUDA_OK(cudaMalloc(&e->stage_obs, n * e->obs_dim * sizeof(float)));
  CUDA_OK(cudaMalloc(&e->stage_rew, n * sizeof(float)));
  CUDA_OK(cudaMalloc(&e->stage_done, n));
  CUDA_OK(cudaMalloc(&e->stage_trunc, n));
  CUDA_OK(cudaEventCreateWithFlags(&e->host_done, cudaEventDisableTiming));
  CUDA_OK(cudaMemset(e->state, 0, n * MB_STATE_STRIDE * sizeof(float)));
  CUDA_OK(cudaMemset(e->rec, 0, n * e->rec_stride * sizeof(float)));
  CUDA_OK(cudaMemset(e->mt, 0, n * 2 * MB_MT_STRIDE * sizeof(uint32_t)));
  CUDA_OK(cudaMemset(e->stats, 0, sizeof(MbStats)));
  CUDA_OK(cudaMalloc(&e->stage_mask, n));
  if (e->phys.warmstart > 0.0f) {
    CUDA_OK(cudaMalloc(&e->warm, n * MB_NWARM * sizeof(float)));
    CUDA_OK(cudaMemset(e->warm, 0, n * MB_NWARM * sizeof(float)));
  }
  CUDA_OK(cudaMalloc(&e->info, n * sizeof(int)));
  CUDA_OK(cudaMemset(e->info, 0xff, n * sizeof(int)));
  return 0;
}

void mb200_destroy(mb200_env* e);

int mb200_create(const char* env_id, int n_envs, int device, const mb200_physics* physics, mb200_env** out) {
  if (!out) return fail("mb200_create: out is NULL");
  *out = nullptr;
  const MbKindOps* K = find_kind(env_id, "");
  if (!K) {
    std::string built;
    for (const MbKindOps* k : g_kinds)
      if (!*k->variant) built += (built.empty() ? "" : ", ") + std::string(k->env_id);
    return fail(std::string("mb200_create: unsupported env id '") + (env_id ? env_id : "(null)") + "' (built: " +
                built + ")");
  }
  if (n_envs <= 0) return fail("mb200_create: n_envs must be positive");
  int count = 0;
  CUDA_OK(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail("mb200_create: no such CUDA device");
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail("mb200_create: device is not compute capability 10.x; this library carries sm_100a code only and has "
                "no CPU or other-arch fallback");
  CUDA_OK(cudaSetDevice(device));
  // opt every kernel of the env id (each variant) in to the dynamic shared memory of a full-width CTA (the attribute
  // is per kernel, not per handle, and several env kinds can live in one process)
  for (const MbKindOps* k : g_kinds)
    if (strcmp(k->env_id, env_id) == 0) {
      const cudaError_t pe = k->prepare();
      if (pe != cudaSuccess) return fail(std::string("mb200_create: shared-memory opt-in: ") + cudaGetErrorString(pe));
    }
  mb200_env* e = new mb200_env();
  memset(e, 0, sizeof(*e));
  e->n = n_envs;
  e->device = device;
  e->ops = K;
  const int nj = K->nj;
  e->rec_stride = K->rec_stride; e->obs_dim = K->obs_dim; e->act_dim = K->act_dim;
  e->warps = K->warps;
  {
    // Small batches: with 14-warp CTAs 1 024 envs occupy 74 of the 148 SMs and the step takes the latency of one
    // env-step; narrower CTAs spread the envs over every SM (2 resident CTAs each).  Pure scheduling (MB_WARPS is the
    // launch's own blockDim), results are unchanged.  MB200_WARPS overrides (tuning / A-B runs).
    const int slots = MB_MINBLOCKS * prop.multiProcessorCount;
    int w = (n_envs + slots - 1) / slots;
    if (w < 4) w = 4;
    if (w < e->warps) e->warps = w;
    if (const char* ov = getenv("MB200_WARPS")) {
      const int v = atoi(ov);
      if (v >= 1 && v <= e->warps) e->warps = v;  // never above the launch bounds the step kernels were compiled with
    }
  }
  e->state_dim = 13 + 2 * nj;
  e->nu = 6 + nj;
  mb200_physics p;
  mb200_default_physics_for(env_id, &p);
  if (physics) p = *physics;
  mb_to_internal(p, &e->phys);
  K->fix_physics(e->phys);
  e->smem = K->smem_per_env * e->warps;
  e->n_pad = grid_for(e) * e->warps;
  e->sort_every = 1;
  if (const char* sv = getenv("MB200_SORT_EVERY")) e->sort_every = atoi(sv);
  if (alloc_buffers(e)) {
    mb200_destroy(e);
    return -1;
  }
  *out = e;
  return 0;
}

void mb200_destroy(mb200_env* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaFree(e->state); cudaFree(e->rec); cudaFree(e->mt); cudaFree(e->stats);
  cudaFree(e->stage_act); cudaFree(e->stage_obs); cudaFree(e->stage_rew); cudaFree(e->stage_done);
  cudaFree(e->stage_trunc); cudaFree(e->stage_mask); cudaFree(e->info); cudaFree(e->warm);
  if (e->host_done) cudaEventDestroy(e->host_done);
  cudaFree(e->dummy_obs); cudaFree(e->dummy_rew); cudaFree(e->dummy_flag); cudaFree(e->dummy_stats);
  cudaFree(e->order); cudaFree(e->key); cudaFree(e->hist); cudaFree(e->cursor);
  cudaFree(e->render_scene);
  delete e;
}

int mb200_dims(const mb200_env* e, int* n_envs, int* obs_dim, int* act_dim, int* state_dim, int* nu) {
  if (!e) return fail("mb200_dims: NULL handle");
  if (n_envs) *n_envs = e->n;
  if (obs_dim) *obs_dim = e->obs_dim;
  if (act_dim) *act_dim = e->act_dim;
  if (state_dim) *state_dim = e->state_dim;
  if (nu) *nu = e->nu;
  return 0;
}

int mb200_seed(mb200_env* e, const uint32_t* mt_host, int at_construction) {
  if (!e || !mt_host) return fail("mb200_seed: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaDeviceSynchronize());
  const size_t n = (size_t)e->n_pad, nreal = (size_t)e->n;
  uint32_t* tmp = (uint32_t*)calloc(n * 2 * MB_MT_STRIDE, sizeof(uint32_t));
  float* rec = (float*)malloc(n * e->rec_stride * sizeof(float));
  if (!tmp || !rec) { free(tmp); free(rec); return fail("mb200_seed: host allocation failed"); }
  if (!at_construction)
    CUDA_OK(cudaMemcpy(tmp, e->mt, n * 2 * MB_MT_STRIDE * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(rec, e->rec, n * e->rec_stride * sizeof(float), cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; ++i) {
    int& aliased = reinterpret_cast<int*>(rec + i * e->rec_stride)[ER_ALIASED];
    uint32_t* env_mt = tmp + (i * 2) * MB_MT_STRIDE;
    uint32_t* robot_mt = env_mt + MB_MT_STRIDE;
    if (at_construction) {
      robot_mt[624] = 624;  // the robot draws from the env's stream (env_base.py:93)
      aliased = 1;
    } else if (aliased) {
      // EnvBase.seed rebinds only the env's RandomState: an aliased robot keeps drawing from the OLD stream,
      // which therefore moves to the robot slot (quirk Q1)
      memcpy(robot_mt, env_mt, 625 * sizeof(uint32_t));
      aliased = 0;
    }
    memcpy(env_mt, mt_host + (i % nreal) * 625, 625 * sizeof(uint32_t));
  }
  CUDA_OK(cudaMemcpy(e->mt, tmp, n * 2 * MB_MT_STRIDE * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(e->rec, rec, n * e->rec_stride * sizeof(float), cudaMemcpyHostToDevice));
  free(tmp);
  free(rec);
  return 0;
}

int mb200_reset(mb200_env* e, const uint8_t* mask_dev, float* obs_dev, void* stream) {
  if (!e || !obs_dev) return fail("mb200_reset: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  const LaunchDims d = {grid_for(e), e->warps * 32, e->smem, (cudaStream_t)stream};
  e->ops->reset(d, e->n, e->phys, e->state, e->rec, e->mt, mask_dev, obs_dev, e->dummy_obs, e->warm);
  e->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// Env.reset with HOST buffers (what a gym user holds): mask_host NULL = all envs.  Only the rows of the envs that
// were reset are written to obs_host.  Synchronous.
int mb200_reset_host(mb200_env* e, const uint8_t* mask_host, float* obs_host, void* stream) {
  if (!e || !obs_host) return fail("mb200_reset_host: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)e->n, row = (size_t)e->obs_dim * sizeof(float);
  if (mask_host) CUDA_OK(cudaMemcpyAsync(e->stage_mask, mask_host, n, cudaMemcpyHostToDevice, st));
  if (mb200_reset(e, mask_host ? e->stage_mask : nullptr, e->stage_obs, stream)) return -1;
  if (!mask_host) {
    CUDA_OK(cudaMemcpyAsync(obs_host, e->stage_obs, n * row, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    return 0;
  }
  float* tmp = (float*)malloc(n * row);
  if (!tmp) return fail("mb200_reset_host: host allocation failed");
  cudaError_t ce = cudaMemcpyAsync(tmp, e->stage_obs, n * row, cudaMemcpyDeviceToHost, st);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
  if (ce != cudaSuccess) { free(tmp); return fail(std::string("mb200_reset_host: ") + cudaGetErrorString(ce)); }
  for (size_t i = 0; i < n; ++i)
    if (mask_host[i]) memcpy(obs_host + i * e->obs_dim, tmp + i * e->obs_dim, row);
  free(tmp);
  return 0;
}

// info dict of the last mb200_step / mb200_step_host as integers, one per env: Walker3DStepperEnv / MikeStepperEnv
// info["steps_reached"] (env_locomotion.py:505-506; -1 = the step did not report it), -1 for the other envs.
int mb200_info(mb200_env* e, int* info_dev, void* stream) {
  if (!e || !info_dev) return fail("mb200_info: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaMemcpyAsync(info_dev, e->info, (size_t)e->n * sizeof(int), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}
int mb200_info_host(mb200_env* e, int* info_host, void* stream) {
  if (!e || !info_host) return fail("mb200_info_host: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaMemcpyAsync(info_host, e->info, (size_t)e->n * sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

static bool sorting(const mb200_env* e) { return e->sort_every > 0 && grid_for(e) > 1; }

// scatter for the step that was just launched (e->steps already counts it)
static int launch_sort(mb200_env* e, void* stream) {
  if (sorting(e)) {
    const int b = (int)((e->steps - 1) & 1);
    k_order_by_key<<<(e->n_pad + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        e->n_pad, e->key, e->hist + 256 * b, e->cursor + 256 * b, e->hist + 256 * (b ^ 1), e->cursor + 256 * (b ^ 1),
        e->order);
    e->launches++;
  }
  CUDA_OK(cudaGetLastError());
  return 0;
}

struct HostOut {
  float* obs;
  float* rew;
  uint8_t* done;
  uint8_t* trunc;
};

static int step_impl(mb200_env* e, const float* act_dev, float* obs_dev, float* rew_dev, uint8_t* done_dev,
                     uint8_t* trunc_dev, float* final_obs_dev, void* stream, bool sort_now,
                     const HostOut* host = nullptr) {
  if (!e || !act_dev || !obs_dev || !rew_dev || !done_dev || !trunc_dev) return fail("mb200_step: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  StepArgs a;
  a.n = e->n; a.phys = e->phys; a.state = e->state; a.rec = e->rec; a.mt = e->mt; a.act = act_dev; a.obs = obs_dev;
  a.rew = rew_dev; a.done = done_dev; a.trunc = trunc_dev; a.final_obs = final_obs_dev; a.stats = e->stats;
  a.dummy_obs = e->dummy_obs; a.dummy_rew = e->dummy_rew; a.dummy_flag = e->dummy_flag; a.dummy_stats = e->dummy_stats;
  a.order = e->order; a.key = e->key;
  a.hist = sorting(e) ? e->hist + 256 * (int)(e->steps & 1) : nullptr;
  a.host_obs = host ? host->obs : nullptr; a.host_rew = host ? host->rew : nullptr;
  a.host_done = host ? host->done : nullptr; a.host_trunc = host ? host->trunc : nullptr;
  a.info = e->info;
  a.warm = e->warm;
  const LaunchDims d = {grid_for(e), e->warps * 32, e->smem, (cudaStream_t)stream};
  e->ops->step(a, host != nullptr, d);
  e->launches++;
  e->steps++;
  CUDA_OK(cudaGetLastError());
  return sort_now ? launch_sort(e, stream) : 0;
}

int mb200_step(mb200_env* e, const float* act_dev, float* obs_dev, float* rew_dev, uint8_t* done_dev,
               uint8_t* trunc_dev, float* final_obs_dev, void* stream) {
  return step_impl(e, act_dev, obs_dev, rew_dev, done_dev, trunc_dev, final_obs_dev, stream, true);
}

// device alias of a pinned / registered host buffer (UVA), nullptr for pageable memory
static void* mapped_alias(const void* host) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (at.type != cudaMemoryTypeHost) return nullptr;
  return at.devicePointer;
}

// MB200_HOST_DIRECT: 0 = always stage through device buffers + cudaMemcpyAsync; 1 = results go to pinned host buffers
// by zero-copy stores from the step kernel; 2 (default) = also read the actions from the pinned host buffer in place
static int host_direct_mode() {
  static int mode = -1;
  if (mode < 0) {
    const char* s = getenv("MB200_HOST_DIRECT");
    mode = s && *s ? atoi(s) : 2;
  }
  return mode;
}

int mb200_step_host(mb200_env* e, const float* act_host, float* obs_host, float* rew_host, uint8_t* done_host,
                    uint8_t* trunc_host, void* stream) {
  if (!e || !act_host || !obs_host || !rew_host || !done_host || !trunc_host)
    return fail("mb200_step_host: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)e->n;
  const int mode = host_direct_mode();
  HostOut ho = {nullptr, nullptr, nullptr, nullptr};
  if (mode >= 1) {
    ho.obs = (float*)mapped_alias(obs_host); ho.rew = (float*)mapped_alias(rew_host);
    ho.done = (uint8_t*)mapped_alias(done_host); ho.trunc = (uint8_t*)mapped_alias(trunc_host);
  }
  const bool direct_out = ho.obs && ho.rew && ho.done && ho.trunc;
  const float* act_dev = mode >= 2 && direct_out ? (const float*)mapped_alias(act_host) : nullptr;
  if (!act_dev) {
    CUDA_OK(cudaMemcpyAsync(e->stage_act, act_host, n * e->act_dim * sizeof(float), cudaMemcpyHostToDevice, st));
    act_dev = e->stage_act;
  }
  int rc = step_impl(e, act_dev, e->stage_obs, e->stage_rew, e->stage_done, e->stage_trunc, nullptr, stream, false,
                     direct_out ? &ho : nullptr);
  if (rc) return rc;
  if (!direct_out) {
    CUDA_OK(cudaMemcpyAsync(obs_host, e->stage_obs, n * e->obs_dim * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(rew_host, e->stage_rew, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(done_host, e->stage_done, n, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(trunc_host, e->stage_trunc, n, cudaMemcpyDeviceToHost, st));
  }
  // the caller needs the results, not the scheduler's re-sort: wait for the results only (the event completes when
  // the kernel's zero-copy stores / the copies have landed) and let the sort of the next step's launch order run
  // while the host picks its actions
  CUDA_OK(cudaEventRecord(e->host_done, st));
  rc = launch_sort(e, stream);
  if (rc) return rc;
  CUDA_OK(cudaEventSynchronize(e->host_done));
  return 0;
}

static int copy_rows(mb200_env* e, const float* src, int ss, float* dst, int ds, int width, void* stream) {
  const int total = e->n * width;
  k_copy_strided<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(e->n, width, src, ss, dst, ds);
  e->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int mb200_get_state(mb200_env* e, float* state_dev, void* stream) {
  if (!e || !state_dev) return fail("mb200_get_state: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  return copy_rows(e, e->state, MB_STATE_STRIDE, state_dev, e->state_dim, e->state_dim, stream);
}
int mb200_set_state(mb200_env* e, const float* state_dev, void* stream) {
  if (!e || !state_dev) return fail("mb200_set_state: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  return copy_rows(e, state_dev, e->state_dim, e->state, MB_STATE_STRIDE, e->state_dim, stream);
}
int mb200_get_record(mb200_env* e, float* rec_dev, void* stream) {
  if (!e || !rec_dev) return fail("mb200_get_record: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaMemcpyAsync(rec_dev, e->rec, (size_t)e->n * e->rec_stride * sizeof(float), cudaMemcpyDeviceToDevice,
                          (cudaStream_t)stream));
  return 0;
}
int mb200_set_record(mb200_env* e, const float* rec_dev, void* stream) {
  if (!e || !rec_dev) return fail("mb200_set_record: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaMemcpyAsync(e->rec, rec_dev, (size_t)e->n * e->rec_stride * sizeof(float), cudaMemcpyDeviceToDevice,
                          (cudaStream_t)stream));
  return 0;
}

// warm-start impulses (phys.warmstart > 0): part of the checkpoint of a batch; width 0 = warm starting off
int mb200_warm_width(const mb200_env* e) { return e && e->warm ? MB_NWARM : 0; }
int mb200_get_warm(mb200_env* e, float* warm_dev, void* stream) {
  if (!e || !warm_dev || !e->warm) return fail("mb200_get_warm: NULL argument or warm starting off");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaMemcpyAsync(warm_dev, e->warm, (size_t)e->n * MB_NWARM * sizeof(float), cudaMemcpyDeviceToDevice,
                          (cudaStream_t)stream));
  return 0;
}
int mb200_set_warm(mb200_env* e, const float* warm_dev, void* stream) {
  if (!e || !warm_dev || !e->warm) return fail("mb200_set_warm: NULL argument or warm starting off");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaMemcpyAsync(e->warm, warm_dev, (size_t)e->n * MB_NWARM * sizeof(float), cudaMemcpyDeviceToDevice,
                          (cudaStream_t)stream));
  return 0;
}

int mb200_rng_words(const mb200_env* e) { return e ? 2 * MB_MT_STRIDE : 0; }
int mb200_get_rng(mb200_env* e, uint32_t* mt_host) {
  if (!e || !mt_host) return fail("mb200_get_rng: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaMemcpy(mt_host, e->mt, (size_t)e->n * 2 * MB_MT_STRIDE * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  return 0;
}
int mb200_set_rng(mb200_env* e, const uint32_t* mt_host) {
  if (!e || !mt_host) return fail("mb200_set_rng: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaMemcpy(e->mt, mt_host, (size_t)e->n * 2 * MB_MT_STRIDE * sizeof(uint32_t), cudaMemcpyHostToDevice));
  return 0;
}

static int step_physics_impl(mb200_env* e, const float* tau_dev, int* rows_dev, int* contacts_dev, float* points_dev,
                             void* stream) {
  if (!e || !tau_dev) return fail("mb200_step_physics: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  const LaunchDims d = {grid_for(e), e->warps * 32, e->smem, (cudaStream_t)stream};
  e->ops->physics(d, e->n, e->phys, e->state, e->rec, tau_dev, rows_dev, contacts_dev, points_dev, e->warm);
  e->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int mb200_step_physics(mb200_env* e, const float* tau_dev, int* rows_dev, int* contacts_dev, void* stream) {
  return step_physics_impl(e, tau_dev, rows_dev, contacts_dev, nullptr, stream);
}

int mb200_contact_point_width(void) { return MB_POINT_WIDTH; }
int mb200_max_contact_points(void) { return MB_MAXC; }

int mb200_step_physics_points(mb200_env* e, const float* tau_dev, int* rows_dev, int* contacts_dev, float* points_dev,
                              void* stream) {
  if (!points_dev) return fail("mb200_step_physics_points: NULL argument");
  return step_physics_impl(e, tau_dev, rows_dev, contacts_dev, points_dev, stream);
}

int mb200_mass_matrix(mb200_env* e, float* M_dev, void* stream) {
  if (!e || !M_dev) return fail("mb200_mass_matrix: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  const LaunchDims d = {grid_for(e), e->warps * 32, e->smem, (cudaStream_t)stream};
  e->ops->debug(d, e->n, e->phys, e->state, 0, nullptr, M_dev);
  e->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int mb200_inverse_dynamics(mb200_env* e, const float* acc_dev, float* tau_dev, void* stream) {
  if (!e || !acc_dev || !tau_dev) return fail("mb200_inverse_dynamics: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  MbPhysics p = e->phys;
  p.lin_damping = 0.0f;  // calculateInverseDynamics has no velocity-damping term
  p.ang_damping = 0.0f;
  const LaunchDims d = {grid_for(e), e->warps * 32, e->smem, (cudaStream_t)stream};
  e->ops->debug(d, e->n, p, e->state, 1, acc_dev, tau_dev);
  e->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int mb200_apply_impulse(mb200_env* e, const int* link_dev, const float* point_dev, const float* impulse_dev,
                        void* stream) {
  if (!e || !link_dev || !point_dev || !impulse_dev) return fail("mb200_apply_impulse: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  const LaunchDims d = {grid_for(e), e->warps * 32, e->smem, (cudaStream_t)stream};
  e->ops->impulse(d, e->n, e->phys, e->state, link_dev, point_dev, impulse_dev);
  e->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// mb200_render, pass 2: one CTA per (camera, 16 x 16 pixel tile), one thread per pixel.  The CTA stages the camera's
// primitive list in shared memory and inverts its proj * view once (double); every thread then casts its pixel's ray
// (mb_render_pixel) and stores RGB, depth and segmentation.
#define MB_RENDER_TILE 16
__global__ void __launch_bounds__(MB_RENDER_TILE* MB_RENDER_TILE)
    k_render_rays(int nprim, const float* scene, const float* view, const float* proj, int W, int H, uint8_t* rgb,
                  float* depth, int* seg) {
  __shared__ __align__(16) float prims[MB_RMAX * MB_RSTRIDE];
  __shared__ MbCamera cam;
  const int c = blockIdx.x, tid = threadIdx.x;
  const int tiles_x = (W + MB_RENDER_TILE - 1) / MB_RENDER_TILE;
  const int tx = blockIdx.y % tiles_x, ty = blockIdx.y / tiles_x;
  const float* src = scene + (size_t)c * MB_RMAX * MB_RSTRIDE;
  for (int i = tid; i < nprim * MB_RSTRIDE; i += blockDim.x) prims[i] = src[i];
  if (tid == 0) mb_render_camera(view + 16 * (size_t)c, proj + 16 * (size_t)c, &cam);
  __syncthreads();
  const int col = tx * MB_RENDER_TILE + tid % MB_RENDER_TILE, row = ty * MB_RENDER_TILE + tid / MB_RENDER_TILE;
  if (col >= W || row >= H) return;
  const size_t px = ((size_t)c * H + row) * W + col;
  uint8_t p3[3];
  float dp;
  int sg;
  mb_render_pixel(cam, prims, nprim, W, H, row, col, rgb ? p3 : nullptr, &dp, &sg);
  if (rgb) { rgb[3 * px] = p3[0]; rgb[3 * px + 1] = p3[1]; rgb[3 * px + 2] = p3[2]; }
  if (depth) depth[px] = dp;
  if (seg) seg[px] = sg;
}

int mb200_render(mb200_env* e, const int* env_ids_dev, int count, const float* view_dev, const float* proj_dev,
                 int width, int height, uint8_t* rgb_dev, float* depth_dev, int32_t* seg_dev, void* stream) {
  if (!e) return fail("mb200_render: NULL argument");
  if (count < 1) return fail("mb200_render: count must be >= 1, got " + std::to_string(count));
  if (width < 1 || width > MB_RENDER_MAXDIM || height < 1 || height > MB_RENDER_MAXDIM)
    return fail("mb200_render: width and height must be in [1, " + std::to_string(MB_RENDER_MAXDIM) + "], got " +
                std::to_string(width) + " x " + std::to_string(height));
  if (!view_dev || !proj_dev) return fail("mb200_render: NULL view or projection matrices");
  CUDA_OK(cudaSetDevice(e->device));
  if (count > e->render_cap) {
    cudaFree(e->render_scene);
    e->render_scene = nullptr;
    e->render_cap = 0;
    CUDA_OK(cudaMalloc(&e->render_scene, (size_t)count * MB_RMAX * MB_RSTRIDE * sizeof(float)));
    e->render_cap = count;
  }
  const cudaStream_t st = (cudaStream_t)stream;
  const LaunchDims d = {(count + e->warps - 1) / e->warps, e->warps * 32, e->smem, st};
  e->ops->render(d, e->n, count, e->phys, e->state, e->rec, env_ids_dev, e->render_scene);
  const int tiles = ((width + MB_RENDER_TILE - 1) / MB_RENDER_TILE) * ((height + MB_RENDER_TILE - 1) / MB_RENDER_TILE);
  k_render_rays<<<dim3(count, tiles), MB_RENDER_TILE * MB_RENDER_TILE, 0, st>>>(
      e->ops->render_nprim, e->render_scene, view_dev, proj_dev, width, height, rgb_dev, depth_dev, seg_dev);
  e->launches += 2;
  CUDA_OK(cudaGetLastError());
  return 0;
}

// mb200_set_param (values == nullptr: `scalar` for every env) and mb200_set_param_array: one of the env's
// MbKindOps::params, checked, into its int record field
static int set_param(mb200_env* e, const char* key, const float* values, int count, float scalar) {
  CUDA_OK(cudaSetDevice(e->device));
  const MbParam* prm = e->ops->params;
  while (prm->key && strcmp(prm->key, key) != 0) ++prm;
  if (!prm->key) return fail(std::string("mb200_set_param: unknown key '") + key + "' for this env");
  const float first = values ? values[0] : scalar;
  if (prm->check)
    for (int i = 0; i < (values ? count : 1); ++i)
      if (const char* err = prm->check(values ? values[i] : scalar, first)) return fail(err);
  if (prm->variant) e->ops = find_kind(e->ops->env_id, prm->variant(first));
  if (!values && prm->boolean) scalar = scalar != 0.0f;
  CUDA_OK(cudaDeviceSynchronize());
  const size_t n = (size_t)e->n_pad;
  float* rec = (float*)malloc(n * e->rec_stride * sizeof(float));
  if (!rec) return fail("mb200_set_param: host allocation failed");
  CUDA_OK(cudaMemcpy(rec, e->rec, n * e->rec_stride * sizeof(float), cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; ++i)
    reinterpret_cast<int*>(rec + i * e->rec_stride)[prm->field] = (int)(values ? values[i % (size_t)count] : scalar);
  CUDA_OK(cudaMemcpy(e->rec, rec, n * e->rec_stride * sizeof(float), cudaMemcpyHostToDevice));
  free(rec);
  return 0;
}

int mb200_set_param(mb200_env* e, const char* key, float value) {
  if (!e || !key) return fail("mb200_set_param: NULL argument");
  return set_param(e, key, nullptr, 0, value);
}

int mb200_set_param_array(mb200_env* e, const char* key, const float* values_host, int count) {
  if (!e || !key || !values_host) return fail("mb200_set_param_array: NULL argument");
  if (count != e->n) return fail("mb200_set_param_array: count must equal the number of envs");
  return set_param(e, key, values_host, count, 0.0f);
}

int mb200_stats(mb200_env* e, double out[8], int reset) {
  if (!e || !out) return fail("mb200_stats: NULL argument");
  CUDA_OK(cudaSetDevice(e->device));
  MbStats s;
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaMemcpy(&s, e->stats, sizeof(s), cudaMemcpyDeviceToHost));
  out[0] = (double)s.episodes; out[1] = s.ret_sum; out[2] = s.len_sum; out[3] = (double)s.nonfinite;
  out[4] = (double)s.overflow; out[5] = (double)s.steps_reached_sum; out[6] = out[7] = 0.0;
  if (reset) CUDA_OK(cudaMemset(e->stats, 0, sizeof(MbStats)));
  return 0;
}

long long mb200_launch_count(const mb200_env* e) { return e ? e->launches : 0; }
int mb200_record_stride(const mb200_env* e) { return e ? e->rec_stride : 0; }

int mb200_measure_fp32_peak(int device, double* tflops_out) {
  if (!tflops_out) return fail("mb200_measure_fp32_peak: NULL argument");
  CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 14;
  float* buf = nullptr;
  CUDA_OK(cudaMalloc(&buf, (size_t)blocks * threads * sizeof(float)));
  cudaEvent_t e0, e1;
  CUDA_OK(cudaEventCreate(&e0));
  CUDA_OK(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_OK(cudaEventRecord(e0));
    k_fma_probe<<<blocks, threads>>>(buf, iters, 0.999f, 1e-3f);
    CUDA_OK(cudaEventRecord(e1));
    CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8.0 * (double)iters * (double)blocks * threads;
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(buf);
  *tflops_out = best;
  return 0;
}

}  // extern "C"
