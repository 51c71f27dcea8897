// mb_kind.cuh -- the kernels of ONE env kind and the launcher table the C ABI (mb200.cu) dispatches through.
// Every env kind is its own translation unit (csrc/kinds/*.cu: model table + MB_DEFINE_KIND), so the kinds compile in
// parallel and a change to one env's epilogue rebuilds one object.  Kernel names keep the k_<what>_<kind> scheme the
// profiles and the driver's launch lists use.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#ifndef MB_WARPS_DEFAULT
#define MB_WARPS_DEFAULT 14 /* envs (warps) per CTA of the step kernels; 2 CTAs per SM (72 registers, <= 114 KB smem) */
#endif
#ifndef MB_WARPS_MAX
#define MB_WARPS_MAX 16
#endif
#define MB_WARPS ((int)(blockDim.x >> 5)) /* device code: warps of this launch */
#ifndef MB_MINBLOCKS
#define MB_MINBLOCKS 2
#endif
#ifndef MB_SYNC
#define MB_SYNC 1
#endif

#include "../../include/mocca_b200.h"
#include "mb_env.cuh"

struct StepArgs {
  int n;
  MbPhysics phys;
  float* state;
  float* rec;
  uint32_t* mt;
  const float* act;
  float* obs;
  float* rew;
  uint8_t* done;
  uint8_t* trunc;
  float* final_obs;
  MbStats* stats;
  float* dummy_obs;
  float* dummy_rew;
  uint8_t* dummy_flag;
  MbStats* dummy_stats;
  const int* order;
  int* key;
  int* hist;  // this step's histogram half, nullptr = scheduler off
  // mb200_step_host with pinned (device-mapped) result buffers: each warp forwards its env's finished rows from the
  // device staging arrays to the host with coalesced zero-copy stores, so the D2H traffic overlaps the rest of the
  // launch instead of following it; nullptr = staged cudaMemcpyAsync (pageable host memory) or device callers
  float* host_obs;
  float* host_rew;
  uint8_t* host_done;
  uint8_t* host_trunc;
  int* info;  // [n] per-step integer info (Stepper: steps_reached, -1 = not reported), may be nullptr
  float* warm;  // [n_pad][MB_NWARM] contact impulses of the previous substep, nullptr = warm starting off
};

struct LaunchDims {
  int grid, threads;
  size_t smem;
  cudaStream_t stream;
};

// what mb200.cu needs to know about a kind
struct MbKindOps {
  const char* env_id;
  const char* variant;  // "" or "pillar"
  int obs_dim, act_dim, rec_stride, nj, warps, info_field;
  size_t smem_per_env;
  void (*default_physics)(mb200_physics&);  // the env's own public defaults (Env::default_physics)
  void (*fix_physics)(MbPhysics&);           // applied after the caller's parameters (Env::fix_physics)
  const MbParam* params;                     // the keys mb200_set_param accepts (Env::PARAMS)
  cudaError_t (*prepare)(void);  // shared-memory opt-in of every kernel of the kind
  void (*step)(const StepArgs&, bool host, const LaunchDims&);
  void (*reset)(const LaunchDims&, int n, const MbPhysics&, float* state, float* rec, uint32_t* mt, const uint8_t* mask,
                float* obs, float* dummy_obs, float* warm);
  void (*physics)(const LaunchDims&, int n, const MbPhysics&, float* state, const float* rec, const float* tau,
                  int* rows_out, int* contacts_out, float* points_out, float* warm);
  void (*debug)(const LaunchDims&, int n, const MbPhysics&, const float* state, int mode, const float* acc, float* out);
};

template <class Env, bool HOST>
__device__ __forceinline__ void step_body(const StepArgs& a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // broadcast from lane 0: tells the compiler the warp index is warp-uniform, so the WarpMem base lives in a uniform
  // register instead of being re-derived from threadIdx (3-4 % of the issued instructions otherwise)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int env = a.order[blockIdx.x * MB_WARPS + warp];  // a permutation of [0, n_pad)
  const bool tail = env >= a.n;
  typename Env::Mem& S = reinterpret_cast<typename Env::Mem*>(smem_raw)[warp];
  if ((threadIdx.x & 31) == 0) S.warm = a.warm ? a.warm + (size_t)env * MB_NWARM : nullptr;
  __syncwarp();
  float* obs = tail ? a.dummy_obs + (size_t)warp * Env::OBS : a.obs + (size_t)env * Env::OBS;
  float* fin = tail ? a.dummy_obs + (size_t)(MB_WARPS_MAX + warp) * Env::OBS
                    : (a.final_obs ? a.final_obs + (size_t)env * Env::OBS : nullptr);
  Env::step(S, a.phys, a.state + (size_t)env * MB_STATE_STRIDE, a.rec + (size_t)env * Env::REC_STRIDE,
            a.mt + (size_t)env * 2 * MB_MT_STRIDE, a.mt + ((size_t)env * 2 + 1) * MB_MT_STRIDE,
            a.act + (size_t)(tail ? 0 : env) * Env::ACT, obs, tail ? a.dummy_rew + warp : a.rew + env,
            tail ? a.dummy_flag + warp : a.done + env, tail ? a.dummy_flag + MB_WARPS_MAX + warp : a.trunc + env, fin,
            tail ? a.dummy_stats : a.stats);
  if (HOST && !tail) {
    // (separate kernel instantiation: the extra epilogue cost the device-buffer kernel 1 % through register
    // allocation when it was a run-time branch)  the row is final here (auto-reset included); lanes read what other
    // lanes of this warp wrote
    __syncwarp();
    const int lane = threadIdx.x & 31;
    const float* src = a.obs + (size_t)env * Env::OBS;
    float* dst = a.host_obs + (size_t)env * Env::OBS;
#pragma unroll
    for (int i = lane; i < Env::OBS; i += 32) dst[i] = __ldcg(src + i);
    if (lane == 0) {
      a.host_rew[env] = __ldcg(a.rew + env);
      a.host_done[env] = __ldcg(a.done + env);
      a.host_trunc[env] = __ldcg(a.trunc + env);
    }
  }
  if ((threadIdx.x & 31) == 0) {
    if (Env::INFO_FIELD >= 0 && a.info && !tail)
      a.info[env] = reinterpret_cast<const int*>(a.rec + (size_t)env * Env::REC_STRIDE)[Env::INFO_FIELD >= 0 ? Env::INFO_FIELD : 0];
    // work estimate for the scheduler: constraint rows of this step
    if (a.hist) {
      // (taken from the step itself, not from the float running sum ER_ROWS, which stops resolving single steps after
      // ~10^7 rows = a few hours of stepping)
      int k = S.step_rows;
      k = 255 - (k < 0 ? 0 : (k > 255 ? 255 : k));  // heaviest first
      a.key[env] = k;
      atomicAdd(&a.hist[k], 1);
    }
  }
}

template <class Env>
__device__ __forceinline__ void reset_body(int n, const MbPhysics& phys, float* state, float* rec, uint32_t* mt,
                                           const uint8_t* mask, float* obs, float* dummy_obs, float* warm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5;
  const int env = blockIdx.x * MB_WARPS + warp;
  const bool tail = env >= n;
  if (!tail && mask && !mask[env]) return;  // no CTA barrier inside reset, early exit is fine
  typename Env::Mem& S = reinterpret_cast<typename Env::Mem*>(smem_raw)[warp];
  if ((threadIdx.x & 31) == 0) S.warm = warm ? warm + (size_t)env * MB_NWARM : nullptr;
  __syncwarp();
  Env::reset(S, phys, rec + (size_t)env * Env::REC_STRIDE, mt + (size_t)env * 2 * MB_MT_STRIDE,
             mt + ((size_t)env * 2 + 1) * MB_MT_STRIDE,
             tail ? dummy_obs + (size_t)warp * Env::OBS : obs + (size_t)env * Env::OBS);
  Env::store_state(S, state + (size_t)env * MB_STATE_STRIDE);
}

// stepSimulation only; rec supplies the static obstacles of the env kind
template <class Env>
__device__ __forceinline__ void physics_body(int n, const MbPhysics& phys, float* state, const float* rec,
                                             const float* tau, int* rows_out, int* contacts_out, float* points_out,
                                             float* warm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5;
  const int env = blockIdx.x * MB_WARPS + warp;
  const bool tail = env >= n;  // pad env: steps with zero torque, outputs discarded
  typename Env::Mem& S = reinterpret_cast<typename Env::Mem*>(smem_raw)[warp];
  if ((threadIdx.x & 31) == 0) S.warm = warm ? warm + (size_t)env * MB_NWARM : nullptr;
  __syncwarp();
  int nc;
  const int rows = mb_physics_step<Env>(
      S, phys, state + (size_t)env * MB_STATE_STRIDE, rec + (size_t)env * Env::REC_STRIDE,
      tail ? nullptr : tau + (size_t)env * Env::Model::NJ,
      points_out && !tail ? points_out + (size_t)env * MB_MAXC * MB_POINT_WIDTH : nullptr, &nc);
  if (tail) return;
  if ((threadIdx.x & 31) == 0) {
    if (rows_out) rows_out[env] = rows;
    if (contacts_out) contacts_out[env] = nc;
  }
}

// mode 0: M (full symmetric, [nu][nu]);  mode 1: tau = M acc - rhs (rhs = -bias with zero applied torque)
template <class Env>
__device__ __forceinline__ void dynamics_debug_body(int n, const MbPhysics& phys, const float* state, int mode,
                                                    const float* acc, float* out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  typedef typename Env::Model EM;
  const int warp = threadIdx.x >> 5;
  const int env = blockIdx.x * MB_WARPS + warp;
  if (env >= n) return;
  typename Env::Mem& S = reinterpret_cast<typename Env::Mem*>(smem_raw)[warp];
  const int NU = EM::NU;
  if ((threadIdx.x & 31) == 0) S.warm = nullptr;
  __syncwarp();
  mb_mass_matrix<Env>(S, phys, state + (size_t)env * MB_STATE_STRIDE);
  MB_LANES(l)
    if (l < NU) {
      if (mode == 0) {
        for (int j = 0; j < NU; ++j) out[((size_t)env * NU + l) * NU + j] = mb_Lget<EM>(S.L, l, j);
      } else {
        float t = -S.rhs[l];
        for (int j = 0; j < NU; ++j) t += mb_Lget<EM>(S.L, l, j) * acc[(size_t)env * NU + j];
        out[(size_t)env * NU + l] = t;
      }
    }
  MB_END
}

// One env kind: step (device / host-buffer instantiations), reset, physics-only and debug kernels + its MbKindOps.
#define MB_DEFINE_KIND(ID, ENV_ID, VARIANT, ENV, WARPS)                                                               \
  __global__ void __launch_bounds__(WARPS * 32, MB_MINBLOCKS) k_step_##ID(StepArgs a) { step_body<ENV, false>(a); }  \
  __global__ void __launch_bounds__(WARPS * 32, MB_MINBLOCKS) k_step_##ID##_host(StepArgs a) {                       \
    step_body<ENV, true>(a);                                                                                         \
  }                                                                                                                   \
  __global__ void __launch_bounds__(MB_WARPS_MAX * 32)                                                                \
      k_reset_##ID(int n, MbPhysics phys, float* state, float* rec, uint32_t* mt, const uint8_t* mask, float* obs,   \
                   float* dummy_obs, float* warm) {                                                                   \
    reset_body<ENV>(n, phys, state, rec, mt, mask, obs, dummy_obs, warm);                                             \
  }                                                                                                                   \
  __global__ void __launch_bounds__(MB_WARPS_MAX * 32)                                                                \
      k_step_physics_##ID(int n, MbPhysics phys, float* state, const float* rec, const float* tau, int* rows_out,    \
                          int* contacts_out, float* points_out, float* warm) {                                        \
    physics_body<ENV>(n, phys, state, rec, tau, rows_out, contacts_out, points_out, warm);                            \
  }                                                                                                                   \
  __global__ void __launch_bounds__(MB_WARPS_MAX * 32)                                                                \
      k_dynamics_debug_##ID(int n, MbPhysics phys, const float* state, int mode, const float* acc, float* out) {     \
    dynamics_debug_body<ENV>(n, phys, state, mode, acc, out);                                                         \
  }                                                                                                                   \
  static cudaError_t prepare_##ID(void) {                                                                             \
    const int bytes = (int)(sizeof(typename ENV::Mem) * WARPS);                                                \
    const cudaFuncAttribute at = cudaFuncAttributeMaxDynamicSharedMemorySize;                                         \
    cudaError_t e;                                                                                                    \
    if ((e = cudaFuncSetAttribute(k_step_##ID, at, bytes)) != cudaSuccess) return e;                                  \
    if ((e = cudaFuncSetAttribute(k_step_##ID##_host, at, bytes)) != cudaSuccess) return e;                           \
    if ((e = cudaFuncSetAttribute(k_reset_##ID, at, bytes)) != cudaSuccess) return e;                                 \
    if ((e = cudaFuncSetAttribute(k_step_physics_##ID, at, bytes)) != cudaSuccess) return e;                          \
    return cudaFuncSetAttribute(k_dynamics_debug_##ID, at, bytes);                                                    \
  }                                                                                                                   \
  static void launch_step_##ID(const StepArgs& a, bool host, const LaunchDims& d) {                                   \
    if (host) k_step_##ID##_host<<<d.grid, d.threads, d.smem, d.stream>>>(a);                                         \
    else k_step_##ID<<<d.grid, d.threads, d.smem, d.stream>>>(a);                                                     \
  }                                                                                                                   \
  static void launch_reset_##ID(const LaunchDims& d, int n, const MbPhysics& p, float* state, float* rec,            \
                                uint32_t* mt, const uint8_t* mask, float* obs, float* dummy_obs, float* warm) {       \
    k_reset_##ID<<<d.grid, d.threads, d.smem, d.stream>>>(n, p, state, rec, mt, mask, obs, dummy_obs, warm);          \
  }                                                                                                                   \
  static void launch_physics_##ID(const LaunchDims& d, int n, const MbPhysics& p, float* state, const float* rec,    \
                                  const float* tau, int* rows_out, int* contacts_out, float* points_out,              \
                                  float* warm) {                                                                      \
    k_step_physics_##ID<<<d.grid, d.threads, d.smem, d.stream>>>(n, p, state, rec, tau, rows_out, contacts_out,       \
                                                                 points_out, warm);                                   \
  }                                                                                                                   \
  static void launch_debug_##ID(const LaunchDims& d, int n, const MbPhysics& p, const float* state, int mode,        \
                                const float* acc, float* out) {                                                       \
    k_dynamics_debug_##ID<<<d.grid, d.threads, d.smem, d.stream>>>(n, p, state, mode, acc, out);                      \
  }                                                                                                                   \
  extern const MbKindOps mb_kind_##ID = {ENV_ID, VARIANT, ENV::OBS, ENV::ACT, ENV::REC_STRIDE, ENV::Model::NJ,       \
                                         WARPS, ENV::INFO_FIELD, sizeof(typename ENV::Mem),                          \
                                         ENV::template default_physics<mb200_physics>, ENV::fix_physics, ENV::PARAMS, \
                                         prepare_##ID,                                                               \
                                         launch_step_##ID, launch_reset_##ID, launch_physics_##ID,                    \
                                         launch_debug_##ID};
