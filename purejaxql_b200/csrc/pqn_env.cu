// Batched environment operator + fused rollout step for sm_100a.
//
// Kernels here are HBM-bound integer/byte work: one env per thread, state in
// registers for the duration of the step, word-major SoA state (128-byte
// coalesced per warp and word), observations written either as fully
// coalesced 16-byte vectors (float obs, staged through shared memory) or as
// 64-byte bit-packed rows (rollout buffer).  Compiled with -fmad=false so the
// fp32 classic-control physics round exactly as written.
//
// Reference seams: see include/pqn_b200.h next to each entry point.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/pqn_b200.h"
#include "api_common.h"
#include "env_breakout.cuh"
#include "env_bsuite.cuh"
#include "env_classic.cuh"
#include "env_minatar_more.cuh"
#include "rollout_logic.cuh"

namespace pqn {

constexpr int ENV_BLOCK = 128;

// ---------------------------------------------------------------------------
// observation writers
// ---------------------------------------------------------------------------
// Shared-memory scratch of a block for binary observations: word-major [OBS_WORDS_PAD][ENV_BLOCK] (thread t owns
// column t: conflict-free).  Env::OBS_IN_REGS games (Breakout) build the words in registers and copy them in;
// the others set bits directly in their column.
template <class Env>
struct ObsScratch {
  static constexpr int WORDS = Env::BINARY_OBS ? Env::OBS_WORDS_PAD * ENV_BLOCK : 1;
};

template <class Env>
__device__ __forceinline__ void obs_to_scratch(const typename Env::State& s, bool active, uint32_t* __restrict__ scratch) {
  uint32_t* col = scratch + threadIdx.x;
  if constexpr (Env::OBS_IN_REGS) {
    uint32_t bits[Env::OBS_WORDS_PAD];
    if (active) Env::obs_bits(s, bits);
#pragma unroll
    for (int w = 0; w < Env::OBS_WORDS_PAD; ++w) col[w * ENV_BLOCK] = active ? bits[w] : 0u;
  } else {
#pragma unroll
    for (int w = 0; w < Env::OBS_WORDS_PAD; ++w) col[w * ENV_BLOCK] = 0u;
    if (active) Env::obs_bits_mem(s, col, ENV_BLOCK);
  }
}

// Binary obs -> float32[N][OBS_DIM]: each warp expands its 32 staged rows and writes the 32*OBS_DIM floats as
// consecutive float4 — 512 contiguous bytes per store instruction.
template <class Env>
__device__ __forceinline__ void write_obs_float_binary(const uint32_t* __restrict__ scratch, float* __restrict__ obs,
                                                       int64_t warp_env0, int64_t N) {
  const int lane = threadIdx.x & 31;
  const uint32_t* __restrict__ sw = scratch + (threadIdx.x & ~31);  // this warp's 32 columns
  __syncwarp();
  constexpr int V = Env::OBS_DIM / 4;  // float4 per env
  const int64_t n_here = (N - warp_env0) < 32 ? (N - warp_env0) : 32;
  float4* __restrict__ out = reinterpret_cast<float4*>(obs + warp_env0 * Env::OBS_DIM);
  const int total = (int)n_here * V;
  for (int g = lane; g < total; g += 32) {
    const int env = g / V;
    const int q = g - env * V;
    const int bit = q * 4;
    const uint32_t nib = (sw[(bit >> 5) * ENV_BLOCK + env] >> (bit & 31)) & 15u;
    float4 v;
    v.x = (nib & 1u) ? 1.f : 0.f; v.y = (nib & 2u) ? 1.f : 0.f;
    v.z = (nib & 4u) ? 1.f : 0.f; v.w = (nib & 8u) ? 1.f : 0.f;
    __stcs(out + g, v);  // streaming store: obs rows are not re-read by this kernel
  }
  __syncwarp();
}

// packed row (OBS_WORDS_PAD words, 16-byte multiple) of this thread's env from its scratch column
template <class Env>
__device__ __forceinline__ void write_obs_packed(const uint32_t* __restrict__ scratch, uint32_t* __restrict__ obs_packed,
                                                 int64_t i) {
  const uint32_t* col = scratch + threadIdx.x;
  uint4* __restrict__ row = reinterpret_cast<uint4*>(obs_packed + i * Env::OBS_WORDS_PAD);
#pragma unroll
  for (int v = 0; v < Env::OBS_WORDS_PAD / 4; ++v)
    row[v] = make_uint4(col[(4 * v) * ENV_BLOCK], col[(4 * v + 1) * ENV_BLOCK], col[(4 * v + 2) * ENV_BLOCK],
                        col[(4 * v + 3) * ENV_BLOCK]);
}

template <class Env>
__device__ __forceinline__ void write_obs_float_dense(const typename Env::State& s, float* __restrict__ obs,
                                                      int64_t i) {
  float o[Env::OBS_DIM];
  Env::obs_float(s, o);
#pragma unroll
  for (int j = 0; j < Env::OBS_DIM; ++j) obs[i * Env::OBS_DIM + j] = o[j];
}

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
template <class Env>
__global__ void __launch_bounds__(ENV_BLOCK) env_reset_kernel(const uint32_t* __restrict__ keys,
                                                              uint32_t* __restrict__ state,
                                                              float* __restrict__ obs, int64_t N, int max_steps,
                                                              int memory_length, int part) {
  __shared__ uint32_t smem[ObsScratch<Env>::WORDS];
  const int64_t i = (int64_t)blockIdx.x * ENV_BLOCK + threadIdx.x;
  const bool active = i < N;
  typename Env::State s;
  if (active) {
    Key k{keys[2 * i], keys[2 * i + 1]};
    env_set_params<Env>(s, memory_length);
    Env::reset_env(k, part, max_steps, s);
    Env::store(s, state, N, i);
    LogState lg;
    log_reset(lg);
    log_store(lg, state, N, i, Env::CORE_WORDS);
  }
  if (obs != nullptr) {
    if constexpr (Env::BINARY_OBS) {
      obs_to_scratch<Env>(s, active, smem);
      const int64_t warp_env0 = (int64_t)blockIdx.x * ENV_BLOCK + (threadIdx.x & ~31);
      if (warp_env0 < N) write_obs_float_binary<Env>(smem, obs, warp_env0, N);
    } else {
      if (active) write_obs_float_dense<Env>(s, obs, i);
    }
  }
}

template <class Env>
__global__ void __launch_bounds__(ENV_BLOCK)
    env_step_kernel(const uint32_t* __restrict__ keys, uint32_t* __restrict__ state,
                    const int32_t* __restrict__ action, float* __restrict__ obs, float* __restrict__ reward,
                    uint8_t* __restrict__ done, float* __restrict__ info_discount,
                    float* __restrict__ info_ret, int32_t* __restrict__ info_len,
                    int32_t* __restrict__ info_t, int64_t N, int max_steps, int part) {
  __shared__ uint32_t smem[ObsScratch<Env>::WORDS];
  const int64_t i = (int64_t)blockIdx.x * ENV_BLOCK + threadIdx.x;
  const bool active = i < N;
  typename Env::State s;
  if (active) {
    Env::load(s, state, N, i);
    LogState lg;
    log_load(lg, state, N, i, Env::CORE_WORDS);
    Key k{keys[2 * i], keys[2 * i + 1]};
    float r;
    bool d;
    env_step_full<Env>(k, part, max_steps, s, lg, action[i], r, d);
    Env::store(s, state, N, i);
    log_store(lg, state, N, i, Env::CORE_WORDS);
    reward[i] = r;
    done[i] = d ? 1 : 0;
    if (info_discount) info_discount[i] = d ? 0.f : 1.f;
    if (info_ret) info_ret[i] = lg.returned_episode_returns;
    if (info_len) info_len[i] = lg.returned_episode_lengths;
    if (info_t) info_t[i] = lg.timestep;
  }
  if (obs != nullptr) {
    if constexpr (Env::BINARY_OBS) {
      obs_to_scratch<Env>(s, active, smem);
      const int64_t warp_env0 = (int64_t)blockIdx.x * ENV_BLOCK + (threadIdx.x & ~31);
      if (warp_env0 < N) write_obs_float_binary<Env>(smem, obs, warp_env0, N);
    } else {
      if (active) write_obs_float_dense<Env>(s, obs, i);
    }
  }
}

template <class Env>
__global__ void __launch_bounds__(ENV_BLOCK)
    env_obs_kernel(const uint32_t* __restrict__ state, float* __restrict__ obs, uint32_t* __restrict__ obs_packed,
                   int64_t N) {
  __shared__ uint32_t smem[ObsScratch<Env>::WORDS];
  const int64_t i = (int64_t)blockIdx.x * ENV_BLOCK + threadIdx.x;
  const bool active = i < N;
  typename Env::State s;
  if (active) Env::load(s, state, N, i);
  if constexpr (Env::BINARY_OBS) {
    obs_to_scratch<Env>(s, active, smem);
    if (obs_packed != nullptr && active) write_obs_packed<Env>(smem, obs_packed, i);
    if (obs != nullptr) {
      const int64_t warp_env0 = (int64_t)blockIdx.x * ENV_BLOCK + (threadIdx.x & ~31);
      if (warp_env0 < N) write_obs_float_binary<Env>(smem, obs, warp_env0, N);
    }
  } else {
    if (obs != nullptr && active) write_obs_float_dense<Env>(s, obs, i);
  }
}

__global__ void eps_greedy_kernel(const uint32_t* __restrict__ keys, const float* __restrict__ q,
                                  const float* __restrict__ eps, int32_t* __restrict__ action, int64_t N, int A,
                                  int part) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  Key k{keys[2 * i], keys[2 * i + 1]};
  float mq;
  action[i] = eps_greedy_one(k, q + i * A, A, eps[0], part, mq);
}

// Fused _step_env body.  grid = (ceil(E/ENV_BLOCK), S); blockIdx.y = seed.
template <class Env>
__global__ void __launch_bounds__(ENV_BLOCK)
    rollout_act_step_kernel(const uint32_t* __restrict__ step_keys, const float* __restrict__ q,
                            const float* __restrict__ eps_p, uint32_t* __restrict__ state,
                            void* __restrict__ obs_next, int32_t* __restrict__ action_out,
                            float* __restrict__ reward_out, uint8_t* __restrict__ done_out,
                            float* __restrict__ maxq_out, double* __restrict__ info_sums, int E, int max_steps,
                            float rew_scale, int part, int64_t obs_seed_stride, int64_t tr_seed_stride,
                            int info_done_only, int E_total, int env_offset) {
  __shared__ uint32_t obs_smem[ObsScratch<Env>::WORDS];
  const int seed = blockIdx.y;
  const int e = blockIdx.x * ENV_BLOCK + threadIdx.x;
  const int64_t N = (int64_t)gridDim.y * E;
  const int64_t i = (int64_t)seed * E + e;
  const bool active = e < E;
  float sums[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  if (active) {
    const Key ka{step_keys[seed * 4 + 0], step_keys[seed * 4 + 1]};
    const Key ks{step_keys[seed * 4 + 2], step_keys[seed * 4 + 3]};
    const float eps = eps_p[0];
    float mq;
    // per-env keys are element (env_offset + e) of split(key, E_total): an env shard of a larger vmap (env-sharded
    // data parallelism) draws exactly the keys the unsharded run gives those envs
    const uint32_t ge = (uint32_t)(env_offset + e);
    const int a = eps_greedy_one(split_at(ka, (uint32_t)E_total, ge, part), q + i * Env::NUM_ACTIONS,
                                 Env::NUM_ACTIONS, eps, part, mq);
    typename Env::State s;
    Env::load(s, state, N, i);
    LogState lg;
    log_load(lg, state, N, i, Env::CORE_WORDS);
    float r;
    bool d;
    env_step_full<Env>(split_at(ks, (uint32_t)E_total, ge, part), part, max_steps, s, lg, a, r, d);
    Env::store(s, state, N, i);
    log_store(lg, state, N, i, Env::CORE_WORDS);
    const int64_t io = (int64_t)seed * obs_seed_stride + e;
    const int64_t it = (int64_t)seed * tr_seed_stride + e;
    action_out[it] = a;
    reward_out[it] = rew_scale * r;
    done_out[it] = d ? 1 : 0;
    maxq_out[it] = mq;
    if constexpr (Env::BINARY_OBS) {
      obs_to_scratch<Env>(s, true, obs_smem);
      write_obs_packed<Env>(obs_smem, reinterpret_cast<uint32_t*>(obs_next), io);
    } else {
      write_obs_float_dense<Env>(s, reinterpret_cast<float*>(obs_next), io);
    }
    sums[0] = lg.returned_episode_returns;
    sums[1] = (float)lg.returned_episode_lengths;
    sums[2] = (float)lg.timestep;
    sums[3] = d ? 1.f : 0.f;
    sums[4] = d ? 0.f : 1.f;
    if (info_done_only && !d) { sums[0] = 0.f; sums[1] = 0.f; sums[2] = 0.f; sums[4] = 0.f; }
  }
  if (info_sums != nullptr) {
    // block reduction in double, one atomic per metric per block
    __shared__ double red[5][ENV_BLOCK / 32];
#pragma unroll
    for (int m = 0; m < 5; ++m) {
      double v = (double)sums[m];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((threadIdx.x & 31) == 0) red[m][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < ENV_BLOCK / 32; ++w) v += red[threadIdx.x][w];
      atomicAdd(info_sums + seed * 5 + threadIdx.x, v);
    }
  }
}

__global__ void rollout_keys_kernel(uint32_t* __restrict__ rng_inout, uint32_t* __restrict__ keys_out, int S, int T,
                                    int part) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  Key c{rng_inout[2 * s], rng_inout[2 * s + 1]};
  for (int t = 0; t < T; ++t) {
    Key c2, ka, ks;
    split3(c, part, c2, ka, ks);
    uint32_t* o = keys_out + ((int64_t)t * S + s) * 4;
    o[0] = ka.k0; o[1] = ka.k1; o[2] = ks.k0; o[3] = ks.k1;
    c = c2;
  }
  rng_inout[2 * s] = c.k0;
  rng_inout[2 * s + 1] = c.k1;
}

// buffers are [S][T][E]; one thread per (seed, env)
__global__ void qlambda_kernel(const float* __restrict__ reward, const uint8_t* __restrict__ done,
                               const float* __restrict__ maxq, const float* __restrict__ q_last,
                               float* __restrict__ targets, int T, int S, int E, int A, float gamma, float lambda) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)S * E) return;
  const int64_t s = i / E, e = i - s * E;
  const int64_t base = s * (int64_t)T * E;
  qlambda_one(reward + base, done + base, maxq + base, q_last + i * A, targets + base, T, (int64_t)E, A, gamma, lambda,
              e);
}

__global__ void rng_split_kernel(const uint32_t* __restrict__ keys, int64_t n, int num, uint32_t* __restrict__ out,
                                 int part) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n * num) return;
  const int64_t k = g / num;
  const int j = (int)(g - k * num);
  const Key c = split_at(Key{keys[2 * k], keys[2 * k + 1]}, (uint32_t)num, (uint32_t)j, part);
  out[2 * g] = c.k0;
  out[2 * g + 1] = c.k1;
}

__global__ void rng_bits_kernel(const uint32_t* __restrict__ keys, int64_t n, int64_t len, uint32_t* __restrict__ out,
                                int part) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n * len) return;
  const int64_t k = g / len;
  const int64_t j = g - k * len;
  out[g] = bits_at(Key{keys[2 * k], keys[2 * k + 1]}, (uint32_t)len, (uint32_t)j, part);
}

__global__ void threefry_kernel(const uint32_t* __restrict__ kp, const uint32_t* __restrict__ cp,
                                uint32_t* __restrict__ out, int64_t n) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  uint32_t x0 = cp[2 * g], x1 = cp[2 * g + 1];
  threefry2x32(kp[2 * g], kp[2 * g + 1], x0, x1);
  out[2 * g] = x0;
  out[2 * g + 1] = x1;
}

// ---------------------------------------------------------------------------
// host-side dispatch
// ---------------------------------------------------------------------------
template <class Env>
static void fill_info(pqn_env_info_t* o) {
  o->state_words = Env::STATE_WORDS;
  o->obs_dim = Env::OBS_DIM;
  o->num_actions = Env::NUM_ACTIONS;
  o->max_steps = Env::DEFAULT_MAX_STEPS;
  o->binary_obs = Env::BINARY_OBS ? 1 : 0;
  if constexpr (Env::BINARY_OBS) {
    o->obs_shape[0] = Env::OBS_H; o->obs_shape[1] = Env::OBS_W; o->obs_shape[2] = Env::OBS_C;
    o->packed_obs_words = Env::OBS_WORDS_PAD;
  } else {
    o->obs_shape[0] = Env::OBS_DIM; o->obs_shape[1] = 1; o->obs_shape[2] = 1;
    o->packed_obs_words = 0;
  }
}

#define PQN_ENV_DISPATCH(env_id, ...)                                           \
  switch (env_id) {                                                             \
    case ENV_BREAKOUT: { using EnvT = BreakoutEnv; __VA_ARGS__; } break;        \
    case ENV_ASTERIX: { using EnvT = AsterixEnv; __VA_ARGS__; } break;          \
    case ENV_FREEWAY: { using EnvT = FreewayEnv; __VA_ARGS__; } break;          \
    case ENV_SPACE_INVADERS: { using EnvT = SpaceInvadersEnv; __VA_ARGS__; } break; \
    case ENV_CARTPOLE: { using EnvT = CartPoleEnv; __VA_ARGS__; } break;        \
    case ENV_ACROBOT: { using EnvT = AcrobotEnv; __VA_ARGS__; } break;          \
    case ENV_MEMORY_CHAIN: { using EnvT = MemoryChainEnv; __VA_ARGS__; } break; \
    default: return set_error(PQN_E_UNSUPPORTED, "env id %d is not built into libpqn_b200", env_id); \
  }

static inline unsigned blocks_for(int64_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

template <class Env>
static int memory_length_or_default(int memory_length) {
  if constexpr (EnvHasMemoryLength<Env>::value) return memory_length > 0 ? memory_length : Env::DEFAULT_MEMORY_LENGTH;
  return 0;
}

// LogWrapper(env).reset over N envs.  params.max_steps <= 0 selects the env default; so does
// params.memory_length <= 0 (pqn_env_reset_params rejects that before it gets here).
static int env_reset(int env_id, const uint32_t* keys, uint32_t* state, float* obs, int64_t N,
                     pqn_env_params_t params, int rng_mode, void* stream, const char* what) {
  if (N == 0) return PQN_OK;
  if (!keys || !state || N < 0) return set_error(PQN_E_INVALID, "%s: bad argument", what);
  PQN_ENV_DISPATCH(env_id, {
    const int ms = params.max_steps > 0 ? params.max_steps : EnvT::DEFAULT_MAX_STEPS;
    const int ml = memory_length_or_default<EnvT>(params.memory_length);
    { LaunchScope _ls(K_ENV_RESET, (cudaStream_t)stream); env_reset_kernel<EnvT><<<blocks_for(N, ENV_BLOCK), ENV_BLOCK, 0, (cudaStream_t)stream>>>(keys, state, obs, N,
                                                                                             ms, ml, rng_mode); }
  });
  return check_launch(what);
}

}  // namespace pqn

using namespace pqn;

extern "C" {

int pqn_env_info(int env_id, pqn_env_info_t* out) {
  if (!out) return set_error(PQN_E_INVALID, "pqn_env_info: out is NULL");
  PQN_ENV_DISPATCH(env_id, fill_info<EnvT>(out));
  return PQN_OK;
}

int pqn_rng_split(const uint32_t* keys, int64_t n, int32_t num, uint32_t* out, int rng_mode, void* stream) {
  if (!keys || !out || n < 0 || num <= 0) return set_error(PQN_E_INVALID, "pqn_rng_split: bad argument");
  if (n == 0) return PQN_OK;
  { LaunchScope _ls(K_RNG, (cudaStream_t)stream); rng_split_kernel<<<blocks_for(n * num, 256), 256, 0, (cudaStream_t)stream>>>(keys, n, num, out, rng_mode); }
  return check_launch("pqn_rng_split");
}

int pqn_rng_bits(const uint32_t* keys, int64_t n, int64_t len, uint32_t* out, int rng_mode, void* stream) {
  if (!keys || !out || n < 0 || len <= 0) return set_error(PQN_E_INVALID, "pqn_rng_bits: bad argument");
  if (n == 0) return PQN_OK;
  { LaunchScope _ls(K_RNG, (cudaStream_t)stream); rng_bits_kernel<<<blocks_for(n * len, 256), 256, 0, (cudaStream_t)stream>>>(keys, n, len, out, rng_mode); }
  return check_launch("pqn_rng_bits");
}

int pqn_threefry2x32(const uint32_t* key_pairs, const uint32_t* ctr_pairs, uint32_t* out_pairs, int64_t n,
                     void* stream) {
  if (!key_pairs || !ctr_pairs || !out_pairs || n < 0) return set_error(PQN_E_INVALID, "pqn_threefry2x32: bad argument");
  if (n == 0) return PQN_OK;
  { LaunchScope _ls(K_RNG, (cudaStream_t)stream); threefry_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(key_pairs, ctr_pairs, out_pairs, n); }
  return check_launch("pqn_threefry2x32");
}

int pqn_env_reset(int env_id, const uint32_t* keys, uint32_t* state, float* obs, int64_t N, int max_steps,
                  int rng_mode, void* stream) {
  const pqn_env_params_t defaults = {max_steps, 0};
  return env_reset(env_id, keys, state, obs, N, defaults, rng_mode, stream, "pqn_env_reset");
}

int pqn_env_reset_params(int env_id, const uint32_t* keys, uint32_t* state, float* obs, int64_t N,
                         const pqn_env_params_t* params_host, int rng_mode, void* stream) {
  if (!params_host) return set_error(PQN_E_INVALID, "pqn_env_reset_params: params_host is NULL");
  bool has_memory_length = false;
  PQN_ENV_DISPATCH(env_id, has_memory_length = EnvHasMemoryLength<EnvT>::value);
  if (has_memory_length && params_host->memory_length < 1)
    return set_error(PQN_E_INVALID, "pqn_env_reset_params: memory_length=%d, must be >= 1", params_host->memory_length);
  return env_reset(env_id, keys, state, obs, N, *params_host, rng_mode, stream, "pqn_env_reset_params");
}

int pqn_env_step(int env_id, const uint32_t* keys, uint32_t* state, const int32_t* action, float* obs,
                 float* reward, uint8_t* done, float* info_discount, float* info_ret, int32_t* info_len,
                 int32_t* info_t, int64_t N, int max_steps, int rng_mode, void* stream) {
  if (N == 0) return PQN_OK;
  if (!keys || !state || !action || !reward || !done || N < 0)
    return set_error(PQN_E_INVALID, "pqn_env_step: bad argument");
  PQN_ENV_DISPATCH(env_id, {
    const int ms = max_steps > 0 ? max_steps : EnvT::DEFAULT_MAX_STEPS;
    { LaunchScope _ls(K_ENV_STEP, (cudaStream_t)stream); env_step_kernel<EnvT><<<blocks_for(N, ENV_BLOCK), ENV_BLOCK, 0, (cudaStream_t)stream>>>(
        keys, state, action, obs, reward, done, info_discount, info_ret, info_len, info_t, N, ms, rng_mode); }
  });
  return check_launch("pqn_env_step");
}

int pqn_env_obs_packed(int env_id, const uint32_t* state, uint32_t* obs_packed, int64_t N, void* stream) {
  if (!state || !obs_packed || N < 0) return set_error(PQN_E_INVALID, "pqn_env_obs_packed: bad argument");
  if (N == 0) return PQN_OK;
  PQN_ENV_DISPATCH(env_id, {
    if (!EnvT::BINARY_OBS) return set_error(PQN_E_UNSUPPORTED, "pqn_env_obs_packed: env %d has float observations", env_id);
    { LaunchScope _ls(K_ENV_OBS, (cudaStream_t)stream); env_obs_kernel<EnvT><<<blocks_for(N, ENV_BLOCK), ENV_BLOCK, 0, (cudaStream_t)stream>>>(state, nullptr,
                                                                                           obs_packed, N); }
  });
  return check_launch("pqn_env_obs_packed");
}

int pqn_env_obs(int env_id, const uint32_t* state, float* obs, int64_t N, void* stream) {
  if (!state || !obs || N < 0) return set_error(PQN_E_INVALID, "pqn_env_obs: bad argument");
  if (N == 0) return PQN_OK;
  PQN_ENV_DISPATCH(env_id, {
    { LaunchScope _ls(K_ENV_OBS, (cudaStream_t)stream); env_obs_kernel<EnvT><<<blocks_for(N, ENV_BLOCK), ENV_BLOCK, 0, (cudaStream_t)stream>>>(state, obs, nullptr, N); }
  });
  return check_launch("pqn_env_obs");
}

int pqn_eps_greedy(const uint32_t* keys, const float* q, const float* eps, int32_t* action, int64_t N, int32_t A,
                   int rng_mode, void* stream) {
  if (!keys || !q || !eps || !action || N < 0 || A <= 0 || A >= 65536)
    return set_error(PQN_E_INVALID, "pqn_eps_greedy: bad argument");
  if (N == 0) return PQN_OK;
  { LaunchScope _ls(K_EPS_GREEDY, (cudaStream_t)stream); eps_greedy_kernel<<<blocks_for(N, 256), 256, 0, (cudaStream_t)stream>>>(keys, q, eps, action, N, A, rng_mode); }
  return check_launch("pqn_eps_greedy");
}

int pqn_rollout_act_step(int env_id, const uint32_t* step_keys, const float* q, const float* eps, uint32_t* state,
                         void* obs_next, int64_t obs_seed_stride, int32_t* action, float* reward, uint8_t* done,
                         float* maxq, int64_t tr_seed_stride, double* info_sums, int info_done_only, int32_t S,
                         int32_t E, int32_t env_total, int32_t env_offset, int max_steps, float rew_scale, int rng_mode,
                         void* stream) {
  if (!step_keys || !q || !eps || !state || !obs_next || !action || !reward || !done || !maxq || S <= 0 || E <= 0)
    return set_error(PQN_E_INVALID, "pqn_rollout_act_step: bad argument");
  if (env_total <= 0) { env_total = E; env_offset = 0; }
  if (env_offset < 0 || env_offset + E > env_total)
    return set_error(PQN_E_INVALID, "pqn_rollout_act_step: env shard [%d, %d) outside [0, %d)", env_offset,
                     env_offset + E, env_total);
  if (S > 65535) return set_error(PQN_E_INVALID, "pqn_rollout_act_step: S=%d exceeds gridDim.y", S);
  PQN_ENV_DISPATCH(env_id, {
    const int ms = max_steps > 0 ? max_steps : EnvT::DEFAULT_MAX_STEPS;
    dim3 grid(blocks_for(E, ENV_BLOCK), (unsigned)S);
    { LaunchScope _ls(K_ROLLOUT_ACT_STEP, (cudaStream_t)stream); rollout_act_step_kernel<EnvT><<<grid, ENV_BLOCK, 0, (cudaStream_t)stream>>>(
        step_keys, q, eps, state, obs_next, action, reward, done, maxq, info_sums, E, ms, rew_scale, rng_mode,
        obs_seed_stride, tr_seed_stride, info_done_only, env_total, env_offset); }
  });
  return check_launch("pqn_rollout_act_step");
}

int pqn_rollout_keys(uint32_t* rng_inout, uint32_t* keys_out, int32_t S, int32_t T, int rng_mode, void* stream) {
  if (!rng_inout || !keys_out || S <= 0 || T <= 0) return set_error(PQN_E_INVALID, "pqn_rollout_keys: bad argument");
  { LaunchScope _ls(K_ROLLOUT_KEYS, (cudaStream_t)stream); rollout_keys_kernel<<<blocks_for(S, 64), 64, 0, (cudaStream_t)stream>>>(rng_inout, keys_out, S, T, rng_mode); }
  return check_launch("pqn_rollout_keys");
}

int pqn_qlambda(const float* reward, const uint8_t* done, const float* maxq, const float* q_last, float* targets,
                int32_t T, int32_t S, int32_t E, int32_t A, float gamma, float lambda, void* stream) {
  if (!reward || !done || !maxq || !q_last || !targets || T <= 0 || S <= 0 || E <= 0 || A <= 0)
    return set_error(PQN_E_INVALID, "pqn_qlambda: bad argument");
  { LaunchScope _ls(K_QLAMBDA, (cudaStream_t)stream); qlambda_kernel<<<blocks_for((int64_t)S * E, 256), 256, 0, (cudaStream_t)stream>>>(reward, done, maxq, q_last,
                                                                                    targets, T, S, E, A, gamma, lambda); }
  return check_launch("pqn_qlambda");
}

}  // extern "C"
