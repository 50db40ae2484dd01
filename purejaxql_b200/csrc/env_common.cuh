// Shared pieces of the batched environment operator: the gymnax Environment.step
// auto-reset contract and the LogWrapper accumulator, one env per thread.
//
// Reference seam: purejaxql/pqn_minatar.py:103-112 (gymnax.make + LogWrapper +
// vmapped reset/step).  gymnax==0.0.6 (third party, not vendored) semantics:
//   Environment.step(key, state, action):
//       key, key_reset = split(key)
//       obs_st, state_st, reward, done, info = step_env(key, state, action)
//       obs_re, state_re = reset_env(key_reset)
//       state = select(done, state_re, state_st); obs = select(done, obs_re, obs_st)
//   LogWrapper.step: arithmetic as restated in-tree at
//       purejaxql/utils/craftax_wrappers.py:173-200.
//
// HBM layout of the env state: word-major SoA, `state[w * N + i]` (uint32 words),
// the env's own words first, then the 5 LogWrapper words.  A warp therefore
// reads/writes 128 contiguous bytes per state word.
#pragma once
#include "threefry.cuh"

namespace pqn {

enum EnvId : int {
  ENV_BREAKOUT = 0,
  ENV_ASTERIX = 1,
  ENV_SPACE_INVADERS = 2,
  ENV_FREEWAY = 3,
  ENV_SEAQUEST = 4,
  ENV_CARTPOLE = 16,
  ENV_ACROBOT = 17,
  ENV_MEMORY_CHAIN = 32,
};

constexpr int LOG_WORDS = 5;

PQN_HD uint32_t f2u(float f) {
#if defined(__CUDA_ARCH__)
  return __float_as_uint(f);
#else
  union { float f; uint32_t u; } cv; cv.f = f; return cv.u;
#endif
}
PQN_HD float u2f(uint32_t u) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(u);
#else
  union { float f; uint32_t u; } cv; cv.u = u; return cv.f;
#endif
}

// gymnax.wrappers.purerl.LogEnvState minus env_state.
struct LogState {
  float episode_returns;
  int32_t episode_lengths;
  float returned_episode_returns;
  int32_t returned_episode_lengths;
  int32_t timestep;
};

PQN_HD void log_reset(LogState& l) {
  l.episode_returns = 0.f; l.episode_lengths = 0;
  l.returned_episode_returns = 0.f; l.returned_episode_lengths = 0; l.timestep = 0;
}

// LogWrapper.step bookkeeping (craftax_wrappers.py:186-199 restates it).
PQN_HD void log_step(LogState& l, float reward, bool done) {
  const float new_ret = l.episode_returns + reward;
  const int32_t new_len = l.episode_lengths + 1;
  const float df = done ? 1.f : 0.f;
  const int32_t di = done ? 1 : 0;
  l.episode_returns = new_ret * (1.f - df);
  l.episode_lengths = new_len * (1 - di);
  l.returned_episode_returns = l.returned_episode_returns * (1.f - df) + new_ret * df;
  l.returned_episode_lengths = l.returned_episode_lengths * (1 - di) + new_len * di;
  l.timestep = l.timestep + 1;
}

template <typename W>
PQN_HD void log_load(LogState& l, const W* __restrict__ st, int64_t N, int64_t i, int w0) {
  l.episode_returns = u2f(st[(int64_t)(w0 + 0) * N + i]);
  l.episode_lengths = (int32_t)st[(int64_t)(w0 + 1) * N + i];
  l.returned_episode_returns = u2f(st[(int64_t)(w0 + 2) * N + i]);
  l.returned_episode_lengths = (int32_t)st[(int64_t)(w0 + 3) * N + i];
  l.timestep = (int32_t)st[(int64_t)(w0 + 4) * N + i];
}
PQN_HD void log_store(const LogState& l, uint32_t* __restrict__ st, int64_t N, int64_t i, int w0) {
  st[(int64_t)(w0 + 0) * N + i] = f2u(l.episode_returns);
  st[(int64_t)(w0 + 1) * N + i] = (uint32_t)l.episode_lengths;
  st[(int64_t)(w0 + 2) * N + i] = f2u(l.returned_episode_returns);
  st[(int64_t)(w0 + 3) * N + i] = (uint32_t)l.returned_episode_lengths;
  st[(int64_t)(w0 + 4) * N + i] = (uint32_t)l.timestep;
}

}  // namespace pqn
