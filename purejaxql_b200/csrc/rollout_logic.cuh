// Per-env pieces of the rollout that are shared by the CUDA kernels and by the
// CPU logic harness used in tests (tests/host_harness.cpp compiles these same
// inline functions with g++; the product never runs them on the host).
#pragma once
#include <type_traits>

#include "env_common.cuh"

namespace pqn {

// Env parameters beyond max_steps (MemoryChain's memory_length) live in the env's state words.  An env that has one
// declares set_memory_length(State&, int); env_set_params writes it before reset_env, which leaves it unchanged.
template <class Env, class = void>
struct EnvHasMemoryLength : std::false_type {};
template <class Env>
struct EnvHasMemoryLength<Env, std::void_t<decltype(&Env::set_memory_length)>> : std::true_type {};

template <class Env>
PQN_HD void env_set_params(typename Env::State& s, int memory_length) {
  if constexpr (EnvHasMemoryLength<Env>::value) Env::set_memory_length(s, memory_length);
}

// gymnax Environment.step (auto-reset) + LogWrapper.step for one env.
template <class Env>
PQN_HD void env_step_full(Key key, int part, int max_steps, typename Env::State& s, LogState& lg, int action,
                          float& reward, bool& done) {
  Key k_step, k_reset;
  split2(key, part, k_step, k_reset);
  Env::step_env(k_step, part, max_steps, s, action, reward, done);
  // reset_env is a pure function of key_reset; evaluating it only where `done`
  // is set is equivalent to gymnax's compute-both-and-select.
  if (done) Env::reset_env(k_reset, part, max_steps, s);
  log_step(lg, reward, done);
}

// eps_greedy_exploration for one env (purejaxql/pqn_minatar.py:115-128).
PQN_HD int eps_greedy_one(Key k, const float* __restrict__ q, int A, float eps, int part, float& maxq) {
  Key rng_a, rng_e;
  split2(k, part, rng_a, rng_e);
  int greedy = 0;
  float best = q[0];
  for (int a = 1; a < A; ++a) {
    const float v = q[a];
    if (v > best) { best = v; greedy = a; }  // strict '>' keeps the first max (jnp.argmax)
  }
  maxq = best;
  const float u = uniform_scalar(rng_e, part);
  const int r = randint_scalar(rng_a, (uint32_t)A, part);
  return (u < eps) ? r : greedy;
}

// Q(lambda) for one env: bootstrap from q_last, reverse scan over T
// (purejaxql/pqn_minatar.py:227-260).  reward/done/maxq/targets are [T][N] views, env column i.
PQN_HD void qlambda_one(const float* __restrict__ reward, const uint8_t* __restrict__ done,
                        const float* __restrict__ maxq, const float* __restrict__ q_last,
                        float* __restrict__ targets, int T, int64_t N, int A, float gamma, float lambda,
                        int64_t i) {
  // q_last points at this env's A bootstrap q-values
  float lq = q_last[0];
  for (int a = 1; a < A; ++a) lq = lq > q_last[a] ? lq : q_last[a];
  const int64_t last = (int64_t)(T - 1) * N + i;
  const float dl = done[last] ? 1.f : 0.f;
  float next_q = lq * (1.f - dl);                       // :252
  float ret = reward[last] + gamma * next_q;            // :253
  targets[last] = ret;
  for (int t = T - 2; t >= 0; --t) {
    const int64_t j = (int64_t)t * N + i;
    const float r = reward[j];
    const float d = done[j] ? 1.f : 0.f;
    const float boot = r + gamma * (1.f - d) * next_q;  // :239-241
    const float delta = ret - next_q;
    ret = boot + gamma * lambda * delta;                // :243-245
    ret = (1.f - d) * ret + d * r;                      // :246-248
    next_q = maxq[j];                                   // :249
    targets[j] = ret;
  }
}

}  // namespace pqn
