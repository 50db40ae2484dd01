// CPU logic harness for MemoryChain — TEST INFRASTRUCTURE ONLY (built by tests/test_memory_chain_host.py).
// Compiles the same inline env functions the CUDA kernels use (csrc/env_bsuite.cuh, rollout_logic.cuh) with g++,
// and drives them the way env_reset_kernel / env_step_kernel do, so the device logic can be checked against the
// oracle without a GPU.
#include <stdint.h>

#include "../purejaxql_b200/csrc/env_bsuite.cuh"
#include "../purejaxql_b200/csrc/rollout_logic.cuh"

using namespace pqn;
using Env = MemoryChainEnv;

extern "C" {
int mc_state_words() { return Env::STATE_WORDS; }

void mc_reset(const uint32_t* keys, uint32_t* state, float* obs, int64_t N, int max_steps, int memory_length,
              int part) {
  for (int64_t i = 0; i < N; ++i) {
    Env::State s;
    env_set_params<Env>(s, memory_length);
    Env::reset_env(Key{keys[2 * i], keys[2 * i + 1]}, part, max_steps, s);
    Env::store(s, state, N, i);
    LogState lg;
    log_reset(lg);
    log_store(lg, state, N, i, Env::CORE_WORDS);
    float o[Env::OBS_DIM];
    Env::obs_float(s, o);
    for (int f = 0; f < Env::OBS_DIM; ++f) obs[i * Env::OBS_DIM + f] = o[f];
  }
}

void mc_step(const uint32_t* keys, uint32_t* state, const int32_t* action, float* obs, float* reward, uint8_t* done,
             int64_t N, int max_steps, int part) {
  for (int64_t i = 0; i < N; ++i) {
    Env::State s;
    Env::load(s, state, N, i);
    LogState lg;
    log_load(lg, state, N, i, Env::CORE_WORDS);
    float r;
    bool d;
    env_step_full<Env>(Key{keys[2 * i], keys[2 * i + 1]}, part, max_steps, s, lg, action[i], r, d);
    Env::store(s, state, N, i);
    log_store(lg, state, N, i, Env::CORE_WORDS);
    reward[i] = r;
    done[i] = d ? 1 : 0;
    float o[Env::OBS_DIM];
    Env::obs_float(s, o);
    for (int f = 0; f < Env::OBS_DIM; ++f) obs[i * Env::OBS_DIM + f] = o[f];
  }
}
}
