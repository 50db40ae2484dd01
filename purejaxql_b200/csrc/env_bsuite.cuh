// bsuite MemoryChain ("MemoryChain-bsuite"), one env per thread.
//
// Restates gymnax==0.0.6 gymnax/environments/bsuite/memory_chain.py (a port of
// bsuite's memory_chain.py; third party, call site purejaxql/pqn_rnn_gymnax.py:134-136)
// with num_bits = 1, which is what gymnax.make builds.  Integer logic plus one
// fp32 true divide in the observation: bit-exact against the oracle.
//
// The env parameter memory_length travels as a state word: pqn_env_reset_params
// writes it before reset_env, and reset_env leaves it as it finds it, so the
// auto-reset inside env_step_full keeps it.
//
// Observation: gymnax's step_env returns get_obs(state) of the state BEFORE the
// step (bsuite's order).  After a step that did not end the episode the old time
// is time - 1; after a reset time is 0 and the reset observation is get_obs(time 0).
// obs_float therefore shows time t = max(time - 1, 0), which is the observation
// the last reset or step returned for this state.
#pragma once
#include "env_common.cuh"

namespace pqn {

struct MemoryChainEnv {
  static constexpr int ID = ENV_MEMORY_CHAIN;
  static constexpr int CORE_WORDS = 6;
  static constexpr int STATE_WORDS = CORE_WORDS + LOG_WORDS;
  static constexpr int NUM_ACTIONS = 2;
  static constexpr int OBS_DIM = 3;
  static constexpr bool BINARY_OBS = false;
  static constexpr bool OBS_IN_REGS = false;
  static constexpr int OBS_WORDS = 1, OBS_WORDS_PAD = 1;
  static constexpr int DEFAULT_MAX_STEPS = 1000;
  static constexpr int DEFAULT_MEMORY_LENGTH = 5;  // gymnax memory_chain.EnvParams()

  struct State {
    int context;        // the one bit to remember (context[0] of gymnax's (num_bits,) array)
    int query;          // always 0 with num_bits = 1
    int total_perfect;
    int total_regret;
    int time;
    int memory_length;  // env parameter, not a gymnax state field
  };

  template <typename W>
  PQN_HD static void load(State& s, const W* __restrict__ st, int64_t N, int64_t i) {
    s.context = (int)st[i]; s.query = (int)st[N + i]; s.total_perfect = (int)st[2 * N + i];
    s.total_regret = (int)st[3 * N + i]; s.time = (int)st[4 * N + i]; s.memory_length = (int)st[5 * N + i];
  }
  PQN_HD static void store(const State& s, uint32_t* __restrict__ st, int64_t N, int64_t i) {
    st[i] = (uint32_t)s.context; st[N + i] = (uint32_t)s.query; st[2 * N + i] = (uint32_t)s.total_perfect;
    st[3 * N + i] = (uint32_t)s.total_regret; st[4 * N + i] = (uint32_t)s.time;
    st[5 * N + i] = (uint32_t)s.memory_length;
  }

  PQN_HD static void set_memory_length(State& s, int memory_length) { s.memory_length = memory_length; }

  PQN_HD static void reset_env(Key key, int part, int /*max_steps*/, State& s) {
    // key_context, key_query = split(key); context = bernoulli(key_context, 0.5, (1,)) = uniform(.., (1,)) < 0.5;
    // query = randint(key_query, (), 0, num_bits) is 0 for num_bits = 1 whatever the key
    Key k_context, k_query;
    split2(key, part, k_context, k_query);
    s.context = uniform_from_bits(bits_at(k_context, 1u, 0u, part), 0.0f, 1.0f) < 0.5f ? 1 : 0;
    s.query = 0;
    s.total_perfect = 0; s.total_regret = 0; s.time = 0;
  }

  PQN_HD static void step_env(Key /*key*/, int /*part*/, int max_steps, State& s, int action, float& reward,
                              bool& done) {
    s.time = s.time + 1;
    const bool mem_full = !(s.time - 1 < s.memory_length);
    const bool correct = action == s.context;  // context[query], query = 0
    const bool mem_correct = mem_full && correct;
    const bool mem_wrong = mem_full && !correct;
    reward = (mem_correct ? 1.0f : 0.0f) - (mem_wrong ? 1.0f : 0.0f);
    s.total_perfect = s.total_perfect + (mem_correct ? 1 : 0);
    s.total_regret = s.total_regret + (mem_wrong ? 2 : 0);
    done = (s.time - 1 == s.memory_length) || s.time >= max_steps;
  }

  PQN_HD static void obs_float(const State& s, float (&o)[OBS_DIM]) {
    const int t = s.time > 0 ? s.time - 1 : 0;
    o[0] = 1.0f - (float)t / (float)s.memory_length;
    o[1] = t == s.memory_length - 1 ? (float)s.query : 0.0f;
    o[2] = t == 0 ? (float)(2 * s.context - 1) : 0.0f;
  }
};

}  // namespace pqn
