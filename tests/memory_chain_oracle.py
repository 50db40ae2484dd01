"""NumPy restatement of bsuite MemoryChain as gymnax==0.0.6 builds it (``MemoryChain-bsuite``, num_bits = 1).

TEST INFRASTRUCTURE, the oracle of ``purejaxql_b200/csrc/env_bsuite.cuh``.  It composes with the gymnax core of
``oracle/gymnax_envs.py`` (``Environment`` auto-reset, ``LogWrapper``), which it does not modify.  PARITY UNPINNED:
gymnax (``gymnax/environments/bsuite/memory_chain.py``, a port of bsuite's ``memory_chain.py``) is not installable here,
so this restates the published algorithm from memory.  Four readings could not be checked; each is recorded in
DESIGN.md and tests/golden/MEMORYCHAIN.md, and ``tests/golden/make_golden_memorychain_from_ref.py`` records the
trajectories that pin them on a machine with jax and gymnax:

1. ``step_env`` returns ``get_obs`` of the state BEFORE the step (bsuite's order);
2. ``key_context, key_query = split(key)``: the first half feeds the context;
3. gymnax's default ``EnvParams().memory_length`` is 5;
4. ``bernoulli(key, 0.5, (1,))`` is ``uniform(key, (1,)) < 0.5``.

Reference call site: ``purejaxql/pqn_rnn_gymnax.py:134-136`` (``EnvParams(memory_length=ENV_KWARGS.get(..., 10))``).
"""
from __future__ import annotations

import numpy as np

from oracle import gymnax_envs as G
from oracle import jax_prng as jr

F32 = np.float32
I32 = np.int32

NAME = "MemoryChain-bsuite"
DEFAULT_MEMORY_LENGTH = 5


class MemoryChain:
    name = NAME
    obs_shape = (1, 3)                    # gymnax's (1, num_bits + 2); FlattenObservationWrapper makes it 3
    num_actions = 2
    num_bits = 1
    state_fields = ("context", "query", "total_perfect", "total_regret", "time")

    def __init__(self, memory_length: int = DEFAULT_MEMORY_LENGTH, max_steps_in_episode: int = 1000):
        self.memory_length = int(memory_length)
        self.max_steps_in_episode = int(max_steps_in_episode)

    def get_obs(self, s):
        n = s["time"].shape[0]
        t = s["time"]
        obs = np.zeros((n, 1, self.num_bits + 2), F32)
        obs[:, 0, 0] = F32(1) - t.astype(F32) / F32(self.memory_length)            # fp32 true divide
        obs[:, 0, 1] = np.where(t == self.memory_length - 1, s["query"], 0).astype(F32)
        obs[:, 0, 2:] = np.where((t == 0)[:, None], 2 * s["context"] - 1, 0).astype(F32)
        return obs

    def reset_env(self, key):
        n = key.shape[0]
        ks = jr.split(key, 2)
        key_context, key_query = ks[:, 0], ks[:, 1]
        context = jr.bernoulli(key_context, 0.5, (self.num_bits,)).astype(I32)    # [N, 1]
        query = jr.randint(key_query, (), 0, self.num_bits)                       # 0 for num_bits = 1
        s = dict(context=context, query=query.astype(I32), total_perfect=np.zeros(n, I32),
                 total_regret=np.zeros(n, I32), time=np.zeros(n, I32))
        return self.get_obs(s), s

    def step_env(self, key, s, action):
        obs = self.get_obs(s)                                                     # reading 1: pre-step observation
        time = (s["time"] + 1).astype(I32)
        mem_not_full = time - 1 < self.memory_length
        correct = action == s["context"][np.arange(action.shape[0]), s["query"]]
        mem_correct = ~mem_not_full & correct
        mem_wrong = ~mem_not_full & ~correct
        reward = (mem_correct.astype(F32) - mem_wrong.astype(F32)).astype(F32)
        ns = dict(context=s["context"].copy(), query=s["query"].copy(),
                  total_perfect=(s["total_perfect"] + mem_correct).astype(I32),
                  total_regret=(s["total_regret"] + 2 * mem_wrong).astype(I32), time=time)
        done = (time - 1 == self.memory_length) | (time >= self.max_steps_in_episode)
        info = {"discount": np.where(done, F32(0.0), F32(1.0)).astype(F32)}
        return obs, ns, reward, done, info


def make(flatten: bool = False, log: bool = True, memory_length: int = DEFAULT_MEMORY_LENGTH,
         max_steps_in_episode: int = 1000):
    """``gymnax.make("MemoryChain-bsuite")`` with ``EnvParams(memory_length, max_steps_in_episode)``, wrapped like
    ``oracle.gymnax_envs.make`` (FlattenObservationWrapper as in pqn_rnn_gymnax.py:137, LogWrapper)."""
    env = G.Environment(MemoryChain(memory_length, max_steps_in_episode), flatten=flatten)
    return G.LogWrapper(env) if log else env
