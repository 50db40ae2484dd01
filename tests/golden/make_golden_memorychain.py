"""Generates tests/golden/memorychain_traj_original.npz from the MemoryChain oracle (see MEMORYCHAIN.md).

    python tests/golden/make_golden_memorychain.py

Produced by tests/memory_chain_oracle.py (NOT by the reference: jax/gymnax are not installable here); it pins the
CUDA env, its host-compiled logic and the oracle to each other.  Key recipe as make_golden.py: key = PRNGKey(seed);
(key, kr) = split(key); reset keys = split(kr, n); every step (key, ka, ks) = split(key, 3);
action_i = randint(split(ka, n)[i], (), 0, 2); env keys = split(ks, n).  Observations are flattened (3 floats), as
pqn_rnn_gymnax runs the env.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import jax_prng as jr  # noqa: E402
import memory_chain_oracle as MC  # noqa: E402

# (memory_length, steps, seed) per set; each set runs several whole episodes (memory_length + 1 steps)
MEMORY_CHAIN_SETS = ((5, 40, 21), (100, 310, 22))
N_ENVS = 8


def trajectory(memory_length, n, steps, seed, part):
    jr.DEFAULT_PARTITIONABLE = part
    try:
        env = MC.make(flatten=True, memory_length=memory_length)
        key = jr.PRNGKey(seed)
        ks = jr.split(key, 2)
        key, kr = ks[0], ks[1]
        rkeys = jr.split(kr, n)
        obs, st = env.reset(rkeys)
        out = {"reset_keys": rkeys, "obs0": obs, "step_keys": [], "action": [], "obs": [], "reward": [], "done": [],
               "ret": [], "len": []}
        for _ in range(steps):
            ks = jr.split(key, 3)
            key, ka, kst = ks[0], ks[1], ks[2]
            act = jr.randint(jr.split(ka, n), (), 0, env.num_actions)
            sk = jr.split(kst, n)
            obs, st, r, d, info = env.step(sk, st, act)
            out["step_keys"].append(sk); out["action"].append(act); out["obs"].append(obs)
            out["reward"].append(r); out["done"].append(d)
            out["ret"].append(info["returned_episode_returns"]); out["len"].append(info["returned_episode_lengths"])
        res = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in out.items()}
        res["final_time"] = st["time"]
        return res
    finally:
        jr.DEFAULT_PARTITIONABLE = False


def fixture():
    """Both threefry layouts x MEMORY_CHAIN_SETS under keys `ml{memory_length}_{original|partitionable}_{field}`."""
    out = {}
    for ml, steps, seed in MEMORY_CHAIN_SETS:
        for part in (False, True):
            res = trajectory(ml, N_ENVS, steps, seed + 10 * part, part)
            tag = f"ml{ml}_{'partitionable' if part else 'original'}"
            out.update({f"{tag}_{k}": v for k, v in res.items()})
    return out


if __name__ == "__main__":
    np.savez_compressed(os.path.join(HERE, "memorychain_traj_original.npz"), **fixture())
    print("wrote memorychain_traj_original.npz")
