"""MemoryChain-bsuite golden vectors FROM THE REAL REFERENCE STACK (jax + gymnax==0.0.6), for the first machine where
those packages can be imported (see MEMORYCHAIN.md).

    python tests/golden/make_golden_memorychain_from_ref.py [--out tests/golden]

Writes memorychain_episodes_<original|partitionable>_ref.npz: for each (memory_length, steps, seed) of
make_golden_memorychain.MEMORY_CHAIN_SETS, keys ml{memory_length}_<field> with the fields of make_golden_memorychain
(reset_keys, obs0, step_keys[T], action[T], obs[T], reward[T], done[T], ret[T], len[T], final_time) plus the reset
state (reset_context, reset_query) and gymnax's default memory_length (default_memory_length).  Same key recipe as
make_golden_memorychain.py.  tests/test_memory_chain_host.py compares the oracle with these files as soon as they
exist; they settle the four readings of tests/memory_chain_oracle.py (pre-step observation, which half of split(key)
feeds the context, gymnax's default memory_length, bernoulli as uniform < p).
"""
import argparse
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden_memorychain import MEMORY_CHAIN_SETS, N_ENVS  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=HERE)
    args = ap.parse_args()
    try:
        import jax
        import jax.numpy as jnp
        import gymnax
        from gymnax.wrappers.purerl import FlattenObservationWrapper, LogWrapper
    except Exception as e:  # pragma: no cover
        print(f"reference stack unavailable: {e!r}")
        return 3
    import numpy as np
    os.makedirs(args.out, exist_ok=True)

    def trajectory(memory_length, n, steps, seed):
        base, params = gymnax.make("MemoryChain-bsuite")
        default_ml = int(params.memory_length)
        params = params.replace(memory_length=memory_length)
        env = LogWrapper(FlattenObservationWrapper(base))
        A = int(env.action_space(params).n)
        vreset = jax.jit(jax.vmap(env.reset, in_axes=(0, None)))
        vstep = jax.jit(jax.vmap(env.step, in_axes=(0, 0, 0, None)))
        vrand = jax.jit(jax.vmap(lambda k: jax.random.randint(k, (), 0, A)))
        key = jax.random.PRNGKey(seed)
        key, kr = jax.random.split(key)
        rkeys = jax.random.split(kr, n)
        obs, st = vreset(rkeys, params)
        out = {"reset_keys": np.asarray(rkeys), "obs0": np.asarray(obs), "reset_context": np.asarray(st.env_state.context),
               "reset_query": np.asarray(st.env_state.query), "default_memory_length": np.asarray(default_ml),
               "step_keys": [], "action": [], "obs": [], "reward": [], "done": [], "ret": [], "len": []}
        for _ in range(steps):
            key, ka, ks = jax.random.split(key, 3)
            act = vrand(jax.random.split(ka, n)).astype(jnp.int32)
            sk = jax.random.split(ks, n)
            obs, st, r, d, info = vstep(sk, st, act, params)
            out["step_keys"].append(np.asarray(sk)); out["action"].append(np.asarray(act))
            out["obs"].append(np.asarray(obs)); out["reward"].append(np.asarray(r)); out["done"].append(np.asarray(d))
            out["ret"].append(np.asarray(info["returned_episode_returns"]))
            out["len"].append(np.asarray(info["returned_episode_lengths"]))
        res = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in out.items()}
        res["final_time"] = np.asarray(st.env_state.time)
        return res

    for part in (False, True):
        jax.config.update("jax_threefry_partitionable", part)
        tag = "partitionable" if part else "original"
        mc = {}
        for ml, steps, seed in MEMORY_CHAIN_SETS:
            res = trajectory(ml, N_ENVS, steps, seed + 10 * part)
            mc.update({f"ml{ml}_{k}": v for k, v in res.items()})
        np.savez_compressed(os.path.join(args.out, f"memorychain_episodes_{tag}_ref.npz"), **mc)
        print("wrote memorychain", tag, flush=True)
    jax.config.update("jax_threefry_partitionable", False)
    return 0


if __name__ == "__main__":
    sys.exit(main())
