"""Recurrent (GRU) PQN on gymnax classic control and bsuite MemoryChain — drop-in for purejaxql/pqn_rnn_gymnax.py.

    python -m purejaxql_b200.pqn_rnn_gymnax +alg=pqn_rnn_cartpole NUM_SEEDS=4
    python -m purejaxql_b200.pqn_rnn_gymnax +alg=pqn_rnn_memory_chain NUM_SEEDS=8

``make_train(config)`` keeps the reference's contract (pqn_rnn_gymnax.py:117-560): config mutation (NUM_UPDATES,
NUM_UPDATES_DECAY, TEST_NUM_STEPS), ``RNNQNetwork`` (MLP trunk -> one-hot last action -> scanned GRU with done-resets ->
Q head), a memory of MEMORY_WINDOW + NUM_STEPS transitions warmed up with random actions, minibatches over ENVS (whole
trajectories) and the Q(lambda) targets computed inside the loss from the window's own q values.  For
MemoryChain-bsuite the env parameters are ``EnvParams(memory_length=ENV_KWARGS.get("memory_length", 10))`` (:134-136);
other envs run with gymnax's defaults.  As in the other
scripts ``train(rngs)`` takes the ``[NUM_SEEDS, 2]`` key array natively.
"""
from __future__ import annotations

from . import _runner, envs
from .engine import prepare_config
from .engine_rnn import PQNRnnEngine


def make_train(config):
    env_kwargs = {}
    if config["ENV_NAME"] == "MemoryChain-bsuite":                         # :134-136
        env_kwargs["memory_length"] = (config.get("ENV_KWARGS") or {}).get("memory_length", 10)
    env, env_params = envs.make(config["ENV_NAME"], flatten_obs=True, env_kwargs=env_kwargs)   # :134-139, validates
    prepare_config(config, env_params.max_steps_in_episode, allow_test_steps_override=True)    # :119-132,140
    engine = PQNRnnEngine(config, env_params=env_params)

    def train(rngs):
        return engine.train(rngs)

    train.engine = engine
    return train


def single_run(config):
    return _runner.single_run(config, make_train, alg_file_name="pqn_rnn")


def main(argv=None):
    return _runner.main(make_train, argv)


if __name__ == "__main__":
    main()
