"""CPU: MemoryChain-bsuite — the oracle against a hand-written table and the golden fixture, the device logic
(csrc/env_bsuite.cuh compiled with g++) against the oracle bit for bit, the preset, and the memory_length check."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import memory_chain_oracle as MC
from oracle import jax_prng as jr

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "memorychain_traj_original.npz")
F32 = np.float32


@pytest.fixture
def layout():
    yield lambda part: setattr(jr, "DEFAULT_PARTITIONABLE", bool(part))
    jr.DEFAULT_PARTITIONABLE = False


# --------------------------------------------------------------------------- #
# the oracle against a hand-written episode table (memory_length = 3)
# --------------------------------------------------------------------------- #
def test_oracle_matches_hand_written_table():
    """Two episodes of one env: the right answer, then the wrong one.  Step k of an episode returns the observation of
    time k-1 (bsuite's pre-step order); the answer is scored on step memory_length + 1, which also ends the episode
    and returns the auto-reset observation."""
    ml = 3
    env = MC.make(flatten=True, memory_length=ml)
    obs, st = env.reset(jr.split(jr.PRNGKey(3), 1))
    sign = obs[0, 2]
    assert sign in (-1.0, 1.0)
    assert obs.tolist() == [[1.0, 0.0, sign]]
    context = int(sign > 0)
    t13, t23 = F32(0.6666666269302368), F32(0.3333333134651184)     # fp32 1 - 1/3 and 1 - 2/3
    ep_return, ep_len = 0.0, 0
    for episode, right in enumerate((True, False)):
        answer = context if right else 1 - context
        #         action, obs emitted,          reward,                   done
        table = [(0, [1.0, 0.0, sign], 0.0, False),
                 (1, [t13, 0.0, 0.0], 0.0, False),
                 (0, [t23, 0.0, 0.0], 0.0, False),
                 (answer, None, 1.0 if right else -1.0, True)]
        for k, (a, want_obs, want_r, want_d) in enumerate(table):
            key = jr.split(jr.PRNGKey(100 + 10 * episode + k), 1)
            if k == 3:   # the scoring step's state before the auto-reset
                inner = {kk: v for kk, v in st.items() if not kk.startswith("log_")}
                ks = jr.split(key, 2)
                _, s_st, _, _, _ = env.env.core.step_env(ks[:, 0], inner, np.array([a], np.int32))
                assert s_st["time"].tolist() == [ml + 1]
                assert (s_st["total_perfect"].tolist(), s_st["total_regret"].tolist()) == (([1], [0]) if right else ([0], [2]))
            obs, st, r, d, info = env.step(key, st, np.array([a], np.int32))
            ep_return, ep_len = ep_return + float(r[0]), ep_len + 1
            if want_obs is not None:
                assert obs.tolist() == [want_obs], (episode, k)
                assert st["time"].tolist() == [k + 1]
            else:                                   # reset observation of the next episode
                assert obs[0, 0] == 1.0 and obs[0, 1] == 0.0 and obs[0, 2] in (-1.0, 1.0)
                assert st["time"].tolist() == [0] and st["total_perfect"].tolist() == [0]
                sign, context = obs[0, 2], int(obs[0, 2] > 0)
            assert r.tolist() == [want_r] and d.tolist() == [want_d], (episode, k)
            assert info["discount"].tolist() == [0.0 if want_d else 1.0]
            assert st["log_episode_returns"].tolist() == [0.0 if want_d else ep_return]
            assert st["log_episode_lengths"].tolist() == [0 if want_d else ep_len]
            assert st["log_timestep"].tolist() == [4 * episode + k + 1]
        assert st["log_returned_episode_returns"].tolist() == [1.0 if right else -1.0]
        assert st["log_returned_episode_lengths"].tolist() == [ml + 1]
        ep_return, ep_len = 0.0, 0


def test_oracle_step_limit_ends_episode_without_reward():
    env = MC.make(flatten=True, memory_length=10, max_steps_in_episode=4)
    obs, st = env.reset(jr.split(jr.PRNGKey(0), 5))
    for k in range(4):
        obs, st, r, d, _ = env.step(jr.split(jr.PRNGKey(k), 5), st, np.zeros(5, np.int32))
        assert (r == 0).all() and d.all() == (k == 3)


def test_default_memory_length_matches_library_default():
    from purejaxql_b200 import envs
    assert MC.DEFAULT_MEMORY_LENGTH == envs.MEMORY_CHAIN_DEFAULT_MEMORY_LENGTH == 5
    src = open(os.path.join(os.path.dirname(HERE), "purejaxql_b200", "csrc", "env_bsuite.cuh")).read()
    assert "DEFAULT_MEMORY_LENGTH = 5;" in src


# --------------------------------------------------------------------------- #
# golden fixture
# --------------------------------------------------------------------------- #
def _sets():
    g = dict(np.load(GOLD))
    from golden.make_golden_memorychain import MEMORY_CHAIN_SETS
    for ml, _, _ in MEMORY_CHAIN_SETS:
        for part, name in ((0, "original"), (1, "partitionable")):
            yield ml, part, {k[len(f"ml{ml}_{name}_"):]: v for k, v in g.items() if k.startswith(f"ml{ml}_{name}_")}


def test_oracle_against_golden(layout):
    seen = 0
    for ml, part, g in _sets():
        layout(part)
        env = MC.make(flatten=True, memory_length=ml)
        obs, st = env.reset(g["reset_keys"])
        assert np.array_equal(obs, g["obs0"])
        for t in range(g["action"].shape[0]):
            obs, st, r, d, info = env.step(g["step_keys"][t], st, g["action"][t])
            assert np.array_equal(obs, g["obs"][t]) and np.array_equal(r, g["reward"][t]), (ml, part, t)
            assert np.array_equal(d, g["done"][t]) and np.array_equal(info["returned_episode_returns"], g["ret"][t])
            assert np.array_equal(info["returned_episode_lengths"], g["len"][t])
        # several whole episodes of memory_length + 1 steps, returns +-1, both answers present
        assert g["done"].sum(0).min() >= 3
        assert set(np.unique(g["ret"][g["done"]])) == {-1.0, 1.0}
        assert (g["len"][g["done"]] == ml + 1).all()
        assert set(np.unique(g["reward"])) == {-1.0, 0.0, 1.0}
        seen += 1
    assert seen == 4


# --------------------------------------------------------------------------- #
# the device logic on the host, bit for bit
# --------------------------------------------------------------------------- #
@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("mc") / "memory_chain_harness.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC",
                           os.path.join(HERE, "memory_chain_harness.cpp"), "-o", so])
    lib = ctypes.CDLL(so)
    vp, i64 = ctypes.c_void_p, ctypes.c_int64
    lib.mc_reset.argtypes = [vp, vp, vp, i64, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.mc_step.argtypes = [vp, vp, vp, vp, vp, vp, i64, ctypes.c_int, ctypes.c_int]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _host_reset(lib, keys, ml, part, max_steps=1000):
    n = keys.shape[0]
    keys = np.ascontiguousarray(keys, np.uint32)
    state = np.zeros((lib.mc_state_words(), n), np.uint32)
    obs = np.zeros((n, 3), np.float32)
    lib.mc_reset(_p(keys), _p(state), _p(obs), n, max_steps, ml, part)
    return obs, state


def _host_step(lib, keys, state, action, part, max_steps=1000):
    n = keys.shape[0]
    keys = np.ascontiguousarray(keys, np.uint32)
    action = np.ascontiguousarray(action, np.int32)
    obs, reward, done = np.zeros((n, 3), np.float32), np.zeros(n, np.float32), np.zeros(n, np.uint8)
    lib.mc_step(_p(keys), _p(state), _p(action), _p(obs), _p(reward), _p(done), n, max_steps, part)
    return obs, reward, done.astype(bool)


def _check_state(state, st, ml):
    assert np.array_equal(state[0], st["context"][:, 0]) and np.array_equal(state[1], st["query"])
    assert np.array_equal(state[2], st["total_perfect"]) and np.array_equal(state[3], st["total_regret"])
    assert np.array_equal(state[4], st["time"]) and (state[5] == ml).all()
    assert np.array_equal(state[6].view(np.float32), st["log_episode_returns"])
    assert np.array_equal(state[7], st["log_episode_lengths"])
    assert np.array_equal(state[8].view(np.float32), st["log_returned_episode_returns"])
    assert np.array_equal(state[9], st["log_returned_episode_lengths"]) and np.array_equal(state[10], st["log_timestep"])


@pytest.mark.parametrize("part", [0, 1])
@pytest.mark.parametrize("ml,steps", [(1, 12), (3, 40), (100, 230)])
def test_device_logic_matches_oracle(harness, layout, part, ml, steps):
    layout(part)
    n = 64
    env = MC.make(flatten=True, memory_length=ml)
    rk = jr.split(jr.PRNGKey(ml), n)
    o_obs, o_st = env.reset(rk)
    h_obs, h_state = _host_reset(harness, rk, ml, part)
    assert np.array_equal(h_obs, o_obs)
    _check_state(h_state, o_st, ml)
    rng = np.random.default_rng(ml)
    for t in range(steps):
        sk = jr.split(jr.PRNGKey(1000 + t), n)
        act = rng.integers(0, 2, n).astype(np.int32)
        o_obs, o_st, o_r, o_d, _ = env.step(sk, o_st, act)
        h_obs, h_r, h_d = _host_step(harness, sk, h_state, act, part)
        assert np.array_equal(h_obs, o_obs) and np.array_equal(h_r, o_r) and np.array_equal(h_d, o_d), t
        _check_state(h_state, o_st, ml)


def test_device_logic_matches_golden(harness, layout):
    for ml, part, g in _sets():
        layout(part)
        h_obs, state = _host_reset(harness, g["reset_keys"], ml, part)
        assert np.array_equal(h_obs, g["obs0"])
        for t in range(g["action"].shape[0]):
            h_obs, h_r, h_d = _host_step(harness, g["step_keys"][t], state, g["action"][t], part)
            assert np.array_equal(h_obs, g["obs"][t]) and np.array_equal(h_r, g["reward"][t]), (ml, part, t)
            assert np.array_equal(h_d, g["done"][t])
        assert np.array_equal(state[4], g["final_time"])


# --------------------------------------------------------------------------- #
# preset and parameter validation
# --------------------------------------------------------------------------- #
def test_preset_composes_to_reference_values():
    from purejaxql_b200 import config_loader as C
    c = C.compose(["+alg=pqn_rnn_memory_chain", "NUM_SEEDS=8"])
    a = c["alg"]
    want = dict(ALG_NAME="pqn_rnn", TOTAL_TIMESTEPS=1e5, TOTAL_TIMESTEPS_DECAY=1e5, NUM_ENVS=32, MEMORY_WINDOW=4,
                NUM_STEPS=128, EPS_START=1.0, EPS_FINISH=0.01, EPS_DECAY=0.1, NUM_MINIBATCHES=16, NUM_EPOCHS=4,
                NORM_INPUT=False, HIDDEN_SIZE=256, NUM_LAYERS=2, NORM_TYPE="layer_norm", LR=0.001, MAX_GRAD_NORM=10,
                LR_LINEAR_DECAY=False, REW_SCALE=1.0, GAMMA=0.99, LAMBDA=0.95, ENV_NAME="MemoryChain-bsuite",
                ENV_KWARGS={"memory_length": 100}, TEST_DURING_TRAINING=True, TEST_INTERVAL=0.05, TEST_NUM_ENVS=128,
                EPS_TEST=0.0)
    for k, v in want.items():
        assert a[k] == v and type(a[k]) is type(v), (k, a[k], v)
    assert "TEST_NUM_STEPS" not in a                        # set from max_steps_in_episode (1000) by make_train
    assert a["TOTAL_TIMESTEPS"] // a["NUM_STEPS"] // a["NUM_ENVS"] == 24
    assert C.compose(["+alg=pqn_rnn_memory_chain", "alg.ENV_KWARGS.memory_length=7"])["alg"]["ENV_KWARGS"] == \
        {"memory_length": 7}


@pytest.mark.parametrize("bad", [0, -3, 2.5])
def test_bad_memory_length_is_rejected_before_device_work(bad, monkeypatch):
    from purejaxql_b200 import _lib, config_loader as C, pqn_rnn_gymnax
    c = C.compose(["+alg=pqn_rnn_memory_chain"])
    cfg = {**c, **c["alg"]}
    cfg["ENV_KWARGS"] = {"memory_length": bad}
    touched = []
    monkeypatch.setattr(_lib, "lib", lambda: touched.append(1))   # any library call would be device work
    with pytest.raises(ValueError, match="memory_length must be an integer"):
        pqn_rnn_gymnax.make_train(cfg)
    assert not touched


def test_env_params_and_state_fields_roundtrip():
    import torch
    from purejaxql_b200 import envs
    with pytest.raises(TypeError, match="memory_length"):
        envs.make("CartPole-v1", env_kwargs={"memory_length": 4})
    _, p = envs.make("MemoryChain-bsuite", env_kwargs={"memory_length": 100})
    assert p == envs.EnvParams(max_steps_in_episode=1000, memory_length=100)
    assert envs.make("MemoryChain-bsuite")[1].memory_length == 5 and envs.make("Acrobot-v1")[1].memory_length is None
    env = MC.make(flatten=True, memory_length=100)
    _, st = env.reset(jr.split(jr.PRNGKey(1), 9))
    for t in range(3):
        _, st, *_ = env.step(jr.split(jr.PRNGKey(t), 9), st, np.ones(9, np.int32))
    f = {k: torch.from_numpy(np.asarray(v)) for k, v in st.items()}
    state = envs.fields_to_state("MemoryChain-bsuite", f, p)
    assert tuple(state.shape) == (11, 9) and (state[5] == 100).all()
    back = envs.state_to_fields("MemoryChain-bsuite", state)
    assert (back.pop("param_memory_length") == 100).all()
    assert set(back) == set(f)
    for k in f:
        assert torch.equal(back[k], f[k].to(back[k].dtype)), k


_REF = {part: os.path.join(HERE, "golden", f"memorychain_episodes_{name}_ref.npz")
        for part, name in ((0, "original"), (1, "partitionable"))}


@pytest.mark.skipif(not any(os.path.exists(p) for p in _REF.values()),
                    reason="no reference-generated MemoryChain vectors committed (jax/gymnax never reachable)")
@pytest.mark.parametrize("part", [0, 1])
def test_oracle_against_reference_generated_memory_chain(layout, part):
    """Settles the four recorded readings once make_golden_memorychain_from_ref.py has run against the real gymnax."""
    if not os.path.exists(_REF[part]):
        pytest.skip("layout not recorded")
    layout(part)
    z = dict(np.load(_REF[part]))
    for ml in (5, 100):
        g = {k[len(f"ml{ml}_"):]: v for k, v in z.items() if k.startswith(f"ml{ml}_")}
        env = MC.make(flatten=True, memory_length=ml)
        obs, st = env.reset(g["reset_keys"])
        assert np.array_equal(st["context"], g["reset_context"].reshape(st["context"].shape))   # readings 2 and 4
        assert np.array_equal(obs, g["obs0"].reshape(obs.shape))
        for t in range(g["action"].shape[0]):
            obs, st, r, d, info = env.step(g["step_keys"][t], st, g["action"][t])
            assert np.array_equal(obs, g["obs"][t].reshape(obs.shape)), (ml, t)                  # reading 1
            assert np.array_equal(r, g["reward"][t]) and np.array_equal(d, g["done"][t]), (ml, t)
            assert np.array_equal(info["returned_episode_lengths"], g["len"][t]), (ml, t)
