"""GPU: MemoryChain-bsuite on the B200 against the oracle (tests/memory_chain_oracle.py) — the env operator with
explicit parameters, the fused rollout step, whole recurrent updates, CUDA-graph replay, the preset with evaluation and
the feed-forward script."""
import numpy as np
import pytest
import torch

import memory_chain_oracle as MC
from oracle import jax_prng as jr
from oracle import pqn_ref as R
from oracle import pqn_rnn_ref as RR
from test_gpu_rnn import _oracle_step

pytestmark = pytest.mark.gpu

NAME = "MemoryChain-bsuite"


def dev():
    return torch.device("cuda:0")


@pytest.fixture
def layout():
    yield lambda part: setattr(jr, "DEFAULT_PARTITIONABLE", bool(part))
    jr.DEFAULT_PARTITIONABLE = False


def _keys(k):
    from purejaxql_b200 import jaxrandom
    return jaxrandom.as_key_tensor(k, dev())


def _check_state(env_name, state, st, ml):
    from purejaxql_b200 import envs
    f = envs.state_to_fields(env_name, state.cpu())
    assert (f.pop("param_memory_length") == ml).all()
    for k, v in st.items():
        got = f[k].numpy()
        assert np.array_equal(got, np.asarray(v).astype(got.dtype)), k


@pytest.mark.parametrize("part", [0, 1])
@pytest.mark.parametrize("ml", [3, 100])
@pytest.mark.parametrize("N", [1000, 65536])
def test_reset_params_and_step_match_oracle(layout, part, ml, N):
    from purejaxql_b200 import envs
    layout(part)
    env, params = envs.make(NAME, flatten_obs=True, rng_mode=part, env_kwargs={"memory_length": ml})
    oenv = MC.make(flatten=True, memory_length=ml)
    rk = jr.split(jr.PRNGKey(7 + ml), N)
    obs, st = env.reset(_keys(rk), params)
    o_obs, o_st = oenv.reset(rk)
    assert np.array_equal(obs.cpu().numpy(), o_obs)
    _check_state(NAME, st, o_st, ml)
    steps = 2 * (ml + 1) + 3                        # two whole episodes and the start of a third
    rng = np.random.default_rng(N + ml)
    for t in range(steps):
        sk = jr.split(jr.PRNGKey(300 + t), N)
        act = rng.integers(0, 2, N).astype(np.int32)
        obs, st, r, d, info = env.step(_keys(sk), st, torch.from_numpy(act).to(dev()), params)
        o_obs, o_st, o_r, o_d, o_info = oenv.step(sk, o_st, act)
        assert np.array_equal(obs.cpu().numpy(), o_obs), t
        assert np.array_equal(r.cpu().numpy(), o_r) and np.array_equal(d.cpu().numpy(), o_d), t
        for k in ("discount", "returned_episode_returns", "returned_episode_lengths", "timestep"):
            assert np.array_equal(info[k].cpu().numpy(), o_info[k]), (t, k)
    _check_state(NAME, st, o_st, ml)
    assert o_st["log_returned_episode_lengths"].min() == ml + 1


@pytest.mark.parametrize("part", [0, 1])
def test_old_reset_uses_default_params(layout, part):
    from purejaxql_b200 import _lib, envs
    layout(part)
    N = 1000
    env, params = envs.make(NAME, flatten_obs=True, rng_mode=part)
    assert params.memory_length == 5
    keys = _keys(jr.split(jr.PRNGKey(4), N))
    obs_p, st_p = env.reset(keys, params)
    st = torch.empty_like(st_p)
    obs = torch.empty_like(obs_p)
    _lib.check(_lib.lib().pqn_env_reset(env.env_id, _lib.p(keys), _lib.p(st), _lib.p(obs), N, 0, part,
                                        _lib.stream_ptr()), "pqn_env_reset")
    torch.cuda.synchronize()
    assert torch.equal(st, st_p) and torch.equal(obs, obs_p) and (st[5] == 5).all()
    # ... and the default episode is memory_length + 1 = 6 steps long
    o_obs, o_st = MC.make(flatten=True).reset(jr.split(jr.PRNGKey(4), N))
    assert np.array_equal(obs.cpu().numpy(), o_obs)


def test_reset_params_rejects_memory_length_below_one():
    from purejaxql_b200 import _lib, envs
    env, _ = envs.make(NAME)
    keys = _keys(jr.split(jr.PRNGKey(0), 8))
    st = torch.zeros((env.state_words, 8), dtype=torch.int32, device=dev())
    rc = _lib.lib().pqn_env_reset_params(env.env_id, _lib.p(keys), _lib.p(st), None, 8, _lib.EnvParams(0, 0), 0,
                                         _lib.stream_ptr())
    assert rc != 0 and b"memory_length" in _lib.lib().pqn_last_error()
    assert (st == 0).all()


@pytest.mark.parametrize("part", [0, 1])
def test_rollout_act_step_matches_oracle(layout, part):
    """pqn_rollout_act_step on MemoryChain: per-env keys split from the step's (rng_a, rng_s), eps-greedy, the env step
    with auto-reset, the transition stores and the per-seed info sums, S = 3 seeds x E = 37 envs."""
    from purejaxql_b200 import _lib, envs
    layout(part)
    S, E, A, ml = 3, 37, 2, 3
    env, params = envs.make(NAME, flatten_obs=True, rng_mode=part, env_kwargs={"memory_length": ml})
    oenv = MC.make(flatten=True, memory_length=ml)
    rk = jr.split(jr.PRNGKey(11), S * E)
    _, state = env.reset(_keys(rk), params)
    o_st = [oenv.reset(rk[s * E:(s + 1) * E])[1] for s in range(S)]
    eps = torch.full((1,), 0.5, device=dev())
    rng = np.random.default_rng(2)
    sums = torch.zeros((S, 5), dtype=torch.float64, device=dev())
    want = np.zeros((S, 5))
    obs_next = torch.empty((S, E, 3), device=dev())
    act, rew = torch.empty((S, E), dtype=torch.int32, device=dev()), torch.empty((S, E), device=dev())
    done, maxq = torch.empty((S, E), dtype=torch.uint8, device=dev()), torch.empty((S, E), device=dev())
    for t in range(3 * (ml + 1)):
        step_keys = jr.split(jr.PRNGKey(50 + t), 2 * S).reshape(S, 2, 2)
        q = rng.standard_normal((S * E, A)).astype(np.float32)
        sk_d = _keys(step_keys.reshape(S * 2, 2)).reshape(S, 2, 2).contiguous()   # held: the launch is asynchronous
        q_d = torch.from_numpy(q).to(dev())
        _lib.check(_lib.lib().pqn_rollout_act_step(
            env.env_id, _lib.p(sk_d), _lib.p(q_d), _lib.p(eps), _lib.p(state), _lib.p(obs_next), E, _lib.p(act),
            _lib.p(rew), _lib.p(done), _lib.p(maxq), E, _lib.p(sums), 0, S, E, 0, 0, 0, 1.0, part, _lib.stream_ptr()),
            "pqn_rollout_act_step")
        torch.cuda.synchronize()
        for s in range(S):
            qs = q[s * E:(s + 1) * E]
            a = R.eps_greedy(jr.split(step_keys[s, 0], E), qs, 0.5)
            o_obs, o_st[s], o_r, o_d, info = oenv.step(jr.split(step_keys[s, 1], E), o_st[s], a)
            assert np.array_equal(act[s].cpu().numpy(), a), (t, s)
            assert np.array_equal(obs_next[s].cpu().numpy(), o_obs), (t, s)
            assert np.array_equal(rew[s].cpu().numpy(), o_r) and np.array_equal(done[s].cpu().numpy(), o_d), (t, s)
            assert np.array_equal(maxq[s].cpu().numpy(), qs.max(-1))
            want[s] += [info["returned_episode_returns"].sum(), info["returned_episode_lengths"].sum(),
                        info["timestep"].sum(), o_d.sum(), info["discount"].sum()]
        assert np.array_equal(sums.cpu().numpy(), want), t
    for s in range(S):
        _check_state(NAME, state[:, s * E:(s + 1) * E], o_st[s], ml)


def _mc_cfg(**kw):
    cfg = dict(ENV_NAME=NAME, ENV_KWARGS={"memory_length": 4}, NUM_ENVS=8, NUM_STEPS=12, MEMORY_WINDOW=3,
               NUM_MINIBATCHES=4, NUM_EPOCHS=2, EPS_START=1.0, EPS_FINISH=1.0, EPS_DECAY=0.2, LR=1e-3, MAX_GRAD_NORM=10,
               GAMMA=0.99, LAMBDA=0.95, NORM_TYPE="layer_norm", NORM_INPUT=False, HIDDEN_SIZE=128, NUM_LAYERS=2,
               LR_LINEAR_DECAY=False, REW_SCALE=1.0, WANDB_MODE="disabled", TEST_DURING_TRAINING=False)
    cfg.update(kw)
    return cfg


def test_rnn_update_steps_match_oracle_on_memory_chain():
    """Two whole updates of pqn_rnn_gymnax.make_train/train on MemoryChain (memory_length 4: episodes of 5 steps end
    inside the 15-step window with +-1 rewards) with eps = 1 against an oracle replay: losses, final parameters and
    the final key."""
    from purejaxql_b200 import pqn_rnn_gymnax
    cfg = _mc_cfg()
    nupd = 2
    cfg["TOTAL_TIMESTEPS"] = cfg["TOTAL_TIMESTEPS_DECAY"] = float(nupd * cfg["NUM_STEPS"] * cfg["NUM_ENVS"])
    train = pqn_rnn_gymnax.make_train(cfg)
    eng = train.engine
    assert eng.env_params.memory_length == 4 and cfg["TEST_NUM_STEPS"] == 1000
    S = 2
    rngs = jr.split(jr.PRNGKey(41), S)
    cap = {}
    orig = eng.spec.init
    eng.spec.init = lambda k, d: cap.setdefault("flat", orig(k, d)).clone()
    out = train(rngs)
    ts = out["runner_state"][0]
    tree0 = eng.spec.unflatten(cap["flat"])
    T, E, W, nmb = cfg["NUM_STEPS"], cfg["NUM_ENVS"], cfg["MEMORY_WINDOW"], cfg["NUM_MINIBATCHES"]
    Bm = E // nmb
    H = 128
    nonzero = 0
    for s in range(S):
        def leaf(tree, path):
            d = tree
            for k in path:
                d = d[k]
            return d[s].cpu().numpy()
        params = {"/".join(p): leaf(tree0, p).astype(np.float32) for p, *_ in eng.spec.entries}
        env = MC.make(flatten=True, memory_length=4)
        k = jr.split(rngs[s], 2); rng = k[0]                               # :255
        k = jr.split(rng, 2); rng = k[0]                                   # :505
        k = jr.split(rng, 2); rng, kR = k[0], k[1]                         # :508
        obs, st = env.reset(jr.split(kR, E))
        hs = np.zeros((E, H), np.float32); ld = np.zeros(E, bool); la = np.zeros(E, np.int32)
        k = jr.split(rng, 2); carry = k[1]                                 # :531
        mem = []
        for _ in range(W + T):
            (hs, obs, ld, la, st, carry), tr, _ = _oracle_step(env, params, hs, obs, ld, la, st, carry, 1.0, 1.0, E)
            mem.append(tr)
        rng = carry
        k = jr.split(rng, 2); rng = k[1]                                   # :541
        opt = R.opt_init(params)
        for u in range(nupd):
            k = jr.split(rng, 2); carry = k[1]                             # :222
            new = []
            for _ in range(T):
                (hs, obs, ld, la, st, carry), tr, info = _oracle_step(env, params, hs, obs, ld, la, st, carry, 1.0, 1.0, E)
                new.append(tr)
            rng = carry
            mem = mem[T:] + new
            stack = {kk: np.stack([m[kk] for m in mem]) for kk in mem[0]}
            nonzero += int((stack["reward"] != 0).sum())
            k = jr.split(rng, 2); r = k[0]                                 # :381
            losses = []
            for _ in range(cfg["NUM_EPOCHS"]):
                k = jr.split(r, 2); r, kperm = k[0], k[1]                  # :368
                perm = jr.permutation_indices(kperm, E)
                r = jr.split(r, 2)[0]                                      # :375
                for mb in range(nmb):
                    idx = perm[mb * Bm:(mb + 1) * Bm]
                    loss, chosen, g = RR.rnn_loss_and_grads(
                        params, stack["last_hs"][0][idx], stack["obs"][:, idx], stack["last_done"][:, idx],
                        stack["last_action"][:, idx], stack["action"][:, idx], stack["reward"][:, idx],
                        stack["done"][:, idx], cfg["GAMMA"], cfg["LAMBDA"])
                    params, opt, _ = R.radam_clip_step(params, g, opt, np.float32(cfg["LR"]), cfg["MAX_GRAD_NORM"])
                    losses.append(loss)
            rng = r
            got = float(out["metrics"]["td_loss"][s, u])
            assert abs(got - np.mean(losses)) < 2e-3 * max(1.0, abs(np.mean(losses))), (u, got, np.mean(losses))
        for p, *_ in eng.spec.entries:
            d = np.abs(leaf(ts.params, p) - params["/".join(p)])
            assert np.quantile(d, 0.99) < 1e-4 and d.max() < 1e-3, (p, d.max())
        assert np.array_equal(out["runner_state"][4][s].cpu().numpy().view(np.uint32), rng)
    assert nonzero > 0


def test_rnn_cuda_graph_replay_equals_eager_on_memory_chain():
    from purejaxql_b200 import pqn_rnn_gymnax
    outs = []
    for graph in (False, True):
        cfg = _mc_cfg(EPS_FINISH=0.1, EPS_DECAY=0.5, TEST_DURING_TRAINING=True, TEST_INTERVAL=0.4, TEST_NUM_ENVS=8,
                      TEST_NUM_STEPS=40, EPS_TEST=0.0, CUDA_GRAPH=graph)
        cfg["TOTAL_TIMESTEPS"] = cfg["TOTAL_TIMESTEPS_DECAY"] = float(5 * cfg["NUM_STEPS"] * cfg["NUM_ENVS"])
        train = pqn_rnn_gymnax.make_train(cfg)
        out = train(jr.split(jr.PRNGKey(5), 2))
        assert train.engine.graph_captured == graph
        outs.append((out["runner_state"][0].params_flat.cpu().numpy(), out["metrics"]["td_loss"].cpu().numpy(),
                     out["metrics"]["test/returned_episode_returns"].cpu().numpy(),
                     out["runner_state"][4].cpu().numpy(), out["runner_state"][2][4].cpu().numpy()))
    for a, b in zip(*outs):
        assert np.array_equal(a, b, equal_nan=True)


def test_memory_chain_preset_shortened_with_eval():
    from purejaxql_b200 import config_loader, envs, pqn_rnn_gymnax
    c = config_loader.compose(["+alg=pqn_rnn_memory_chain", "NUM_SEEDS=2", "SAVE_PATH=null",
                               "alg.TOTAL_TIMESTEPS=16384", "alg.TOTAL_TIMESTEPS_DECAY=16384", "alg.TEST_NUM_ENVS=16",
                               "alg.TEST_INTERVAL=0.5"])
    cfg = {**c, **c["alg"]}
    ml = cfg["ENV_KWARGS"]["memory_length"]
    train = pqn_rnn_gymnax.make_train(cfg)
    assert cfg["TEST_NUM_STEPS"] == 1000 and cfg["NUM_UPDATES"] == 4
    out = train(jr.split(jr.PRNGKey(0), 2))
    m = out["metrics"]
    for k in ("td_loss", "qvals", "returned_episode_returns", "returned_episode_lengths"):
        assert torch.isfinite(m[k]).all(), k
    assert "test/returned_episode_returns" in m and "env_frame" not in m
    # greedy evaluation over 1000 steps: every finished episode is memory_length + 1 steps long with return +-1
    assert (m["test/returned_episode_lengths"] == ml + 1).all()
    assert (m["test/returned_episode_returns"].abs() <= 1).all()
    mem = out["runner_state"][1]
    rw, dn = mem.reward.cpu().numpy(), mem.done.cpu().numpy().astype(bool)
    assert set(np.unique(rw[dn])) <= {-1.0, 1.0} and (rw[~dn] == 0).all() and dn.any()
    f = envs.state_to_fields(NAME, out["runner_state"][2][4].cpu())
    done_once = f["log_returned_episode_lengths"] > 0
    assert done_once.any() and (f["log_returned_episode_lengths"][done_once] == ml + 1).all()
    assert set(f["log_returned_episode_returns"][done_once].abs().unique().tolist()) == {1.0}
    assert (f["param_memory_length"] == ml).all()


def test_pqn_gymnax_smoke_on_memory_chain_default_params():
    """The feed-forward script runs MemoryChain with gymnax's default parameters (memory_length 5) on the MLP, whose
    thin first layer takes the 3-float observation."""
    from purejaxql_b200 import config_loader, envs, pqn_gymnax
    c = config_loader.compose(["+alg=pqn_cartpole", "alg.ENV_NAME=MemoryChain-bsuite", "NUM_SEEDS=2", "SAVE_PATH=null",
                               "alg.TOTAL_TIMESTEPS=16384", "alg.TOTAL_TIMESTEPS_DECAY=16384", "alg.TEST_NUM_ENVS=16",
                               "alg.TEST_INTERVAL=0.5", "alg.TEST_NUM_STEPS=64"])
    cfg = {**c, **c["alg"]}
    train = pqn_gymnax.make_train(cfg)
    assert train.engine.env.obs_dim == 3 and train.engine.env_params.memory_length == 5
    out = train(jr.split(jr.PRNGKey(1), 2))
    m = out["metrics"]
    assert torch.isfinite(m["td_loss"]).all() and torch.isfinite(m["qvals"]).all()
    assert (m["test/returned_episode_lengths"] == 6).all()
    assert (m["returned_episode_lengths"] <= 6).all()
    f = envs.state_to_fields(NAME, out["runner_state"][1][1].cpu())
    assert (f["param_memory_length"] == 5).all()
    assert set(f["log_returned_episode_lengths"].unique().tolist()) == {6}
