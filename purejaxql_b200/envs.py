"""Host-side mirror of the gymnax environment protocol over libpqn_b200's
batched environment operator.

Mirrors what the reference uses of gymnax (purejaxql/pqn_minatar.py:103-112):

    env, env_params = make("Breakout-MinAtar")       # gymnax.make + LogWrapper
    obs, state = env.reset(keys, env_params)          # keys: uint32[N,2] (already split)
    obs, state, reward, done, info = env.step(keys, state, action, env_params)
    env.action_space(env_params).n, env.observation_space(env_params).shape,
    env_params.max_steps_in_episode

The functional protocol is kept (state in, state out) but batched natively —
there is no ``jax.vmap`` to wrap it with — and ``state`` is the library's
word-major SoA block (``uint32[state_words, N]`` CUDA tensor).
``state_to_fields`` / ``fields_to_state`` convert to and from gymnax's field
names for interop and parity tests (pure tensor ops, usable on CPU tensors).
"""
from __future__ import annotations

import numbers
from dataclasses import dataclass, replace
from types import SimpleNamespace

import torch

from . import _lib

ENV_IDS = {
    "Breakout-MinAtar": 0,
    "Asterix-MinAtar": 1,
    "SpaceInvaders-MinAtar": 2,
    "Freeway-MinAtar": 3,
    "CartPole-v1": 16,
    "Acrobot-v1": 17,
    "MemoryChain-bsuite": 32,
}
# PQN_ENV_SEAQUEST (4) is reserved in include/pqn_b200.h but not built: gymnax 0.0.6 (the reference's pin) does not
# register "Seaquest-MinAtar" in gymnax.make either (DESIGN.md section 8), so the reference cannot run it.
MINATAR_GAMES = ("Breakout-MinAtar", "Asterix-MinAtar", "SpaceInvaders-MinAtar", "Freeway-MinAtar")

LOG_FIELDS = ("episode_returns", "episode_lengths", "returned_episode_returns",
              "returned_episode_lengths", "timestep")


# gymnax memory_chain.EnvParams().memory_length; the library's pqn_env_reset uses the same default
MEMORY_CHAIN_DEFAULT_MEMORY_LENGTH = 5


@dataclass
class EnvParams:
    max_steps_in_episode: int
    memory_length: int | None = None      # MemoryChain-bsuite only


def _check_memory_length(v):
    """memory_length as an int >= 1 (a config may hand over 100 or 100.0).  Episodes are memory_length + 1 steps:
    the context is shown at step 0 and the answer is scored at step memory_length, so 0 has no episode to play."""
    if isinstance(v, bool) or not isinstance(v, numbers.Real) or not float(v).is_integer() or not 1 <= v < 2 ** 31:
        raise ValueError(f"MemoryChain-bsuite: memory_length must be an integer in [1, 2^31), got {v!r}")
    return int(v)


def _u2f(t):
    return t.contiguous().view(torch.float32)


def _f2u(t):
    return t.to(torch.float32).contiguous().view(torch.int32)


# --------------------------------------------------------------------------- #
# state <-> gymnax field conversion (int32 views of the uint32 words)
# --------------------------------------------------------------------------- #
def state_to_fields(env_name: str, state: torch.Tensor) -> dict:
    """uint32/int32[state_words, N] -> dict of gymnax EnvState + LogEnvState fields."""
    st = state.view(torch.int32) if state.dtype != torch.int32 else state
    f = {}
    if env_name == "Breakout-MinAtar":
        w = st[0]
        f["ball_y"] = w & 15
        f["ball_x"] = (w >> 4) & 15
        f["ball_dir"] = (w >> 8) & 3
        f["pos"] = (w >> 10) & 15
        f["last_y"] = (w >> 14) & 15
        f["last_x"] = (w >> 18) & 15
        f["strike"] = ((w >> 22) & 1).bool()
        f["terminal"] = ((w >> 23) & 1).bool()
        f["time"] = st[1]
        n = st.shape[1]
        p = torch.arange(100, device=st.device)
        words = st[2:6].to(torch.int64) & 0xFFFFFFFF                       # [4, N]
        bits = (words[p >> 5] >> (p & 31).unsqueeze(1)) & 1                # [100, N]
        f["brick_map"] = bits.t().reshape(n, 10, 10).to(torch.float32)
        core = 6
    elif env_name == "Freeway-MinAtar":
        w = st[0]
        f["pos"] = w & 15
        f["move_timer"] = (w >> 4) & 3
        f["terminal"] = ((w >> 6) & 1).bool()
        f["time"] = st[1]
        cars = []
        for c in range(8):
            v = (st[2 + c // 2] >> (16 * (c % 2))) & 0xFFFF
            cars.append(torch.stack([v & 15, torch.full_like(v, c + 1), (v >> 4) & 7, ((v >> 7) & 15) - 5], -1))
        f["cars"] = torch.stack(cars, 1)                                    # [N, 8, 4] = (x, y, timer, speed)
        core = 6
    elif env_name == "Asterix-MinAtar":
        w, w1 = st[0], st[1]
        f["player_x"] = w & 15
        f["player_y"] = (w >> 4) & 15
        f["spawn_speed"] = (w >> 8) & 15
        f["spawn_timer"] = (w >> 12) & 15
        f["move_speed"] = (w >> 16) & 7
        f["move_timer"] = (w >> 19) & 7
        f["shot_timer"] = (w >> 22) & 7
        f["terminal"] = ((w >> 25) & 1).bool()
        f["ramp_timer"] = (w1 & 255) - 1
        f["ramp_index"] = (w1 >> 8) & 255
        f["time"] = st[2]
        ents = []
        for e in range(8):
            v = (st[3 + e // 4] >> (8 * (e % 4))) & 255
            fill = (v >> 6) & 1
            ents.append(torch.stack([v & 15, fill * (e + 1), (v >> 4) & 1, (v >> 5) & 1, fill], -1))
        f["entities"] = torch.stack(ents, 1)                                # [N, 8, 5] = (x, y, lr, is_gold, filled)
        core = 5
    elif env_name == "SpaceInvaders-MinAtar":
        w = st[0]
        f["pos"] = w & 15
        f["alien_dir"] = ((w >> 4) & 1) * 2 - 1
        f["enemy_move_interval"] = (w >> 5) & 15
        f["alien_move_timer"] = (w >> 9) & 15
        f["alien_shot_timer"] = (w >> 13) & 15
        f["shot_timer"] = (w >> 17) & 7
        f["terminal"] = ((w >> 20) & 1).bool()
        f["ramp_index"] = (w >> 21) & 15
        f["time"] = st[1]
        n = st.shape[1]
        p = torch.arange(100, device=st.device)
        for name, base in (("alien_map", 2), ("f_bullet_map", 6), ("e_bullet_map", 10)):
            words = st[base:base + 4].to(torch.int64) & 0xFFFFFFFF
            bits = (words[p >> 5] >> (p & 31).unsqueeze(1)) & 1
            f[name] = bits.t().reshape(n, 10, 10).to(torch.int32)
        core = 14
    elif env_name == "CartPole-v1":
        for j, k in enumerate(("x", "x_dot", "theta", "theta_dot")):
            f[k] = _u2f(st[j])
        f["time"] = st[4]
        core = 5
    elif env_name == "Acrobot-v1":
        for j, k in enumerate(("joint_angle1", "joint_angle2", "velocity_1", "velocity_2")):
            f[k] = _u2f(st[j])
        f["time"] = st[4]
        core = 5
    elif env_name == "MemoryChain-bsuite":
        f["context"] = st[0].unsqueeze(1)                                    # [N, num_bits = 1]
        f["query"] = st[1]
        f["total_perfect"] = st[2]
        f["total_regret"] = st[3]
        f["time"] = st[4]
        f["param_memory_length"] = st[5]    # not a gymnax field: the env parameter, kept in the state words
        core = 6
    else:
        raise KeyError(env_name)
    f["log_episode_returns"] = _u2f(st[core + 0])
    f["log_episode_lengths"] = st[core + 1]
    f["log_returned_episode_returns"] = _u2f(st[core + 2])
    f["log_returned_episode_lengths"] = st[core + 3]
    f["log_timestep"] = st[core + 4]
    return f


def fields_to_state(env_name: str, f: dict, params: EnvParams | None = None) -> torch.Tensor:
    """Inverse of :func:`state_to_fields` -> int32[state_words, N].  MemoryChain's memory_length word comes from
    ``params`` (gymnax's default when None or unset), not from the gymnax fields."""
    i32 = lambda t: torch.as_tensor(t).to(torch.int32)
    if env_name == "Breakout-MinAtar":
        w = (i32(f["ball_y"]) | (i32(f["ball_x"]) << 4) | (i32(f["ball_dir"]) << 8) | (i32(f["pos"]) << 10)
             | (i32(f["last_y"]) << 14) | (i32(f["last_x"]) << 18) | (i32(f["strike"]) << 22)
             | (i32(f["terminal"]) << 23))
        n = w.shape[0]
        bm = (torch.as_tensor(f["brick_map"]).reshape(n, 100) != 0).to(torch.int64)
        words = []
        for k in range(4):
            lo, hi = 32 * k, min(100, 32 * k + 32)
            sh = torch.arange(hi - lo, device=bm.device)
            v = (bm[:, lo:hi] << sh).sum(1)
            v = torch.where(v >= 2 ** 31, v - 2 ** 32, v).to(torch.int32)
            words.append(v)
        core = [w, i32(f["time"])] + words
    elif env_name == "Freeway-MinAtar":
        cars = i32(f["cars"])
        words = []
        for k in range(4):
            v = torch.zeros_like(cars[:, 0, 0])
            for h in range(2):
                c = 2 * k + h
                v = v | ((cars[:, c, 0] | (cars[:, c, 2] << 4) | ((cars[:, c, 3] + 5) << 7)) << (16 * h))
            words.append(v)
        core = [i32(f["pos"]) | (i32(f["move_timer"]) << 4) | (i32(f["terminal"]) << 6), i32(f["time"])] + words
    elif env_name == "Asterix-MinAtar":
        ent = i32(f["entities"])
        w = (i32(f["player_x"]) | (i32(f["player_y"]) << 4) | (i32(f["spawn_speed"]) << 8) | (i32(f["spawn_timer"]) << 12)
             | (i32(f["move_speed"]) << 16) | (i32(f["move_timer"]) << 19) | (i32(f["shot_timer"]) << 22)
             | (i32(f["terminal"]) << 25))
        w1 = (i32(f["ramp_timer"]) + 1) | (i32(f["ramp_index"]) << 8)
        words = []
        for k in range(2):
            v = torch.zeros_like(w)
            for h in range(4):
                e = 4 * k + h
                b = (ent[:, e, 0] | (ent[:, e, 2] << 4) | (ent[:, e, 3] << 5) | (1 << 6)) * ent[:, e, 4]
                v = v | (b << (8 * h))
            words.append(v)
        core = [w, w1, i32(f["time"])] + words
    elif env_name == "SpaceInvaders-MinAtar":
        w = (i32(f["pos"]) | ((i32(f["alien_dir"]) > 0).to(torch.int32) << 4) | (i32(f["enemy_move_interval"]) << 5)
             | (i32(f["alien_move_timer"]) << 9) | (i32(f["alien_shot_timer"]) << 13) | (i32(f["shot_timer"]) << 17)
             | (i32(f["terminal"]) << 20) | (i32(f["ramp_index"]) << 21))
        n = w.shape[0]
        core = [w, i32(f["time"])]
        for name in ("alien_map", "f_bullet_map", "e_bullet_map"):
            bm = (torch.as_tensor(f[name]).reshape(n, 100) != 0).to(torch.int64)
            for k in range(4):
                lo, hi = 32 * k, min(100, 32 * k + 32)
                sh = torch.arange(hi - lo, device=bm.device)
                v = (bm[:, lo:hi] << sh).sum(1)
                core.append(torch.where(v >= 2 ** 31, v - 2 ** 32, v).to(torch.int32))
    elif env_name == "CartPole-v1":
        core = [_f2u(torch.as_tensor(f[k])) for k in ("x", "x_dot", "theta", "theta_dot")] + [i32(f["time"])]
    elif env_name == "Acrobot-v1":
        core = [_f2u(torch.as_tensor(f[k])) for k in
                ("joint_angle1", "joint_angle2", "velocity_1", "velocity_2")] + [i32(f["time"])]
    elif env_name == "MemoryChain-bsuite":
        ml = params.memory_length if params is not None and params.memory_length is not None \
            else MEMORY_CHAIN_DEFAULT_MEMORY_LENGTH
        t = i32(f["time"])
        core = [i32(f["context"]).reshape(t.shape[0], -1)[:, 0], i32(f["query"]), i32(f["total_perfect"]),
                i32(f["total_regret"]), t, torch.full_like(t, _check_memory_length(ml))]
    else:
        raise KeyError(env_name)
    log = [_f2u(torch.as_tensor(f["log_episode_returns"])), i32(f["log_episode_lengths"]),
           _f2u(torch.as_tensor(f["log_returned_episode_returns"])), i32(f["log_returned_episode_lengths"]),
           i32(f["log_timestep"])]
    return torch.stack(core + log).contiguous()


def pack_observation(obs: torch.Tensor) -> torch.Tensor:
    """{0,1} observations [N, ...] (e.g. the float32 (10,10,C) rows gymnax returns) ->
    int32[N, packed_obs_words] rows in the bit layout the CNN kernels read
    (bit f of a row = element f of the flattened observation; rows padded to 16 bytes)."""
    n = obs.shape[0]
    flat = (obs.reshape(n, -1) != 0).to(torch.int64)
    nb = flat.shape[1]
    pw = ((nb + 31) // 32 + 3) // 4 * 4
    padded = torch.zeros((n, pw * 32), dtype=torch.int64, device=obs.device)
    padded[:, :nb] = flat
    sh = torch.arange(32, device=obs.device, dtype=torch.int64)
    words = (padded.view(n, pw, 32) << sh).sum(-1)
    words = torch.where(words >= 2 ** 31, words - 2 ** 32, words)
    return words.to(torch.int32).contiguous()


# --------------------------------------------------------------------------- #
# the batched environment
# --------------------------------------------------------------------------- #
class BatchedEnv:
    """``LogWrapper(gymnax.make(name)[0])`` (optionally with
    ``FlattenObservationWrapper``), batched over the leading axis."""

    def __init__(self, name: str, flatten_obs: bool = False, rng_mode: int = 0):
        if name not in ENV_IDS:
            raise KeyError(f"unknown env {name!r}; known: {sorted(ENV_IDS)}")
        self.name = name
        self.env_id = ENV_IDS[name]
        info = _lib.EnvInfo()
        _lib.check(_lib.lib().pqn_env_info(self.env_id, info), "pqn_env_info")
        self.info = info
        self.state_words = info.state_words
        self.obs_dim = info.obs_dim
        self.binary_obs = bool(info.binary_obs)
        self.packed_obs_words = info.packed_obs_words
        self.num_actions = info.num_actions
        shape = tuple(info.obs_shape) if self.binary_obs else (info.obs_dim,)
        self._obs_shape = (info.obs_dim,) if flatten_obs else shape
        self.default_params = EnvParams(
            max_steps_in_episode=info.max_steps,
            memory_length=MEMORY_CHAIN_DEFAULT_MEMORY_LENGTH if name == "MemoryChain-bsuite" else None)
        self.rng_mode = rng_mode

    # gymnax spaces -------------------------------------------------------
    def action_space(self, params=None):
        return SimpleNamespace(n=self.num_actions)

    def observation_space(self, params=None):
        return SimpleNamespace(shape=self._obs_shape)

    # protocol ------------------------------------------------------------
    def reset(self, keys: torch.Tensor, params: EnvParams | None = None):
        params = params or self.default_params
        n = keys.shape[0]
        state = torch.empty((self.state_words, n), dtype=torch.int32, device=keys.device)
        obs = torch.empty((n,) + self._obs_shape, dtype=torch.float32, device=keys.device)
        _lib.check(_lib.lib().pqn_env_reset_params(self.env_id, _lib.p(keys), _lib.p(state), _lib.p(obs), n,
                                                   c_params(params), self.rng_mode, _lib.stream_ptr()),
                   "pqn_env_reset_params")
        return obs, state

    def step(self, keys: torch.Tensor, state: torch.Tensor, action: torch.Tensor,
             params: EnvParams | None = None, inplace: bool = False):
        params = params or self.default_params
        n = keys.shape[0]
        dev = keys.device
        state = state if inplace else state.clone()
        obs = torch.empty((n,) + self._obs_shape, dtype=torch.float32, device=dev)
        reward = torch.empty(n, dtype=torch.float32, device=dev)
        done = torch.empty(n, dtype=torch.uint8, device=dev)
        disc = torch.empty(n, dtype=torch.float32, device=dev)
        ret = torch.empty(n, dtype=torch.float32, device=dev)
        ln = torch.empty(n, dtype=torch.int32, device=dev)
        ts = torch.empty(n, dtype=torch.int32, device=dev)
        _lib.check(_lib.lib().pqn_env_step(
            self.env_id, _lib.p(keys), _lib.p(state), _lib.p(action.to(torch.int32).contiguous()), _lib.p(obs),
            _lib.p(reward), _lib.p(done), _lib.p(disc), _lib.p(ret), _lib.p(ln), _lib.p(ts), n,
            params.max_steps_in_episode, self.rng_mode, _lib.stream_ptr()), "pqn_env_step")
        done_b = done.bool()
        info = {"discount": disc, "returned_episode_returns": ret, "returned_episode_lengths": ln,
                "timestep": ts, "returned_episode": done_b}
        return obs, state, reward, done_b, info


def c_params(params: EnvParams) -> _lib.EnvParams:
    """EnvParams -> the library's pqn_env_params_t.  memory_length None is passed as 0: envs without the parameter
    ignore it, MemoryChain rejects it (its params always carry one, see BatchedEnv.default_params)."""
    ml = params.memory_length
    return _lib.EnvParams(int(params.max_steps_in_episode), 0 if ml is None else int(ml))


def make(env_name: str, flatten_obs: bool = False, rng_mode: int = 0, env_kwargs: dict | None = None):
    """``gymnax.make(env_name)`` -> (env, env_params); the LogWrapper is built in.
    ``env_kwargs``: EnvParams fields to override, as ``EnvParams(**env_kwargs)`` would (only MemoryChain-bsuite's
    ``memory_length`` exists beyond the defaults).  They are validated here, before any device work."""
    kw = dict(env_kwargs or {})
    if env_name not in ENV_IDS:
        raise KeyError(f"unknown env {env_name!r}; known: {sorted(ENV_IDS)}")
    allowed = {"memory_length"} if env_name == "MemoryChain-bsuite" else set()
    unknown = set(kw) - allowed
    if unknown:
        raise TypeError(f"{env_name}: unknown env parameter(s) {sorted(unknown)}")
    if "memory_length" in kw:
        kw["memory_length"] = _check_memory_length(kw["memory_length"])
    env = BatchedEnv(env_name, flatten_obs=flatten_obs, rng_mode=rng_mode)
    return env, replace(env.default_params, **kw)
