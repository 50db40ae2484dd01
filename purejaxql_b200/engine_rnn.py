"""The recurrent (GRU) PQN training program: host-side restatement of ``make_train`` in
purejaxql/pqn_rnn_gymnax.py:117-560 with the seed axis taken natively.

All compute is libpqn_b200 kernels: ``pqn_rnn_step`` (one step of the recurrent Q-network for the rollout, the memory
warm-up and the evaluation), ``pqn_rollout_act_step`` (eps-greedy + env step + LogWrapper, shared with the feed-forward
engine), ``pqn_rnn_loss_grad`` (window forward, in-loss Q(lambda) targets, BPTT) and ``pqn_radam_clip_step``.  This
module owns the buffers, walks the reference's PRNG key chain — including its re-bindings of ``rng`` to the final
carry of the rollout scans (:222-228, :531-537) — and keeps the memory of the last MEMORY_WINDOW + NUM_STEPS
transitions.  Minibatches are whole env trajectories: ``jax.random.permutation(rng, x, axis=1)`` (:368-379).
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np
import torch

from . import _lib, envs, jaxrandom as jr
from .engine import INFO_KEYS, TrainState, linear_schedule, radam_schedule_table, _f32
from .networks import NET_RNN, QNetworkSpec


class PQNRnnEngine:
    def __init__(self, config: dict, device=None, env_params: envs.EnvParams | None = None):
        self.cfg = c = config
        self.device = torch.device(device or "cuda")
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise _lib.PqnError("purejaxql_b200 needs a CUDA device: there is no CPU fallback")
        _lib.lib()
        if c.get("NORM_TYPE", "layer_norm") != "layer_norm" or c.get("NORM_INPUT", False):
            raise NotImplementedError("the GRU network is built for NORM_TYPE=layer_norm, NORM_INPUT=False "
                                      "(the shipped pqn_rnn_cartpole.yaml)")
        self.rng_mode = int(c.get("JAX_THREEFRY_PARTITIONABLE", 0))
        self.env, self.env_params = envs.make(c["ENV_NAME"], flatten_obs=True, rng_mode=self.rng_mode)
        if env_params is not None:                                    # e.g. MemoryChain's memory_length (:134-136)
            self.env_params = env_params
        if self.env.binary_obs:
            raise NotImplementedError("the recurrent script is built for the classic-control envs")
        self.max_steps = int(self.env_params.max_steps_in_episode)
        self.T, self.E, self.NU = int(c["NUM_STEPS"]), int(c["NUM_ENVS"]), int(c["NUM_UPDATES"])
        self.W = int(c["MEMORY_WINDOW"])
        self.A, self.D = self.env.num_actions, self.env.obs_dim
        self.H = int(c.get("HIDDEN_SIZE", 128))
        self.spec = QNetworkSpec(NET_RNN, self.D, self.A, self.H, int(c.get("NUM_LAYERS", 2)))
        self.nmb, self.epochs = int(c["NUM_MINIBATCHES"]), int(c["NUM_EPOCHS"])
        assert self.E % self.nmb == 0, "NUM_MINIBATCHES must divide NUM_ENVS (minibatches are whole env trajectories)"
        self.Bm = self.E // self.nmb
        self.gamma, self.lam = float(c["GAMMA"]), float(c["LAMBDA"])
        self.rew_scale = float(c.get("REW_SCALE", 1))
        self.test = bool(c.get("TEST_DURING_TRAINING", False))
        self._ws = None

    # ------------------------------------------------------------------ #
    def _workspace(self, S, rows):
        need = int(_lib.lib().pqn_net_workspace_bytes(self.spec.desc, S, rows))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws

    def step(self, params, hs, obs, last_done, last_action, q, S, N):
        """network.apply(params, hs, obs[None], done[None], last_action[None], train=False) for S x N envs; hs in place."""
        _lib.check(_lib.lib().pqn_rnn_step(self.spec.desc, _lib.p(params), _lib.p(hs), _lib.p(obs), N, _lib.p(last_done),
                                           _lib.p(last_action), _lib.p(q), S, N, _lib.p(self._workspace(S, N)),
                                           _lib.stream_ptr()), "pqn_rnn_step")

    def _act_step(self, S, N, step_keys, q, eps, state, obs_next, action, reward, done, maxq, sums, done_only, rew_scale):
        L = _lib.lib()
        _lib.check(L.pqn_rollout_act_step(self.env.env_id, _lib.p(step_keys), _lib.p(q), _lib.p(eps), _lib.p(state),
                                          _lib.p(obs_next), N, _lib.p(action), _lib.p(reward), _lib.p(done), _lib.p(maxq), N,
                                          _lib.p(sums), done_only, S, N, 0, 0, self.max_steps, rew_scale, self.rng_mode,
                                          _lib.stream_ptr()), "pqn_rollout_act_step")

    def _reset(self, key, S, N):
        """vmap_reset(N)(key, env_params): obs [S,N,D], state."""
        dev, mode, L = self.device, self.rng_mode, _lib.lib()
        state = torch.empty((self.env.state_words, S * N), dtype=torch.int32, device=dev)
        obs = torch.empty((S, N, self.D), dtype=torch.float32, device=dev)
        _lib.check(L.pqn_env_reset_params(self.env.env_id, _lib.p(jr.split(key, N, mode).reshape(S * N, 2).contiguous()),
                                          _lib.p(state), _lib.p(obs), S * N, envs.c_params(self.env_params), mode,
                                          _lib.stream_ptr()), "pqn_env_reset_params")
        return obs, state

    # ------------------------------------------------------------------ #
    def train(self, rngs):
        c, dev, L, mode = self.cfg, self.device, _lib.lib(), self.rng_mode
        T, E, A, NU, W, H, D, Bm = self.T, self.E, self.A, self.NU, self.W, self.H, self.D, self.Bm
        Tm = W + T
        keys = jr.as_key_tensor(rngs, dev)
        S = keys.shape[0]
        spec, P = self.spec, self.spec.total
        nud = c["NUM_UPDATES_DECAY"]
        eps_table = torch.tensor([linear_schedule(c["EPS_START"], c["EPS_FINISH"], c["EPS_DECAY"] * nud, n)
                                  for n in range(max(NU, 1))], dtype=torch.float32, device=dev)
        total_grad_steps = NU * self.nmb * self.epochs
        if c.get("LR_LINEAR_DECAY", False):
            lr_fn = lambda i: linear_schedule(c["LR"], 1e-20, nud * self.nmb * self.epochs, i)
        else:
            lr_fn = lambda i: _f32(c["LR"])
        sched = torch.from_numpy(radam_schedule_table(total_grad_steps, lr_fn)).to(dev)

        # ---- key chain (:255-256, :505-543)
        k = jr.split(keys, 2, mode)
        rng = k[:, 0].contiguous()                                   # :255  rng, _rng = split(rng)
        params = spec.init(rng, dev)                                 # :256  create_agent(rng)  (the CARRIED key)
        mu, nu, grads = torch.zeros_like(params), torch.zeros_like(params), torch.zeros_like(params)
        step_counter = torch.zeros(1, dtype=torch.int32, device=dev)
        gnorm = torch.zeros(S * 64, device=dev)
        k = jr.split(rng, 2, mode)
        rng, kT = k[:, 0].contiguous(), k[:, 1].contiguous()         # :505
        test_metrics = self.get_test_metrics(params, kT) if self.test else None
        k = jr.split(rng, 2, mode)
        rng, kR = k[:, 0].contiguous(), k[:, 1].contiguous()         # :508
        last_obs, state = self._reset(kR, S, E)                      # :509
        last_done = torch.zeros((S, E), dtype=torch.uint8, device=dev)
        last_action = torch.zeros((S, E), dtype=torch.int32, device=dev)
        hs = torch.zeros((S, E, H), dtype=torch.float32, device=dev)

        mem = SimpleNamespace(
            hs=torch.zeros((S, Tm, E, H), device=dev), obs=torch.zeros((S, Tm, E, D), device=dev),
            action=torch.zeros((S, Tm, E), dtype=torch.int32, device=dev), reward=torch.zeros((S, Tm, E), device=dev),
            done=torch.zeros((S, Tm, E), dtype=torch.uint8, device=dev),
            last_done=torch.zeros((S, Tm, E), dtype=torch.uint8, device=dev),
            last_action=torch.zeros((S, Tm, E), dtype=torch.int32, device=dev))
        q = torch.zeros((S * E, A), device=dev)
        maxq = torch.zeros((S, E), device=dev)
        info_sums = torch.zeros((S, 5), dtype=torch.float64, device=dev)
        new_obs = torch.empty_like(last_obs)
        eps_one = torch.ones(1, device=dev)
        eps_dev = torch.zeros(1, device=dev)

        act_t = torch.empty((S, E), dtype=torch.int32, device=dev)
        rew_t = torch.empty((S, E), device=dev)
        done_t = torch.empty((S, E), dtype=torch.uint8, device=dev)

        def rollout(carry_key, n_steps, slot0, eps):
            """n_steps x _step_env / _random_step starting from the expl_state above; transitions go to memory slots
            slot0..; returns the scan's final carry key (the reference re-binds `rng` to it).  Only static buffers are
            touched, so the update's rollout can be replayed from a CUDA graph."""
            step_keys = torch.zeros((n_steps, S, 2, 2), dtype=torch.int32, device=dev)
            carry = carry_key.clone()
            _lib.check(L.pqn_rollout_keys(_lib.p(carry), _lib.p(step_keys), S, n_steps, mode, _lib.stream_ptr()),
                       "pqn_rollout_keys")
            for t in range(n_steps):
                s = slot0 + t
                mem.hs[:, s].copy_(hs); mem.obs[:, s].copy_(last_obs)
                mem.last_done[:, s].copy_(last_done); mem.last_action[:, s].copy_(last_action)
                self.step(params, hs, last_obs, last_done, last_action, q, S, E)
                self._act_step(S, E, step_keys[t], q, eps, state, new_obs, act_t, rew_t, done_t, maxq, info_sums, 0,
                               self.rew_scale)
                mem.action[:, s].copy_(act_t); mem.reward[:, s].copy_(rew_t); mem.done[:, s].copy_(done_t)
                last_obs.copy_(new_obs)
                last_done.copy_(done_t); last_action.copy_(act_t)
            return carry

        # ---- memory warm-up with random actions (:514-537); `rng` becomes the scan's final carry
        k = jr.split(rng, 2, mode)
        rng = rollout(k[:, 1].contiguous(), Tm, 0, eps_one)
        k = jr.split(rng, 2, mode)                                   # :541
        rng = k[:, 1].contiguous()                                   # runner rng = _rng

        metric_names = ["env_step", "update_steps", "grad_steps", "td_loss", "qvals", *INFO_KEYS]
        metrics = {m: torch.zeros((S, max(NU, 1)), dtype=torch.float64, device=dev) for m in metric_names}
        test_hist = {kk: torch.zeros((S, max(NU, 1)), dtype=torch.float64, device=dev) for kk in INFO_KEYS} if self.test else None
        test_every = int(NU * c["TEST_INTERVAL"]) if self.test else None
        loss_sum, qsa_sum = torch.zeros(S, device=dev), torch.zeros(S, device=dev)
        ws = self._workspace(S, max(Tm * Bm, E))
        perm_ws = jr.permutation_workspace(E, S, dev)
        timesteps = grad_steps = 0
        denom = float(self.epochs * self.nmb)
        on_update_end = getattr(self, "on_update_end", None)
        # static buffers of the update step (graph capturable, like engine.PQNEngine)
        rng_buf = rng.clone()
        kT_buf = torch.zeros((S, 2), dtype=torch.int32, device=dev)
        upd_idx = torch.zeros(1, dtype=torch.int64, device=dev)
        m_cur = torch.zeros((S, 7), dtype=torch.float64, device=dev)

        def update_body():
            # ================= SAMPLE PHASE (:190-236)
            eps_dev.copy_(eps_table.index_select(0, upd_idx))
            k = jr.split(rng_buf, 2, mode)                           # :222
            info_sums.zero_()
            for name in ("hs", "obs", "action", "reward", "done", "last_done", "last_action"):   # :239-243 shift the memory
                buf = getattr(mem, name)
                buf[:, :W].copy_(buf[:, T:T + W].clone())
            rng = rollout(k[:, 1].contiguous(), T, W, eps_dev)       # rng := final carry of the scan (:223-228)
            # ================= NETWORKS UPDATE (:246-386)
            loss_sum.zero_(); qsa_sum.zero_()
            k = jr.split(rng, 2, mode)                               # :381  (the scan carry starts at `rng`)
            r = k[:, 0].contiguous()
            for _ in range(self.epochs):
                k = jr.split(r, 2, mode)                             # :368
                r, kperm = k[:, 0].contiguous(), k[:, 1].contiguous()
                perm = jr.permutation_indices(kperm, E, mode, workspace=perm_ws).to(torch.int64)   # permutation of the ENV axis
                r = jr.split(r, 2, mode)[:, 0].contiguous()          # :375
                for mbi in range(self.nmb):
                    idx = perm[:, mbi * Bm:(mbi + 1) * Bm]                             # [S, Bm]
                    i3 = idx[:, None, :].expand(S, Tm, Bm)

                    def g3(x):
                        return x.gather(2, i3).contiguous()
                    obs_mb = mem.obs.gather(2, i3[..., None].expand(S, Tm, Bm, D)).contiguous()
                    hs0 = mem.hs[:, 0].gather(1, idx[:, :, None].expand(S, Bm, H)).contiguous()
                    ld, la, ac, rw, dn = g3(mem.last_done), g3(mem.last_action), g3(mem.action), g3(mem.reward), g3(mem.done)
                    _lib.check(L.pqn_rnn_loss_grad(spec.desc, _lib.p(params), _lib.p(hs0), _lib.p(obs_mb), _lib.p(ld),
                                                   _lib.p(la), _lib.p(ac), _lib.p(rw), _lib.p(dn), _lib.p(grads),
                                                   _lib.p(loss_sum), _lib.p(qsa_sum), S, Tm, Bm, self.gamma, self.lam,
                                                   _lib.p(ws), _lib.stream_ptr()), "pqn_rnn_loss_grad")
                    _lib.check(L.pqn_radam_clip_step(_lib.p(params), _lib.p(grads), _lib.p(mu), _lib.p(nu), _lib.p(sched),
                                                     _lib.p(step_counter), _lib.p(gnorm), S, P, float(c["MAX_GRAD_NORM"]),
                                                     0.9, 0.999, 1e-8, _lib.stream_ptr()), "pqn_radam_clip_step")
            if self.test:                                            # :398  rng, _rng = split(rng)
                k = jr.split(r, 2, mode)
                r = k[:, 0].contiguous()
                kT_buf.copy_(k[:, 1])
            rng_buf.copy_(r)
            m_cur[:, 0] = loss_sum.double() / denom
            m_cur[:, 1] = qsa_sum.double() / denom
            m_cur[:, 2:7] = info_sums / float(T * E)
            upd_idx.add_(1)

        # CUDA graph: these runs are launch-bound (32 envs x 64 steps: thousands of small launches per update), so the
        # update is captured after the first eager one and replayed unless CUDA_GRAPH is false
        want_graph = c.get("CUDA_GRAPH", "auto")
        use_graph = (True if want_graph == "auto" else bool(want_graph)) and NU > 2
        graph = None
        self.graph_captured = False
        for n_updates in range(NU):
            if graph is not None:
                graph.replay()
            else:
                update_body()
                if use_graph and n_updates == 0:
                    try:
                        torch.cuda.synchronize(dev)
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g):
                            update_body()
                        graph = g
                        self.graph_captured = True
                    except Exception as e:                            # capture is an optimisation only
                        import warnings
                        warnings.warn(f"CUDA graph capture of the recurrent update failed ({e!r}); running eagerly")
                        graph, use_graph = None, False
                        torch.cuda.synchronize(dev)
            timesteps += T * E
            grad_steps += self.nmb * self.epochs
            col = n_updates
            metrics["env_step"][:, col] = timesteps
            metrics["update_steps"][:, col] = n_updates + 1
            metrics["grad_steps"][:, col] = grad_steps
            metrics["td_loss"][:, col] = m_cur[:, 0]
            metrics["qvals"][:, col] = m_cur[:, 1]
            for j, kk in enumerate(INFO_KEYS):
                metrics[kk][:, col] = m_cur[:, 2 + j]
            if on_update_end is not None:
                on_update_end(n_updates, dict(mem=mem, params=params, rng=rng_buf))
            if self.test:                                            # :398-408
                if test_every > 0 and (n_updates + 1) % test_every == 0:
                    test_metrics = self.get_test_metrics(params, kT_buf.clone())
                for kk in INFO_KEYS:
                    test_hist[kk][:, col] = test_metrics[kk]
        rng = rng_buf
        torch.cuda.synchronize(dev)
        out_metrics = {m: v[:, :NU].float() if m in ("td_loss", "qvals", *INFO_KEYS) else v[:, :NU].to(torch.int64)
                       for m, v in metrics.items()}
        if self.test:
            out_metrics.update({f"test/{kk}": v[:, :NU].float() for kk, v in test_hist.items()})
        F = spec.in_c
        bs = spec.init_stats(S, dev)
        train_state = TrainState(
            params=spec.unflatten(params), params_flat=params, batch_stats=spec.unflatten_stats(bs), batch_stats_flat=bs,
            opt_state=SimpleNamespace(mu=mu, nu=nu, count=grad_steps),
            timesteps=torch.full((S,), timesteps, dtype=torch.int64), n_updates=torch.full((S,), NU),
            grad_steps=torch.full((S,), grad_steps))
        expl_state = (hs, last_obs, last_done, last_action, state)
        return {"runner_state": (train_state, mem, expl_state, test_metrics, rng), "metrics": out_metrics}

    # ------------------------------------------------------------------ #
    def get_test_metrics(self, params, rng):
        """Greedy evaluation (:411-503): reset with `_rng`, the scan carry starts at the same `_rng`, every step splits
        (rng, rng_a, rng_s) like the training rollout."""
        c, dev, L, mode = self.cfg, self.device, _lib.lib(), self.rng_mode
        S = rng.shape[0]
        N, steps = int(c["TEST_NUM_ENVS"]), int(c["TEST_NUM_STEPS"])
        kr = jr.split(rng, 2, mode)[:, 1].contiguous()               # :475
        obs, state = self._reset(kr, S, N)
        nxt = torch.empty_like(obs)
        hs = torch.zeros((S, N, self.H), device=dev)
        ld = torch.zeros((S, N), dtype=torch.uint8, device=dev)
        la = torch.zeros((S, N), dtype=torch.int32, device=dev)
        q = torch.zeros((S * N, self.A), device=dev)
        rw, mq = torch.zeros((S, N), device=dev), torch.zeros((S, N), device=dev)
        act = torch.zeros((S, N), dtype=torch.int32, device=dev)
        dn = torch.zeros((S, N), dtype=torch.uint8, device=dev)
        sums = torch.zeros((S, 5), dtype=torch.float64, device=dev)
        eps = torch.full((1,), float(c["EPS_TEST"]), device=dev)
        step_keys = torch.zeros((steps, S, 2, 2), dtype=torch.int32, device=dev)
        carry = kr.clone()
        _lib.check(L.pqn_rollout_keys(_lib.p(carry), _lib.p(step_keys), S, steps, mode, _lib.stream_ptr()), "pqn_rollout_keys")
        for t in range(steps):
            self.step(params, hs, obs, ld, la, q, S, N)
            self._act_step(S, N, step_keys[t], q, eps, state, nxt, act, rw, dn, mq, sums, 1, 1.0)
            obs, nxt = nxt, obs
            ld.copy_(dn); la.copy_(act)
        cnt = sums[:, 3]
        return {kk: torch.where(cnt > 0, sums[:, j] / cnt.clamp(min=1), torch.full_like(cnt, float("nan")))
                for j, kk in enumerate(INFO_KEYS)}
