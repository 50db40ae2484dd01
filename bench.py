#!/usr/bin/env python
"""bench.py — MinAtar-Breakout PQN env-steps/s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...          # CPU arm (oracle port; see below)

One "step" = one full `_update_step` of the reference's train() (pqn_minatar.py:176-369)
for every seed on this rank: a 32-step rollout of 4096 envs (Q-network forward +
fused eps-greedy/env-step per step), the bootstrap forward + Q(lambda) scan, and
2 epochs x 32 minibatches of loss/grad + clip + RAdam.  Workload = BASELINE
configs[1]: Breakout-MinAtar, NUM_ENVS=4096, 128 seeds in total, sharded over
the ranks (seeds are independent runs: no data-path collective; total work is
fixed as N grows => "strong" scaling).

Keys of the JSON line: see the task contract.  `value` is whole-job env-steps/s
with everything resident in HBM; `e2e` runs the same K updates through the
public API (`make_train(config)` / `train(rngs)`) from HOST buffers — key upload,
parameter init, env reset, the K updates, and the device->host read of metrics
and final parameters are all inside the timed region.

`--impl reference`: the reference itself (JAX + gymnax) cannot be installed
here (no jax/gymnax/flax/optax wheels, no network), so the CPU arm is the
oracle port (oracle/, NumPy, one process + one BLAS thread per host core, one
independent seed each) on a bounded sample of the same workload: the true
NUM_ENVS=4096 and minibatch=4096, but 4 of the 32 rollout steps per "step"
(=> 4 of the 32 minibatches x 2 epochs: the same grad-steps per env-step);
`cpu_baseline.kind` = "port" and `cpu_baseline.sample` says so.

`--config acrobot65536` / `--config minatar5` measure BASELINE configs[3] / [2]
(their own metric strings); the default is the headline configs[1].
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TOTAL_SEEDS = 128
NUM_ENVS = 4096
NUM_STEPS = 32
METRIC = "MinAtar-Breakout env steps/sec @4096 envs x128 seeds"


def metric_name(args):
    """BASELINE.json's metric; non-default --envs / --seeds runs say so in the name."""
    if args.envs == NUM_ENVS and args.seeds == TOTAL_SEEDS:
        return METRIC
    return f"MinAtar-Breakout env steps/sec @{args.envs} envs x{args.seeds} seeds"


UNIT = "env_steps/s"
# algorithmic work per env-step (SURVEY.md section 8(d); restated in DESIGN.md)
FLOPS_FWD_PER_SAMPLE = 2 * (64 * 36 * 16 + 1024 * 128 + 128 * 3)        # conv + dense + head MACs x2
ALG_FLOPS = {  # per launch-unit sample, by kernel (DESIGN.md section 3)
    "dense_fwd": 2 * 1024 * 128, "wgrad": 2 * 1024 * 128, "dgrad": 2 * 1024 * 128,
    "tc_dense_fwd": 2 * 1024 * 128, "tc_wgrad": 2 * 1024 * 128, "tc_dgrad": 2 * 1024 * 128,
    "tc_dense_fwd_head": 2 * 1024 * 128 + 2 * 128 * 3,
    "conv_fwd": 2 * 64 * 36 * 16, "conv_bwd": 2 * 2 * 64 * 36 * 16,
}
ALG_BYTES = {  # HBM bytes per sample per launch the kernel must move (DESIGN.md section 3)
    "tc_dense_fwd": 4096 + 2 * 512 + 4,          # h1 in; h2 + xhat2 + rstd out (training epilogue)
    "tc_dense_fwd_head": 4096 + 12,              # h1 in; q[A] out (rollout epilogue)
    "tc_wgrad": 4096 + 2 * 512,                  # h1 in; dz2 + its tf32-lo in
    "tc_dgrad": 2 * 512 + 128 + 4096,            # dz2 (+lo), packed ReLU mask in; dy1 out
    "conv_fwd": 64 + 4096,                       # rollout variant; training adds xhat (4096) + rstd (256) + mask (128)
    "conv_bwd": 64 + 2 * 4096 + 256,             # obs, dy1, xhat, rstd in
}
CONV_FWD_TRAIN_BYTES = 64 + 2 * 4096 + 256 + 128


def base_config(num_updates, num_envs=NUM_ENVS, test=False):
    total = float(num_updates * NUM_STEPS * num_envs)
    return dict(ENV_NAME="Breakout-MinAtar", ALG_NAME="pqn", TOTAL_TIMESTEPS=total,
                TOTAL_TIMESTEPS_DECAY=1e7, NUM_ENVS=num_envs, NUM_STEPS=NUM_STEPS, NUM_MINIBATCHES=32, NUM_EPOCHS=2,
                EPS_START=1.0, EPS_FINISH=0.05, EPS_DECAY=0.1, LR=5e-4, MAX_GRAD_NORM=10, LR_LINEAR_DECAY=True,
                GAMMA=0.99, LAMBDA=0.65, NORM_TYPE="layer_norm", WANDB_MODE="disabled",
                TEST_DURING_TRAINING=test, TEST_INTERVAL=0.05, TEST_NUM_ENVS=128, EPS_TEST=0.0)


# --------------------------------------------------------------------------- #
# clocks sampling (nvidia-smi, during the timed region)
# --------------------------------------------------------------------------- #
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark(self):
        """Start of the timed region: samples taken before this index belong to the warm-up."""
        self.start_idx = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)                      # let the last 200 ms sample of the timed region land
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = self.rows[getattr(self, "start_idx", 0):]
        window = "timed region"
        if not rows:                          # timed region shorter than one sampling period: use the loaded
            rows = self.rows[-3:]             # warm-up samples right before it
            window = "last warm-up samples (timed region < 200 ms)"
        self.window = window
        for r in rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for n, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- #
# CPU arm: oracle port on a bounded sample
# --------------------------------------------------------------------------- #
SAMPLE_T = 1          # rollout steps per CPU "step" (of the workload's 32): bounded sample
SAMPLE_E = 1024       # envs per CPU worker (of the workload's 4096) => minibatch 1024 rows: large enough for BLAS to
                      # run at its large-GEMM rate; 128 workers x 4096 envs made one sample step take ~60 s


def cpu_port_steps(num_steps, warmup=0, sample_envs=SAMPLE_E, sample_t=SAMPLE_T):
    """Times `num_steps` sample steps of the oracle port for ONE seed: `sample_envs` envs, a rollout of `sample_t` of
    the 32 steps, Q(lambda), and sample_t minibatches x 2 epochs of `sample_envs` rows (the workload has T*E/32 = E
    rows per minibatch).  Returns (env_steps_per_s, seconds)."""
    from oracle import gymnax_envs as G
    from oracle import jax_prng as jr
    from oracle import pqn_ref as R
    cfg = base_config(10 ** 6, num_envs=sample_envs)
    cfg["NUM_STEPS"] = sample_t
    cfg["NUM_MINIBATCHES"] = sample_t
    cfg["NUM_UPDATES_DECAY"] = cfg["TOTAL_TIMESTEPS_DECAY"] // NUM_STEPS // NUM_ENVS
    env = G.make("Breakout-MinAtar")
    params = R.random_params(R.cnn_param_shapes(4, 3), 0)
    opt = R.opt_init(params)
    bs = {"mean": np.zeros(4, np.float32), "var": np.ones(4, np.float32)}
    obs, st = env.reset(jr.split(jr.PRNGKey(1), sample_envs))
    rng = jr.PRNGKey(2)
    lr_fn = lambda i: np.float32(5e-4)
    t0 = time.perf_counter()
    for u in range(warmup + num_steps):
        if u == warmup:
            t0 = time.perf_counter()
        params, opt, bs, obs, st, rng, m, _, _ = R.update_step(env, "cnn", params, opt, bs, obs, st, rng, cfg, u, lr_fn)
    dt = time.perf_counter() - t0
    return num_steps * sample_t * sample_envs / dt, dt


def _cpu_worker(q, num_steps, warmup, sample_envs, seed):
    # one independent seed per worker process, single BLAS thread each (seeds are independent runs,
    # exactly like the reference's vmap over seeds): this is the layout that uses every host core
    try:
        v, dt = cpu_port_steps(num_steps, warmup, sample_envs)
        q.put((v, dt))
    except Exception as e:  # pragma: no cover
        q.put(("error", repr(e)))


def cpu_port_parallel(num_steps, warmup=0, sample_envs=SAMPLE_E, max_workers=128):
    """Oracle port on all host cores: one process (1 BLAS thread) per core, one seed each.
    Returns (aggregate env_steps_per_s, seconds of the slowest worker's timed region, workers)."""
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0))
    n = max(1, min(cores, max_workers))
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_cpu_worker, args=(q, num_steps, warmup, sample_envs, i)) for i in range(n)]
    for p_ in procs:
        p_.start()
    res = [q.get() for _ in procs]
    for p_ in procs:
        p_.join()
    if any(r[0] == "error" for r in res):
        raise RuntimeError(str(res))
    # throughput from the workers' own timed regions (excludes interpreter start-up / imports)
    slowest = max(r[1] for r in res)
    return n * num_steps * SAMPLE_T * sample_envs / slowest, slowest, n


def cpu_sample_text(workers, steps, dt):
    return (f"{steps} sample steps of {workers} independent seeds (one process + 1 BLAS thread per host core); each sample "
            f"step = a bounded sample of the workload's update step: {SAMPLE_E} of the {NUM_ENVS} envs and {SAMPLE_T} of "
            f"the {NUM_STEPS} rollout steps per seed (Q forward + eps-greedy + env step, Q(lambda), then {SAMPLE_T} "
            f"minibatch(es) x 2 epochs of {SAMPLE_E} rows: the workload's grad-steps per env-step), {dt:.1f} s; oracle "
            f"port (NumPy) -- the reference's JAX-CPU path is not installable here (no jax/gymnax wheels)")


def headline_config(seeds_total, world, envs, with_eval=False, env_sharded=False):
    per = (seeds_total + world - 1) // world
    if env_sharded and world > 1:
        return {"workload": f"Breakout-MinAtar pqn_minatar NUM_ENVS={envs} x {seeds_total} seeds, envs sharded "
                            f"{envs // world}/GPU (every rank trains every seed), TEST_DURING_TRAINING=False",
                "num_steps": NUM_STEPS, "num_minibatches": 32, "num_epochs": 2,
                "l2": "per-step working set exceeds the 126 MB L2" if seeds_total * envs >= 1 << 16 else
                      "small run: the working set fits the L2; launch/latency bound",
                "parallelism": f"env-sharded x{world}: one NCCL all-reduce (mean) of the flat [S][P] gradient per "
                               f"minibatch step (64 per update), per-rank minibatch permutation"}
    return {"workload": f"Breakout-MinAtar pqn_minatar NUM_ENVS={envs} x {seeds_total} seeds "
                        f"(BASELINE configs[1]), seeds sharded {per}/GPU, TEST_DURING_TRAINING="
                        + ("True (greedy eval of 128 envs x 1000 steps every 3 updates inside the timed "
                           "region; its env-steps are not counted)" if with_eval else "False"),
            "num_steps": NUM_STEPS, "num_minibatches": 32, "num_epochs": 2,
            "l2": "per-step working set (obs rows + activations, >2 GB) exceeds the 126 MB L2",
            "parallelism": f"seed-sharded x{world}, no data-path collective"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)
    val, dt, workers = cpu_port_parallel(steps, warm)
    line = {"impl": "reference", "metric": metric_name(args), "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": headline_config(args.seeds, max(world, args.gpus), args.envs),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": workers, "kind": "port",
                             "sample": cpu_sample_text(workers, steps, dt)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# per-kernel algorithmic work (DESIGN.md section 3): bytes / flops per unit the launch processes
#   unit "mb"  : one sample of a minibatch launch (T*E/32 samples per seed)
#   unit "env" : one env of a rollout / evaluation launch (E per seed)
# --------------------------------------------------------------------------- #
KERNELS = {
    "conv_fwd": dict(unit="mb", bound="hbm", bytes=64 + 2 * 4096 + 256 + 128,
                     note="conv3x3+LayerNorm+ReLU (training): 64 B packed obs in; h1, xhat, rstd, ReLU bitmask out"),
    "conv_fwd_infer": dict(unit="env", bound="hbm", bytes=64 + 4096,
                           note="conv3x3+LayerNorm+ReLU (rollout): 64 B packed obs in, h1 out"),
    "conv_bwd": dict(unit="mb", bound="hbm", bytes=64 + 2 * 4096 + 256,
                     note="LayerNorm backward + conv weight gradient: obs, dy1, xhat, rstd in; reduced gradients out"),
    "tc_dense_fwd": dict(unit="mb", bound="tensor", flops=2 * 1024 * 128, bytes=4096 + 2 * 512 + 4),
    "tc_dense_fwd_head": dict(unit="env", bound="tensor", flops=2 * 1024 * 128 + 2 * 128 * 3, bytes=4096 + 12),
    "tc_wgrad": dict(unit="mb", bound="tensor", flops=2 * 1024 * 128, bytes=4096 + 2 * 512),
    "tc_dgrad": dict(unit="mb", bound="tensor", flops=2 * 1024 * 128, bytes=2 * 512 + 128 + 4096),
    "row_bwd": dict(unit="mb", bound="hbm", bytes=3 * 512 + 4 + 2 * 512 + 12,
                    note="head/loss/LayerNorm(128) backward: h2, xhat2, rstd in; dz2 (+lo) out"),
    "rollout_act_step": dict(unit="env", bound="hbm", bytes=(44 + 12) + (44 + 64 + 4 + 4 + 1 + 4),
                             note="fused eps-greedy + env step + packed-obs/transition stores"),
}
NCU_NAMES = {"conv_bwd": "conv_bwd", "conv_fwd": "conv_fwd", "conv_fwd_infer": "conv_fwd_infer",
             "tc_dense_fwd_head": "tc_dense_fwd_head", "tc_dense_fwd": "tc_dense_fwd", "tc_wgrad": "tc_wgrad",
             "tc_dgrad": "tc_dgrad", "row_bwd": "row_bwd"}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def load_traffic():
    """dram bytes per launch of each kernel id from the committed `ncu --set full` capture of this round
    (profiles/r2_traffic.json: {kernel id: bytes}); empty if the file is absent."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
    except Exception:
        return {}


def roofline_for(dom, prof, S, envs, peaks, traffic, headline_geometry):
    d_ms, d_n = prof[dom]
    k = KERNELS.get(dom)
    hbm = peaks.get("hbm_gbs", 6650.0)
    peak_src_h = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6.65 TB/s (of fallback)"
    base = {"kernel": dom, "avg_launch_ms": round(d_ms / d_n, 4), "launches": d_n,
            "traffic": traffic.get(dom) if headline_geometry else None,
            "traffic_source": "profiles/r2_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum "
                              "per launch, same workload)" if (headline_geometry and dom in traffic) else None}
    if k is None:
        return {"bound": "hbm", "achieved": None, "peak": hbm, "unit": "GB/s", "frac": None, **base}
    mb = NUM_STEPS * envs // 32
    units = S * (mb if k["unit"] == "mb" else envs)            # per launch
    if k["bound"] == "hbm":
        gbs = k["bytes"] * units / (d_ms / d_n / 1e3) / 1e9
        return {"bound": "hbm", "achieved": round(gbs, 1), "peak": hbm, "unit": "GB/s", "frac": round(gbs / hbm, 4),
                "peak_source": peak_src_h, "alg_bytes_per_unit": k["bytes"], "units_per_launch": units,
                "note": k.get("note", ""), **base}
    peak = peaks.get("bf16_tflops_sustained") or 1400.0
    tf = k["flops"] * units / (d_ms / d_n / 1e3) / 1e12
    gbs = k["bytes"] * units / (d_ms / d_n / 1e3) / 1e9
    return {"bound": "tensor", "achieved": round(tf, 2), "peak": peak, "unit": "TFLOP/s", "frac": round(tf / peak, 4),
            "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks
                            else "fallback 1.4 PF sustained (of fallback)"),
            "alg_flops_per_unit": k["flops"], "units_per_launch": units,
            "note": "fp32-accurate split-precision GEMM on tcgen05 (3 tensor-core products per algorithmic one); the "
                    "fraction is algorithmic fp32 FLOP/s against the dense bf16 peak -- see DESIGN.md section 3 for the "
                    "format-equivalent peak",
            "hbm_gbs": round(gbs, 1), "hbm_frac": round(gbs / hbm, 4), **base}


# --------------------------------------------------------------------------- #
# standalone env.step roofline (north star: "achieved fraction of the HBM roofline"), with clocks
# --------------------------------------------------------------------------- #
def env_step_roofline(dev, local_rank, peaks, names=("Breakout-MinAtar",)):
    import torch
    from purejaxql_b200 import _lib, envs, jaxrandom as jr
    L = _lib.lib()
    hbm = peaks.get("hbm_gbs", 6650.0)
    out = {}
    for name in names:
        n = (1 << 20) if name.endswith("MinAtar") else (1 << 24)
        env, params = envs.make(name)
        keys = jr.split(jr.PRNGKey(0, dev), n)
        obs, st = env.reset(keys, params)
        del obs
        act = torch.randint(0, env.num_actions, (n,), dtype=torch.int32, device=dev)
        o = torch.empty((n, env.obs_dim), dtype=torch.float32, device=dev)
        r = torch.empty(n, device=dev); d = torch.empty(n, dtype=torch.uint8, device=dev)
        i0 = torch.empty(n, device=dev); i1 = torch.empty(n, device=dev)
        i2 = torch.empty(n, dtype=torch.int32, device=dev); i3 = torch.empty(n, dtype=torch.int32, device=dev)

        def step():
            _lib.check(L.pqn_env_step(env.env_id, _lib.p(keys), _lib.p(st), _lib.p(act), _lib.p(o), _lib.p(r), _lib.p(d),
                                      _lib.p(i0), _lib.p(i1), _lib.p(i2), _lib.p(i3), n, 0, 0, _lib.stream_ptr()))
        for _ in range(5):
            step()
        torch.cuda.synchronize(dev)
        sampler = ClockSampler(local_rank)
        sampler.start()
        iters = 600 if name.endswith("MinAtar") else 300       # >= 0.4 s so that the clock sampler sees the load
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        time.sleep(0.25)
        sampler.mark()
        a.record()
        for _ in range(iters):
            step()
        b.record()
        torch.cuda.synchronize(dev)
        clocks = sampler.stop()
        ms = a.elapsed_time(b) / iters
        sw = env.state_words * 4
        bytes_per = (sw + 4 + 8) + (sw + env.obs_dim * 4 + 4 + 1 + 16)   # read state/action/key; write state/obs/r/done/info
        gbs = bytes_per * n / (ms * 1e-3) / 1e9
        out[name] = {"kernel": "env_step_kernel (standalone LogWrapper(env).step, fp32 obs)", "envs": n,
                     "avg_launch_ms": round(ms, 4), "launches": iters, "alg_bytes_per_env_step": bytes_per,
                     "env_steps_per_s": n / (ms * 1e-3), "achieved": round(gbs, 1), "peak": hbm, "unit": "GB/s",
                     "frac": round(gbs / hbm, 4), "clocks": clocks,
                     "l2": f"state + outputs of {n} envs ({bytes_per * n / 1e6:.0f} MB per launch) exceed the 126 MB L2"}
        del o, r, d, i0, i1, i2, i3, st, keys, act
    return out


# --------------------------------------------------------------------------- #
# GPU arm
# --------------------------------------------------------------------------- #
def timed_train(module, cfg, rngs_host, warmup, dev, world, local_rank, profile=False, shard=None):
    """One train() of warmup+K updates; updates warmup.. are bracketed by CUDA events on the launching stream
    (hook called on the host between updates).  Returns (ms, launches in the timed region, clocks, out, per-kernel
    spans or None)."""
    import torch
    import torch.distributed as dist
    from purejaxql_b200 import _lib
    L = _lib.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    train = module.make_train(cfg)
    eng = train.engine
    if shard is not None:
        eng.env_shard = shard
    ev = {"start": torch.cuda.Event(enable_timing=True), "end": torch.cuda.Event(enable_timing=True)}
    sampler = ClockSampler(local_rank)
    state = {"launch0": 0, "replays0": 0}

    def on_update(n):
        if n == warmup:
            barrier()
            if profile:
                L.pqn_profile_read((_lib.c_double * L.pqn_num_kernels())(), (_lib.c_longlong * L.pqn_num_kernels())(), 1)
                L.pqn_profile_enable(1)
            state["launch0"] = L.pqn_launch_count()
            state["replays0"] = getattr(eng, "graph_replays", 0)
            sampler.mark()
            ev["start"].record(torch.cuda.current_stream(dev))
    eng.on_update_begin = on_update
    sampler.start()                           # runs through the warm-up; mark() at the start of the timed region
    out = train(rngs_host)
    ev["end"].record(torch.cuda.current_stream(dev))
    barrier()
    clocks = sampler.stop()
    launches = L.pqn_launch_count() - state["launch0"]
    launches += (eng.graph_replays - state["replays0"]) * eng.graph_launches_per_replay
    prof = None
    if profile:
        L.pqn_profile_enable(0)
        prof = _lib.profile_read(reset=True)
    ms = ev["start"].elapsed_time(ev["end"])
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), int(launches), clocks, out, prof, eng


DUMP_MAX_ELEMS = 1 << 20     # per array; a larger output is dumped as a fixed, seeded sample of its flattened entries
DUMP_MAX_BYTES = 64 << 20    # all files of one --dump-outputs together


def dump_outputs(out_dir, out):
    """Writes what train() returned after its last update as <out_dir>/<name>.npy, so that two builds run with the
    same arguments can be compared output for output: the last column of every metric, the final parameters, RAdam
    moments, normalisation statistics, observations, env state and runner key.  Floating-point arrays are written as
    float32, integer ones (packed observation words, env state, counters) as float64, which holds them exactly.  An
    array of more than DUMP_MAX_ELEMS entries keeps the flattened entries at the sorted positions
    np.random.default_rng(0).choice(size, DUMP_MAX_ELEMS, replace=False): the same positions on every run."""
    train_state, (obs, env_state), _, rng = out["runner_state"]
    arrays = {f"metrics_{k.replace('/', '_')}": v[:, -1] for k, v in out["metrics"].items()}
    arrays.update(params=train_state.params_flat, radam_mu=train_state.opt_state.mu,
                  radam_nu=train_state.opt_state.nu, batch_stats=train_state.batch_stats_flat,
                  obs_packed=obs, env_state=env_state, rng=rng)
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.cpu().numpy().reshape(-1)
        a = a.astype(np.float32 if np.issubdtype(a.dtype, np.floating) else np.float64)
        if a.size > DUMP_MAX_ELEMS:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        total += a.nbytes
        assert total <= DUMP_MAX_BYTES, f"--dump-outputs would exceed {DUMP_MAX_BYTES} bytes"
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


E2E_PARTS = {}     # wall-clock split of the last e2e_train call (this rank)


def e2e_train(module, cfg, rngs_host, dev, world, shard=None):
    import torch
    import torch.distributed as dist
    import gc
    gc.collect()                          # the previous engine's buffers go back to the caching allocator now, not
    gc.disable()                          # in the middle of the timed call (a collection pause is host time)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    train2 = module.make_train(cfg)
    if shard is not None:
        train2.engine.env_shard = shard
    marks = [torch.cuda.Event(enable_timing=True)]           # per-update GPU time of this run (diagnostic, no sync)
    marks[0].record()

    def _mark(n, dbg):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append(ev)
    train2.engine.on_update_end = _mark
    t1 = time.perf_counter()
    out2 = train2(rngs_host)                                   # H2D of the keys happens inside; train() ends synchronised
    t2 = time.perf_counter()
    metrics_host = {k: v.cpu() for k, v in out2["metrics"].items()}
    params_host = out2["runner_state"][0].params_flat.cpu()
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    gc.enable()
    E2E_PARTS.update(make_train_s=round(t1 - t0, 4), train_s=round(t2 - t1, 4), d2h_s=round(t0 + e2e_s - t2, 4))
    E2E_PARTS["gpu_ms_init_then_per_update"] = [round(marks[i].elapsed_time(marks[i + 1]), 1) for i in range(len(marks) - 1)]
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    d2h = sum(v.numel() * v.element_size() for v in metrics_host.values()) + params_host.numel() * 4
    return float(te.item()), rngs_host.nbytes, d2h


def run_gpu(args, rank, world, local_rank):
    import torch
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from purejaxql_b200 import jaxrandom as jr, pqn_minatar

    seeds_total = args.seeds
    env_sharded = args.data_parallel == "envs" or (args.data_parallel == "auto" and seeds_total < world)
    all_rngs = jr.to_numpy_u32(jr.split(jr.PRNGKey(0, dev), seeds_total))      # same split as single_run
    if env_sharded:      # every rank trains every seed on its shard of the envs; one gradient all-reduce per minibatch step
        per, S = seeds_total, seeds_total
        rngs_host = np.ascontiguousarray(all_rngs)
        assert args.envs % world == 0
    else:
        per = (seeds_total + world - 1) // world
        lo, hi = min(seeds_total, rank * per), min(seeds_total, (rank + 1) * per)
        S = hi - lo
        rngs_host = np.ascontiguousarray(all_rngs[lo:hi])
    shard = (rank, world) if env_sharded and world > 1 else None

    # ---- (1) the timed region: W warm-up + K timed updates of ONE train(), no per-kernel profiling; the update is
    # replayed from a CUDA graph when the engine's "auto" rule applies (S*E*T <= 2^21, e.g. 16 seeds/GPU), exactly
    # what `single_run` users get
    cfg = base_config(args.warmup + args.steps, num_envs=args.envs, test=args.with_eval)
    if args.with_eval:  # the reference's cadence at this config: a greedy evaluation every 3 updates (int(76 * 0.05))
        cfg["TEST_INTERVAL"] = 3.5 / (args.warmup + args.steps)
    ms_max, launches, clocks, out, _, eng = timed_train(pqn_minatar, cfg, rngs_host, args.warmup, dev, world, local_rank,
                                                        shard=shard)
    graph_used = bool(eng.graph_captured)
    env_steps = seeds_total * args.steps * NUM_STEPS * args.envs
    value = env_steps / (ms_max / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)

    # ---- (2) e2e through the public API from host buffers
    e2e_s, h2d, d2h = e2e_train(pqn_minatar, base_config(args.steps, num_envs=args.envs), rngs_host, dev, world, shard=shard)
    e2e_val = env_steps / e2e_s

    # ---- (3) per-kernel CUDA-event spans from a second, eager pass of the same updates (1 warm-up + 2 profiled):
    # every library launch is bracketed by an event pair on the launching stream, which costs ~1 % of the step --
    # that is why `value` comes from pass (1)
    pcfg = base_config(3, num_envs=args.envs)
    pcfg["CUDA_GRAPH"] = False
    p_ms, _, _, _, prof, _ = timed_train(pqn_minatar, pcfg, rngs_host, 1, dev, world, local_rank, profile=True, shard=shard)
    if rank != 0:
        return
    peaks = load_peaks()
    traffic = load_traffic()
    headline_geometry = (S == 128 and args.envs == NUM_ENVS)
    total_k_ms = sum(v[0] for v in prof.values()) or 1.0
    breakdown = {k: {"ms_per_update": round(v[0] / 2, 3), "launches_per_update": v[1] // 2,
                     "share": round(v[0] / total_k_ms, 4)}
                 for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    dom = max(prof.items(), key=lambda kv: kv[1][0])[0] if prof else None
    roof = roofline_for(dom, prof, S, args.envs, peaks, traffic, headline_geometry) if dom else None
    if roof is not None:
        roof["measured_in"] = ("second pass of the same workload inside this bench.py run (2 eager updates, every "
                               "launch bracketed by CUDA events on the launching stream); profiled step = "
                               f"{p_ms / 2:.1f} ms vs {ms_max / args.steps:.1f} ms unprofiled")
    rooflines = {k: roofline_for(k, prof, S, args.envs, peaks, traffic, headline_geometry)
                 for k in prof if k in KERNELS and k != dom}

    # ---- (4) standalone env.step against the HBM roofline, with its own clock samples
    env_roof = None
    if not args.no_env_roofline:
        env_roof = env_step_roofline(dev, local_rank, peaks)

    # ---- (5) cpu baseline (bounded sample, rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu:
        v, dt, workers = cpu_port_parallel(3, 1)
        cpu = {"value": v, "unit": UNIT, "cores": workers, "kind": "port", "sample": cpu_sample_text(workers, 3, dt)}

    # (R) rollout-engine throughput (SURVEY section 8(d)): env step + eps-greedy + Q forward + Q(lambda), from the
    # CUDA-event spans of the rollout-phase kernels of pass (3) (kernel time only, this rank)
    roll_keys = ("rollout_act_step", "rollout_keys", "qlambda", "conv_fwd_infer", "tc_dense_fwd_head")
    roll_ms = sum(prof[k][0] for k in roll_keys if k in prof)
    if "tc_split" in prof and "tc_dense_fwd_head" in prof:  # the weight split runs once per forward, either phase
        n_fwd = prof["tc_dense_fwd_head"][1] + prof.get("tc_dense_fwd", (0, 0))[1]
        roll_ms += prof["tc_split"][0] * prof["tc_dense_fwd_head"][1] / max(n_fwd, 1)
    rollout_engine = None
    if roll_ms > 0:
        rollout_engine = {"value": S * 2 * NUM_STEPS * args.envs / (roll_ms / 1e3) * world, "unit": UNIT,
                          "kernel_ms_per_update": round(roll_ms / 2, 3),
                          "what": "rollout phase only (env step + eps-greedy + Q-network forward + Q(lambda) targets): "
                                  "sum of the per-kernel CUDA-event spans of rank 0 in pass (3), x n_gpus"}

    line = {"metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": headline_config(seeds_total, world, args.envs, args.with_eval, env_sharded),
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d / args.steps,
                    "d2h_bytes_per_step": d2h / args.steps,
                    "what": "make_train(config)+train(host rngs): key upload, init, reset, K updates, D2H of metrics+params",
                    "wall_split_rank0": dict(E2E_PARTS)},
            "gpu_launches": int(launches), "cuda_graph": graph_used,
            "roofline": roof, "env_step": env_roof, "rollout_engine": rollout_engine, "kernel_breakdown": breakdown,
            "other_rooflines": rooflines,
            "td_loss_last": float(out["metrics"]["td_loss"][:, -1].mean())}
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# the other BASELINE configs (each prints its own line; not the driver's headline)
# --------------------------------------------------------------------------- #
def run_acrobot(args, rank, world, local_rank):
    """BASELINE configs[3]: Acrobot-v1 pqn_gymnax NUM_ENVS=65536 fp32 on one B200 (TOTAL_TIMESTEPS overridden,
    SURVEY 8: the shipped value gives 0 updates)."""
    import torch
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from purejaxql_b200 import config_loader, jaxrandom as jr, pqn_gymnax
    E = 65536

    def cfg_for(n):
        c = config_loader.compose(["+alg=pqn_cartpole", "alg.ENV_NAME=Acrobot-v1", "NUM_SEEDS=1", "SAVE_PATH=null",
                                   f"alg.NUM_ENVS={E}", "alg.TEST_DURING_TRAINING=False"])
        c = {**c, **c["alg"]}
        c["TOTAL_TIMESTEPS"] = c["TOTAL_TIMESTEPS_DECAY"] = float(n * c["NUM_STEPS"] * E)
        return c
    rngs = np.ascontiguousarray(jr.to_numpy_u32(jr.split(jr.PRNGKey(0, dev), 1)))
    c = cfg_for(args.warmup + args.steps)
    T = int(c["NUM_STEPS"])
    ms, launches, clocks, out, _, eng = timed_train(pqn_gymnax, c, rngs, args.warmup, dev, 1, local_rank)
    env_steps = args.steps * T * E
    e2e_s, h2d, d2h = e2e_train(pqn_gymnax, cfg_for(args.steps), rngs, dev, 1)
    pc = cfg_for(3)
    pc["CUDA_GRAPH"] = False
    _, _, _, _, prof, _ = timed_train(pqn_gymnax, pc, rngs, 1, dev, 1, local_rank, profile=True)
    peaks = load_peaks()
    total = sum(v[0] for v in prof.values()) or 1.0
    breakdown = {k: {"ms_per_update": round(v[0] / 2, 3), "launches_per_update": v[1] // 2, "share": round(v[0] / total, 4)}
                 for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    env_roof = env_step_roofline(dev, local_rank, peaks, names=("Acrobot-v1",))
    line = {"metric": "Acrobot-v1 pqn_gymnax env steps/sec @65536 envs, 1 seed (BASELINE configs[3])",
            "value": env_steps / (ms / 1e3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"Acrobot-v1 pqn_gymnax (pqn_cartpole.yaml) NUM_ENVS={E}, NUM_STEPS={T}, "
                                   f"{c['NUM_MINIBATCHES']} minibatches x {c['NUM_EPOCHS']} epochs, MLP "
                                   f"{c.get('HIDDEN_SIZE')}x{c.get('NUM_LAYERS')}, 1 seed",
                       "l2": "rollout buffers + activations of 4.2 M samples per update exceed the 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": env_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d / args.steps,
                    "d2h_bytes_per_step": d2h / args.steps},
            "gpu_launches": launches, "cuda_graph": bool(eng.graph_captured), "env_step": env_roof,
            "roofline": env_roof["Acrobot-v1"] | {"bound": "hbm"}, "kernel_breakdown": breakdown}
    print(json.dumps(line), flush=True)


def run_minatar5(args, rank, world, local_rank):
    """BASELINE configs[2]: the MinAtar suite at NUM_ENVS=1024 x 16 seeds on one B200 -- one line per game that gymnax
    0.0.6 registers (Seaquest-MinAtar is not registered there; DESIGN.md section 8)."""
    import torch
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from purejaxql_b200 import config_loader, envs, jaxrandom as jr, pqn_minatar
    peaks = load_peaks()
    for game in envs.MINATAR_GAMES:
        def cfg_for(n):
            c = config_loader.compose(["+alg=pqn_minatar", f"alg.ENV_NAME={game}", "NUM_SEEDS=16", "SAVE_PATH=null",
                                       "alg.NUM_ENVS=1024", "alg.TEST_DURING_TRAINING=False"])
            c = {**c, **c["alg"]}
            c["TOTAL_TIMESTEPS"] = float(n * c["NUM_STEPS"] * 1024)
            return c
        rngs = np.ascontiguousarray(jr.to_numpy_u32(jr.split(jr.PRNGKey(0, dev), 16)))
        ms, launches, clocks, out, _, eng = timed_train(pqn_minatar, cfg_for(args.warmup + args.steps), rngs, args.warmup,
                                                        dev, 1, local_rank)
        env_steps = 16 * args.steps * 32 * 1024
        e2e_s, h2d, d2h = e2e_train(pqn_minatar, cfg_for(args.steps), rngs, dev, 1)
        env_roof = env_step_roofline(dev, local_rank, peaks, names=(game,))
        line = {"metric": f"{game} pqn_minatar env steps/sec @1024 envs x16 seeds (BASELINE configs[2])",
                "value": env_steps / (ms / 1e3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"{game} pqn_minatar.yaml NUM_ENVS=1024 x 16 seeds, 32 steps, 32 minibatches x 2 epochs"},
                "clocks": clocks,
                "e2e": {"value": env_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d / args.steps,
                        "d2h_bytes_per_step": d2h / args.steps},
                "gpu_launches": launches, "cuda_graph": bool(eng.graph_captured),
                "roofline": env_roof[game] | {"bound": "hbm"}, "env_step": env_roof}
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--seeds", type=int, default=TOTAL_SEEDS)
    ap.add_argument("--envs", type=int, default=NUM_ENVS)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-env-roofline", action="store_true")
    ap.add_argument("--config", default="headline", choices=["headline", "acrobot65536", "minatar5"])
    ap.add_argument("--data-parallel", default="auto", choices=["auto", "seeds", "envs"],
                    help="seeds: shard the independent seeds (no collective); envs: shard NUM_ENVS of every seed and "
                         "all-reduce the gradient once per minibatch step; auto: envs when --seeds < #GPUs")
    ap.add_argument("--with-eval", action="store_true",
                    help="TEST_DURING_TRAINING=True with the reference's cadence (SURVEY 8(d): report both)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed updates, write what train() returned after the last one as DIR/<name>.npy "
                         "(headline config; with several GPUs, rank 0's seeds)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "b200" or args.config != "headline"):
        ap.error("--dump-outputs is implemented for the headline config of the CUDA path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.config == "acrobot65536":
            if rank == 0:
                run_acrobot(args, rank, world, local_rank)
        elif args.config == "minatar5":
            if rank == 0:
                run_minatar5(args, rank, world, local_rank)
        else:
            run_gpu(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
