#!/usr/bin/env python
"""Learning and timing of the recurrent PQN on MemoryChain-bsuite with the shipped preset
(+alg=pqn_rnn_memory_chain: memory_length 100, 1e5 steps, 8 seeds).  Prints one JSON line: the behaviour-policy and
greedy-eval returns over the updates, wall time per update (host clock between device synchronises, evaluation
excluded) and per evaluation, and the GPU name and power limit read in the same run.

    python scripts/learn_memory_chain.py [--out FILE] [hydra-style overrides ...]
"""
import json, os, subprocess, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from purejaxql_b200 import config_loader, pqn_rnn_gymnax, jaxrandom as jr

args = sys.argv[1:]
out_path = None
if "--out" in args:
    i = args.index("--out")
    out_path = args[i + 1]
    del args[i:i + 2]
seeds = 8
c = config_loader.compose(["+alg=pqn_rnn_memory_chain", f"NUM_SEEDS={seeds}", "SAVE_PATH=null"] + args)
cfg = {**c, **c["alg"]}
assert torch.cuda.is_available(), "needs a GPU"


def gpu_power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


t0 = time.perf_counter()
train = pqn_rnn_gymnax.make_train(cfg)
eng = train.engine
marks, eval_s = [], []
_eval = eng.get_test_metrics


def timed_eval(params, rng):
    torch.cuda.synchronize()
    ts = time.perf_counter()
    r = _eval(params, rng)
    torch.cuda.synchronize()
    eval_s.append(time.perf_counter() - ts)
    return r


def on_update_end(n, _state):
    torch.cuda.synchronize()
    marks.append((time.perf_counter(), len(eval_s)))


eng.get_test_metrics = timed_eval
eng.on_update_end = on_update_end
out = train(jr.to_numpy_u32(jr.split(jr.PRNGKey(0), seeds)))
torch.cuda.synchronize()
wall = time.perf_counter() - t0
# update n spans marks[n-1] -> marks[n] minus the evaluations run in between (those follow update n-1's end)
upd = [(b - a) - sum(eval_s[ea:eb]) for (a, ea), (b, eb) in zip(marks, marks[1:])]
m = out["metrics"]
ret = m["returned_episode_returns"].cpu().numpy()
tst = m["test/returned_episode_returns"].cpu().numpy()
tlen = m["test/returned_episode_lengths"].cpu().numpy()
n = ret.shape[1]
res = {"env": cfg["ENV_NAME"], "memory_length": cfg["ENV_KWARGS"]["memory_length"], "seeds": seeds,
       "total_timesteps": cfg["TOTAL_TIMESTEPS"], "num_updates": n, "num_envs": cfg["NUM_ENVS"],
       "window_steps_Tm": cfg["MEMORY_WINDOW"] + cfg["NUM_STEPS"], "hidden": cfg["HIDDEN_SIZE"],
       "test_num_envs": cfg["TEST_NUM_ENVS"], "test_num_steps": cfg["TEST_NUM_STEPS"],
       "gpu": torch.cuda.get_device_name(0), "gpu_power_limit": gpu_power_limit(),
       "cuda_graph": bool(eng.graph_captured), "wall_s_total": round(wall, 2),
       "update_ms_steady_median": round(1e3 * float(np.median(upd[1:])), 2) if len(upd) > 1 else None,
       "update_ms_all_after_first": [round(1e3 * u, 2) for u in upd],
       "eval_ms_median": round(1e3 * float(np.median(eval_s)), 2) if eval_s else None, "evaluations": len(eval_s),
       "train_return_mean_over_seeds@update": {i: round(float(ret[:, i].mean()), 4) for i in range(n)},
       "greedy_eval_return_mean_over_seeds@update": {i: round(float(np.nanmean(tst[:, i])), 4) for i in range(n)},
       "greedy_eval_return_per_seed_last": [round(float(x), 4) for x in tst[:, -1]],
       "greedy_eval_episode_length_last": round(float(np.nanmean(tlen[:, -1])), 2),
       "td_loss_last": round(float(m["td_loss"][:, -1].mean()), 6)}
line = json.dumps(res)
print(line)
if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write(line + "\n")
