"""Host vs device greedy evaluator (evaluate.evaluate_vec vs evaluate.evaluate_vec_device, DESIGN.md section 4.9).

    python tools/eval_probe.py --boards 16x16x40 --out profiles/eval_probe_16x16x40.json
    python tools/eval_probe.py --boards 16x30x99 --out profiles/eval_probe_16x30x99.json

For each board (16x16x40, 16x30x99), policy (parity.scripted_policy: cheap forward; the random-init medium
cnn_residual in fp32: a realistic forward) and num_envs in --sizes, both evaluators run with the same seed and
max(num_envs, --min-episodes) episodes.  The host evaluator runs only while its predicted time (the last host
run scaled by the episode ratio) stays under --host-limit seconds; where it stopped is recorded.  Reported per size:
wall seconds, episodes/s, per-step ms, belief pairs, the time of the final belief computation (copy + AUROC +
ECE) on its own, and whether the two dicts are equal.  A separate pass times forward / argmax / analytics /
accounting / env step per step with CUDA events.  The GPU name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import minesweeper_ppo_b200 as m  # noqa: E402
from minesweeper_ppo_b200 import evaluate as E  # noqa: E402
import parity as P  # noqa: E402

BOARDS = {"16x16x40": (16, 16, 40), "16x30x99": (16, 30, 99)}


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def make_policy(kind: str, H: int, W: int) -> torch.nn.Module:
    if kind == "scripted":
        return P.scripted_policy(H, W, seed=3).cuda()
    torch.manual_seed(0)
    return m.build_model("cnn_residual", obs_shape=(10, H, W),
                         model_cfg=dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256)).cuda()


def same(a: dict, b: dict) -> bool:
    for k, w in b.items():
        v = a[k]
        if isinstance(w, float) and math.isnan(w):
            if not math.isnan(v):
                return False
        elif k == "avg_progress":
            if abs(v - w) > 1e-12 * abs(w):
                return False
        elif v != w:
            return False
    return set(a) == set(b)


@torch.no_grad()
def device_run(model, cfg, episodes, num_envs, seed):
    """evaluate_vec_device's body, with the step loop and the final belief computation timed apart."""
    model.eval()
    vec = m.VecMinesweeper(num_envs, cfg, seed=seed, api="torch")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ev = E._DeviceEvaluator(model, vec, 0, 512)
    remaining = episodes
    while remaining > 0:
        bs = min(num_envs, remaining)
        ev.new_batch()
        while ev.run_step(bs) < bs:
            pass
        ev.check_budget()
        remaining -= bs
    t1 = time.perf_counter()
    c = {k: int(v) for k, v in zip(m._lib.EVAL_COUNTERS, ev.counters.cpu().tolist())}
    pairs = sum(int(t.numel()) for t in ev.probs)
    p, y = ev.belief_pairs()
    d = E._device_metrics(c, p, y, episodes, vec.HW)
    t2 = time.perf_counter()
    return d, {"wall_s": t2 - t0, "loop_s": t1 - t0, "belief_s": t2 - t1, "steps": ev.step_index,
               "belief_pairs": pairs, "episodes_per_s": episodes / (t2 - t0),
               "ms_per_step": 1e3 * (t1 - t0) / max(1, ev.step_index)}


def host_run(model, cfg, episodes, num_envs, seed):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d = E.evaluate_vec(model, cfg, episodes=episodes, seed=seed, num_envs=num_envs)
    t = time.perf_counter() - t0
    return d, {"wall_s": t, "episodes_per_s": episodes / t}


@torch.no_grad()
def split_run(model, cfg, num_envs, seed, steps):
    """CUDA events between the phases of `steps` evaluator steps (after 3 warm-up steps)."""
    model.eval()
    vec = m.VecMinesweeper(num_envs, cfg, seed=seed, api="torch")
    ev = E._DeviceEvaluator(model, vec, 0, 512)
    ev.new_batch()
    phases = [("forward", ev.forward), ("argmax", ev.act), ("analytics", ev.analytics),
              ("account_pre", lambda: ev.account_pre(num_envs)), ("env_step", ev.step), ("account_post", ev.account_post)]
    tot = {k: 0.0 for k, _ in phases}
    for s in range(3 + steps):
        if int(ev.finished_host[0]) >= num_envs:          # every env counted: start a new batch
            ev.new_batch()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(phases) + 1)]
        evs[0].record()
        for j, (_, fn) in enumerate(phases):
            fn()
            evs[j + 1].record()
        torch.cuda.synchronize()
        if s >= 3:
            for j, (k, _) in enumerate(phases):
                tot[k] += evs[j].elapsed_time(evs[j + 1])
    return {k: v / steps for k, v in tot.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "eval_probe.json"))
    ap.add_argument("--sizes", default="64,1024,8192,65536")
    ap.add_argument("--min-episodes", type=int, default=8192)
    ap.add_argument("--host-limit", type=float, default=90.0)
    ap.add_argument("--split-steps", type=int, default=20)
    ap.add_argument("--boards", default="16x16x40,16x30x99")
    ap.add_argument("--policies", default="scripted,cnn")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_probe needs a CUDA device")
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    sizes = [int(s) for s in a.sizes.split(",")]
    res = {"gpu": gpu_info(), "seed": 11, "max_steps_per_episode": 512,
           "cudnn_deterministic": True, "runs": [], "split_ms_per_step": []}
    for bname in a.boards.split(","):
        H, W, M = BOARDS[bname]
        cfg = m.EnvConfig(H=H, W=W, mine_count=M, step_penalty=1e-4)
        for pol in a.policies.split(","):
            model = make_policy(pol, H, W)
            device_run(model, cfg, 64, 64, 1)                       # warm-up: modules, cuDNN, allocator
            host_t, host_ep, host_stopped = None, None, None
            for n in sizes:
                ep = max(n, a.min_episodes)
                dd, dt = device_run(model, cfg, ep, n, 11)
                row = {"board": bname, "policy": pol, "num_envs": n, "episodes": ep, "device": dt}
                predicted = None if host_t is None else host_t * ep / host_ep      # host work ~ episodes
                if host_stopped is None and (predicted is None or predicted <= a.host_limit):
                    hd, ht = host_run(model, cfg, ep, n, 11)
                    row["host"] = ht
                    row["dicts_equal"] = same(dd, hd)
                    row["speedup"] = ht["wall_s"] / dt["wall_s"]
                    host_t, host_ep = ht["wall_s"], ep
                else:
                    host_stopped = host_stopped or n
                    row["host"] = f"not run: predicted {predicted:.0f} s > {a.host_limit:.0f} s"
                res["runs"].append(row)
                print(json.dumps(row), flush=True)
            for n in (1024, 65536):
                if n in sizes:
                    sp = {"board": bname, "policy": pol, "num_envs": n, **split_run(model, cfg, n, 11, a.split_steps)}
                    res["split_ms_per_step"].append(sp)
                    print(json.dumps(sp), flush=True)
            del model
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
