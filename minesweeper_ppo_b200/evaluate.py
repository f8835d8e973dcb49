"""Greedy vectorised evaluation through the reference-shaped (NumPy) env API -- BASELINE.json
configs[0] (C1).

This is `eval.evaluate_vec` (eval.py:265-511) restated on the drop-in boundary: the callee builds
`VecMinesweeper(num_envs, env_cfg, seed)`, reads NumPy obs/mask each step, plays the greedy argmax of
the masked logits, reads `vec.envs[i].first_click_done / revealed / flags / mine_mask` for the belief
statistics (eval.py:350-360), calls `analyze_forced_modules(env)` and `analyze_avoidability(env, cell)`
per live env (eval.py:362-398) -- here two batched kernel launches per step behind the reference's
call shape -- then `vec.step(actions)` and the `infos["aux"] / ["outcome"]` lists (eval.py:405-416),
with the reference's episode accounting (only the first finished episode per env and batch counts,
eval.py:411-428).  Returns the reference's metric dict, key for key.  `tests/golden/c1_eval.npz` holds
the dict the unmodified reference produced for a scripted policy; `test_eval_matches_reference_metrics`
replays the same mine layouts through this function on the CUDA env and compares.

`evaluate_vec_device` returns the same dict with nothing per env crossing the bus: greedy action
(msw_masked_argmax), both analytics and the episode accounting (msw_eval_pre_step / msw_eval_post_step) run
on the device, and one 4-byte `finished` count is read back per step (DESIGN.md section 4.9).
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, List, Optional

import numpy as np
import torch

from . import _lib
from .avoidability import analyze_avoidability
from .env import EnvConfig, StepOut, VecMinesweeper
from .rules import analyze_forced_modules


def _auroc(labels: np.ndarray, scores: np.ndarray) -> float:
    """Rank AUROC as the reference computes it (eval.py:54-66): plain argsort ranks, ties not averaged."""
    labels, scores = labels.reshape(-1), scores.reshape(-1)
    n_pos, n_neg = float((labels == 1).sum()), float((labels == 0).sum())
    if n_pos == 0 or n_neg == 0:
        return float("nan")
    order = scores.argsort()
    ranks = np.empty(len(scores), dtype=np.float64)
    ranks[order] = np.arange(1, len(scores) + 1, dtype=np.float64)
    return float((ranks[labels == 1].sum() - n_pos * (n_pos + 1.0) / 2.0) / (n_pos * n_neg))


def _ece(probs: np.ndarray, labels: np.ndarray, bins: int = 15) -> float:
    """Expected calibration error over equal-width bins, last bin closed (eval.py:69-90)."""
    probs, labels = probs.reshape(-1), labels.reshape(-1)
    if probs.shape[0] == 0:
        return float("nan")
    edges = np.linspace(0.0, 1.0, bins + 1)
    total = 0.0
    for k in range(bins):
        sel = (probs >= edges[k]) & ((probs <= edges[k + 1]) if k == bins - 1 else (probs < edges[k + 1]))
        cnt = sel.sum()
        if cnt:
            total += (cnt / probs.shape[0]) * abs(labels[sel].mean() - probs[sel].mean())
    return float(total)


def _wilson(successes: int, total: int, z: float = 1.96):
    """95 % Wilson score interval (eval.py:447-458)."""
    if total <= 0:
        return float("nan"), float("nan")
    phat = successes / float(total)
    denom = 1.0 + (z * z) / total
    center = phat + (z * z) / (2.0 * total)
    rad = z * np.sqrt((phat * (1.0 - phat) / total) + (z * z) / (4.0 * total * total))
    return float((center - rad) / denom), float((center + rad) / denom)


def _ratio(num: float, den: float) -> float:
    return num / float(den) if den > 0 else float("nan")


@torch.no_grad()
def evaluate_vec(model: torch.nn.Module, env_cfg: EnvConfig, episodes: int = 1000, seed: int = 0,
                 num_envs: int = 256, max_steps_per_episode: int = 512,
                 vec_factory: Optional[Callable[..., VecMinesweeper]] = None) -> Dict[str, float]:
    """`vec_factory(num_envs=, cfg=, seed=)` lets a harness substitute the env the reference would build
    itself (the parity test injects the reference's mine layouts that way)."""
    device = next(model.parameters()).device
    was_training = model.training
    model.eval()                                                          # eval.py:278-279
    vec = (vec_factory or VecMinesweeper)(num_envs=num_envs, cfg=env_cfg, seed=seed)   # NumPy API
    batch = vec.reset()
    HW = env_cfg.H * env_cfg.W
    remaining, wins, total_steps, total_progress, invalids = episodes, 0, 0, 0.0, 0
    probs, labels = [], []
    forced_steps = forced_correct = guess_attempts = guess_success = 0
    reveal_total = forced_guess_total = forced_guess_success = forced_guess_episodes = 0
    safe_option_total = safe_option_hits = safe_option_misses = safe_cells = 0
    component_sizes: List[int] = []
    chosen_sizes: List[int] = []
    while remaining > 0:
        batch_size = min(num_envs, remaining)
        finished = 0
        counted = np.zeros(num_envs, dtype=bool)
        step_counters = np.zeros(num_envs, dtype=np.int32)
        ep_unavoidable = np.zeros(num_envs, dtype=bool)
        while finished < batch_size:
            obs = torch.from_numpy(batch["obs"]).to(device=device, dtype=torch.float32)
            mask = torch.from_numpy(batch["action_mask"]).to(device=device, dtype=torch.bool)
            empty = ~mask.any(dim=1)
            if empty.any():
                mask[empty] = True
            logits, _, mine_logits = model(obs, return_mine=True)         # fp32, no autocast (eval.py:333)
            assert logits.shape[1] == mask.shape[1] == vec.envs[0].action_space      # eval.py:22-27
            actions = logits.masked_fill(~mask, -1e9).argmax(dim=-1).cpu().numpy().astype(np.int32)
            picked = mask.cpu().numpy()[np.arange(num_envs), actions]
            invalids += int((~picked).sum())
            mine_prob = torch.sigmoid(mine_logits).cpu().numpy() if mine_logits is not None else None
            for idx, env in enumerate(vec.envs):                          # eval.py:350-398
                if counted[idx] or idx >= batch_size:
                    continue
                cell = int(actions[idx])
                safe = not env.mine_mask[cell // env.W, cell % env.W]
                if mine_prob is not None:
                    unknown = (~env.revealed) & (~env.flags)
                    if unknown.any():
                        probs.append(mine_prob[idx, 0][unknown].reshape(-1))
                        labels.append(env.mine_mask[unknown].astype(np.float32).reshape(-1))
                # forced reveals by the subset rule (eval.py:362-379); one batched kernel per step
                if cell in analyze_forced_modules(env)["subset_reveal"]:
                    forced_steps += 1; forced_correct += safe
                else:
                    guess_attempts += 1; guess_success += safe
                if env.first_click_done:                                  # eval.py:381-398, batched likewise
                    res = analyze_avoidability(env, cell)
                    component_sizes.extend(res.component_sizes)
                    if res.chosen_component_size is not None:
                        chosen_sizes.append(res.chosen_component_size)
                    reveal_total += 1
                    if res.avoidable:
                        safe_option_total += 1
                        safe_cells += res.count_forced_safe_cells
                        if res.chosen_is_forced_safe:
                            safe_option_hits += 1
                        else:
                            safe_option_misses += 1
                    else:
                        forced_guess_total += 1
                        ep_unavoidable[idx] = True
                        forced_guess_success += safe
            batch, rewards, dones, infos = vec.step(actions)
            step_counters += 1
            for i in range(num_envs):                                     # eval.py:405-428
                if not counted[i]:
                    total_progress += int(infos["aux"][i].get("last_new_reveals", 0)) / float(HW)
                if not counted[i] and dones[i]:
                    wins += infos["outcome"][i] == "win"
                    total_steps += int(step_counters[i]); step_counters[i] = 0
                    counted[i] = True; finished += 1
                    forced_guess_episodes += bool(ep_unavoidable[i])
                if not counted[i] and 0 < max_steps_per_episode <= step_counters[i]:
                    total_steps += int(step_counters[i]); step_counters[i] = 0
                    counted[i] = True; finished += 1
        remaining -= batch_size
    if was_training:
        model.train()
    p = np.concatenate(probs) if probs else np.zeros(0)
    y = np.concatenate(labels) if labels else np.zeros(0)
    ci_low, ci_high = _wilson(wins, max(1, episodes))
    reveal_den = float(max(1, reveal_total))
    return {                                                              # eval.py:490-510, key for key
        "win_rate": wins / max(1, episodes), "win_ci_low": ci_low, "win_ci_high": ci_high,
        "avg_steps": total_steps / max(1, episodes), "avg_progress": total_progress / max(1, episodes),
        "invalid_rate": invalids / max(1, total_steps),
        "forced_guess_rate": forced_guess_total / reveal_den,
        "forced_guess_success_rate": _ratio(forced_guess_success, forced_guess_total),
        "forced_guess_episode_rate": forced_guess_episodes / float(max(1, episodes)),
        "safe_option_rate": safe_option_total / reveal_den,
        "safe_option_miss_rate": _ratio(safe_option_misses, safe_option_total),
        "safe_option_pick_rate": _ratio(safe_option_hits, safe_option_total),
        "avg_safe_options_per_turn": _ratio(safe_cells, safe_option_total),
        "avg_frontier_component_size": _ratio(float(sum(component_sizes)), len(component_sizes)),
        "avg_selected_component_size": _ratio(float(sum(chosen_sizes)), len(chosen_sizes)),
        "belief_auroc": _auroc(y, p) if len(p) else float("nan"),
        "belief_ece": _ece(p, y) if len(p) else float("nan"),
        "wins": float(wins), "episodes": float(episodes),
        # extra (not in the reference dict): the subset-rule step statistics eval.py:362-379 accumulates
        "forced_step_rate": forced_steps / max(1, forced_steps + guess_attempts),
        "forced_step_accuracy": forced_correct / max(1, forced_steps),
        "guess_success_rate": guess_success / max(1, guess_attempts),
    }


def masked_argmax(logits: torch.Tensor, mask: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """int32 `logits.masked_fill(~mask, -1e9).argmax(-1)` of fp32 [n, A] logits in one launch (msw_masked_argmax),
    torch's tie and NaN rules included.  A row of `mask` without a legal action is made all-legal in place first."""
    if logits.device.type != "cuda":
        raise RuntimeError("masked_argmax runs on CUDA only (no CPU fallback in this package)")
    n, A = logits.shape
    if logits.dtype != torch.float32 or not logits.is_contiguous():
        raise ValueError("masked_argmax: logits must be a contiguous float32 [n, A] tensor")
    if mask.dtype != torch.bool or tuple(mask.shape) != (n, A) or not mask.is_contiguous() or mask.device != logits.device:
        raise ValueError("masked_argmax: mask must be a contiguous bool [n, A] tensor on the logits device")
    if out is None:
        out = torch.empty((n,), dtype=torch.int32, device=logits.device)
    if out.dtype != torch.int32 or tuple(out.shape) != (n,) or not out.is_contiguous() or out.device != logits.device:
        raise ValueError("masked_argmax: out must be a contiguous int32 [n] tensor on the logits device")
    with torch.cuda.device(logits.device):
        _lib.check(_lib.load().msw_masked_argmax(logits.data_ptr(), mask.data_ptr(), n, A, out.data_ptr(),
                                                 torch.cuda.current_stream().cuda_stream), "msw_masked_argmax")
    return out


_K = {name: k for k, name in enumerate(_lib.EVAL_COUNTERS)}
_INT64_MAX = (1 << 63) - 1


class _DeviceEvaluator:
    """State and per-step phases of `evaluate_vec_device`; every buffer is allocated once.  The phases are methods
    so that tools/eval_probe.py can time them one by one with CUDA events."""

    def __init__(self, model: torch.nn.Module, vec: VecMinesweeper, search_budget: int, max_steps: int):
        self.model, self.vec = model, vec
        self.search_budget, self.max_steps = int(search_budget), int(max_steps)
        n, HW, wpb, dev = vec.num_envs, vec.HW, vec.wpb, vec.device
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        self.out = StepOut(obs=z((n, _lib.OBS_CHANNELS, vec.H, vec.W), torch.float32), action_mask=z((n, HW), torch.bool),
                           rewards=z((n,), torch.float32), dones=z((n,), torch.bool))
        self.actions = z((n,), torch.int32)
        self.subset = z((n, wpb), torch.int32)
        self.safe, self.coc, self.cs = z((n, wpb), torch.int32), z((n, HW), torch.int16), z((n, HW), torch.int16)
        self.avoid_flags = z((n,), torch.uint8)
        self.counted, self.ep_unavoidable = z((n,), torch.uint8), z((n,), torch.uint8)
        self.step_counter = z((n,), torch.int32)
        self.sel, self.sel_mask = z((n, HW), torch.uint8), z((n, HW), torch.bool)
        self.prob: Optional[torch.Tensor] = None
        self.counters = z((len(_lib.EVAL_COUNTERS),), torch.int64)
        self.counters[_K["error_key"]] = _INT64_MAX
        self.finished = z((1,), torch.int32)
        self.finished_host = torch.zeros((1,), dtype=torch.int32).pin_memory()
        self.probs: List[torch.Tensor] = []
        self.labels: List[torch.Tensor] = []
        self.step_index = 0
        self.infos: Dict[str, torch.Tensor] = {}
        self.mine_logits: Optional[torch.Tensor] = None
        self.logits: Optional[torch.Tensor] = None
        vec.reset(out=self.out)

    def new_batch(self) -> None:
        for t in (self.counted, self.ep_unavoidable, self.step_counter, self.finished):
            t.zero_()

    def forward(self) -> None:
        logits, _, mine_logits = self.model(self.out.obs, return_mine=True)   # fp32, no autocast (eval.py:333)
        n, HW = self.vec.num_envs, self.vec.HW
        assert logits.shape[1] == self.out.action_mask.shape[1] == HW          # eval.py:22-27
        if logits.dtype != torch.float32:
            raise TypeError(f"evaluate_vec_device: the policy returned {logits.dtype} logits; it needs an fp32 forward")
        self.logits, self.mine_logits = logits.contiguous(), mine_logits

    def act(self) -> None:
        masked_argmax(self.logits, self.out.action_mask, out=self.actions)

    def analytics(self) -> None:
        self.vec._launch_forced_subset(self.subset)
        self.vec._launch_avoidability(self.safe, self.coc, self.cs, self.avoid_flags, self.search_budget)

    def account_pre(self, batch_size: int) -> None:
        vec, n, HW = self.vec, self.vec.num_envs, self.vec.HW
        belief = self.mine_logits is not None
        if belief:
            if self.prob is None:
                self.prob = torch.empty((n, HW), dtype=torch.float32, device=vec.device)
            torch.sigmoid(self.mine_logits.reshape(n, HW), out=self.prob)
        with torch.cuda.device(vec.device):
            _lib.check(vec._L.msw_eval_pre_step(
                C.byref(vec._desc), C.byref(vec._state), n, int(batch_size), self.actions.data_ptr(),
                self.out.action_mask.data_ptr(), self.subset.data_ptr(), self.safe.data_ptr(), self.coc.data_ptr(),
                self.cs.data_ptr(), self.avoid_flags.data_ptr(), self.counted.data_ptr(), self.ep_unavoidable.data_ptr(),
                self.sel.data_ptr() if belief else None, self.counters.data_ptr(), self.step_index, vec._stream()),
                "msw_eval_pre_step")
        if belief:      # the reference's order: step, env, cell in row-major order (eval.py:352-358)
            torch.ne(self.sel, 0, out=self.sel_mask)
            self.probs.append(self.prob.masked_select(self.sel_mask))
            self.labels.append(self.sel.masked_select(self.sel_mask))

    def step(self) -> None:
        _, _, _, self.infos = self.vec.step(self.actions, out=self.out, want_infos=True)

    def account_post(self) -> int:
        vec, it = self.vec, self.infos
        with torch.cuda.device(vec.device):
            _lib.check(vec._L.msw_eval_post_step(
                vec.num_envs, self.out.dones.data_ptr(), it["outcome_code"].data_ptr(), it["last_new_reveals"].data_ptr(),
                self.counted.data_ptr(), self.step_counter.data_ptr(), self.ep_unavoidable.data_ptr(), self.max_steps,
                self.counters.data_ptr(), self.finished.data_ptr(), vec._stream()), "msw_eval_post_step")
        self.step_index += 1
        self.finished_host.copy_(self.finished, non_blocking=True)
        torch.cuda.current_stream(vec.device).synchronize()
        return int(self.finished_host[0])

    def run_step(self, batch_size: int) -> int:
        self.forward()
        self.act()
        self.analytics()
        self.account_pre(batch_size)
        self.step()
        return self.account_post()

    def check_budget(self) -> None:
        key = int(self.counters[_K["error_key"]])
        if key != _INT64_MAX:
            n = self.vec.num_envs
            raise RuntimeError(f"evaluate_vec_device: exact search of env {key % n} exceeded its step budget at "
                               f"evaluation step {key // n}; pass a larger search_budget")

    def belief_pairs(self):
        """(probabilities f32, labels f32) of every belief pair, copied to the host once."""
        if not self.probs:
            return np.zeros(0), np.zeros(0)
        p = torch.cat(self.probs).cpu().numpy()
        y = (torch.cat(self.labels) - 1).cpu().numpy().astype(np.float32)
        return p, y


@torch.no_grad()
def evaluate_vec_device(model: torch.nn.Module, env_cfg: EnvConfig, episodes: int = 1000, seed: int = 0,
                        num_envs: int = 256, max_steps_per_episode: int = 512,
                        vec_factory: Optional[Callable[..., VecMinesweeper]] = None,
                        search_budget: int = 0) -> Dict[str, float]:
    """`evaluate_vec` with the per-env work on the device: the same metric dict, key for key.

    `vec_factory(num_envs=, cfg=, seed=, api="torch")` builds the env (default VecMinesweeper); `search_budget` is
    msw_avoidability's per-lane step budget (0 = its default), and an analysed env that exceeds it raises
    RuntimeError, as `analyze_avoidability` does.  `avg_progress` agrees with `evaluate_vec` to float64 summation
    order (DESIGN.md section 4.9); every other key is equal."""
    device = next(model.parameters()).device
    was_training = model.training
    model.eval()                                                          # eval.py:278-279
    vec = (vec_factory or VecMinesweeper)(num_envs=num_envs, cfg=env_cfg, seed=seed, api="torch")
    if vec.device != device:
        raise ValueError(f"evaluate_vec_device: model on {device}, env on {vec.device}")
    ev = _DeviceEvaluator(model, vec, search_budget, max_steps_per_episode)
    remaining = episodes
    try:
        while remaining > 0:
            batch_size = min(vec.num_envs, remaining)
            ev.new_batch()
            finished = 0
            while finished < batch_size:
                finished = ev.run_step(batch_size)
            ev.check_budget()
            remaining -= batch_size
    finally:
        if was_training:
            model.train()
    c = {k: int(v) for k, v in zip(_lib.EVAL_COUNTERS, ev.counters.cpu().tolist())}
    p, y = ev.belief_pairs()
    return _device_metrics(c, p, y, episodes, vec.HW)


def _device_metrics(c: Dict[str, int], p: np.ndarray, y: np.ndarray, episodes: int, HW: int) -> Dict[str, float]:
    """The dict of evaluate_vec (eval.py:490-510) from the device counters and the belief pairs."""
    wins, total_steps = c["wins"], c["total_steps"]
    ci_low, ci_high = _wilson(wins, max(1, episodes))
    reveal_den = float(max(1, c["reveal_total"]))
    forced_steps, guess_attempts = c["forced_steps"], c["guess_attempts"]
    return {
        "win_rate": wins / max(1, episodes), "win_ci_low": ci_low, "win_ci_high": ci_high,
        "avg_steps": total_steps / max(1, episodes),
        "avg_progress": c["new_reveals"] / float(HW) / max(1, episodes),
        "invalid_rate": c["invalid"] / max(1, total_steps),
        "forced_guess_rate": c["forced_guess_total"] / reveal_den,
        "forced_guess_success_rate": _ratio(c["forced_guess_success"], c["forced_guess_total"]),
        "forced_guess_episode_rate": c["forced_guess_episodes"] / float(max(1, episodes)),
        "safe_option_rate": c["safe_option_total"] / reveal_den,
        "safe_option_miss_rate": _ratio(c["safe_option_misses"], c["safe_option_total"]),
        "safe_option_pick_rate": _ratio(c["safe_option_hits"], c["safe_option_total"]),
        "avg_safe_options_per_turn": _ratio(c["safe_cells"], c["safe_option_total"]),
        "avg_frontier_component_size": _ratio(float(c["comp_size_sum"]), c["comp_count"]),
        "avg_selected_component_size": _ratio(float(c["chosen_size_sum"]), c["chosen_count"]),
        "belief_auroc": _auroc(y, p) if len(p) else float("nan"),
        "belief_ece": _ece(p, y) if len(p) else float("nan"),
        "wins": float(wins), "episodes": float(episodes),
        "forced_step_rate": forced_steps / max(1, forced_steps + guess_attempts),
        "forced_step_accuracy": c["forced_correct"] / max(1, forced_steps),
        "guess_success_rate": c["guess_success"] / max(1, guess_attempts),
    }
