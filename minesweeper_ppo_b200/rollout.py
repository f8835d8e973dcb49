"""Device-resident rollout collector with the reference's `collect_rollout` signature
(train_rl.py:155-289).

Per step the reference crosses the host/device boundary five times (obs/mask H2D, aux labels H2D,
actions D2H + sync, rewards/dones H2D; train_rl.py:198-199, 203-219, 239, 246-247) and then copies
seven tensors into the buffer (buffers.py:53-59).  Here nothing leaves the device and nothing is
copied: the env kernel writes obs_{t+1} / mask_{t+1} / labels_{t+1} / valid_{t+1} into slot t+1 and
reward_t / done_t into slot t of the `RolloutBuffer`, the fused sampler (msw_masked_sample) reads the
mask the env kernel just wrote and writes actions / log-probs into slot t, and there is no host
synchronisation inside the T loop.  The policy forward is the unchanged PyTorch/cuDNN module under
fp16 autocast (train_rl.py:222-227).
"""
from __future__ import annotations

import time
from contextlib import nullcontext
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib
from .buffers import CompactRolloutBuffer, RolloutBuffer
from .env import StepOut, VecMinesweeper
from .fused_forward import make_rollout_forward, supports_fused

_DTYPE_CODE = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def masked_sample(logits: torch.Tensor, mask: torch.Tensor, *, seed: int, step_index: int, row_id_base: int = 0,
                  actions64: Optional[torch.Tensor] = None, actions32: Optional[torch.Tensor] = None,
                  logp: Optional[torch.Tensor] = None, epoch: Optional[torch.Tensor] = None
                  ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Masked Categorical sample + log_prob in one launch (replaces train_rl.py:229-235, :239)."""
    L = _lib.load()
    if logits.device.type != "cuda":
        raise RuntimeError("masked_sample runs on CUDA only (no CPU fallback in this package)")
    n, A = logits.shape
    logits = logits.contiguous()
    if logits.dtype not in _DTYPE_CODE:
        logits = logits.float()
    if mask.dtype != torch.bool or tuple(mask.shape) != (n, A) or not mask.is_contiguous():
        raise ValueError("masked_sample: mask must be a contiguous bool [n, A] tensor")
    dev = logits.device
    if actions64 is None:
        actions64 = torch.empty((n,), dtype=torch.int64, device=dev)
    if actions32 is None:
        actions32 = torch.empty((n,), dtype=torch.int32, device=dev)
    if logp is None:
        logp = torch.empty((n,), dtype=torch.float32, device=dev)
    for t, dt in ((actions64, torch.int64), (actions32, torch.int32), (logp, torch.float32)):
        if t.dtype != dt or tuple(t.shape) != (n,) or not t.is_contiguous() or t.device != dev:
            raise ValueError("masked_sample: outputs must be contiguous [n] tensors of the right dtype on the logits device")
    with torch.cuda.device(dev):
        rc = L.msw_masked_sample(logits.data_ptr(), _DTYPE_CODE[logits.dtype], mask.data_ptr(), n, A,
                                 int(seed) & 0xFFFFFFFFFFFFFFFF, int(step_index) & 0xFFFFFFFFFFFFFFFF,
                                 None if epoch is None else epoch.data_ptr(),
                                 int(row_id_base), actions64.data_ptr(), actions32.data_ptr(), logp.data_ptr(),
                                 torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "msw_masked_sample")
    return actions64, actions32, logp


class RolloutCollector:
    """Reusable collector: owns the buffer and scratch tensors so repeated rollouts allocate nothing."""

    def __init__(self, vec: VecMinesweeper, steps: int, aux_maps: bool, sample_seed: int = 0, fused: bool = True,
                 compact: bool = False, graph: bool = False):
        if vec.api != "torch":
            raise ValueError("RolloutCollector needs VecMinesweeper(api='torch')")
        self.vec, self.steps, self.aux_maps = vec, int(steps), bool(aux_maps)
        N, dev = vec.num_envs, vec.device
        vec.aux_maps = self.aux_maps
        self.compact = bool(compact)
        if self.compact:      # SURVEY 8 f2: transitions stored as bitboards, two dense scratch slots for the forward
            self.buffer = CompactRolloutBuffer(vec, self.steps, aux_maps=self.aux_maps)
            self._scratch = [vec._alloc_encode(), vec._alloc_encode()]
        else:
            self.buffer = RolloutBuffer(N, self.steps, (vec.obs_channels(), vec.H, vec.W), vec.action_space(), dev,
                                        aux_maps=self.aux_maps)
        self.last = vec._alloc_encode()                       # observation after the final step (bootstrap)
        self.actions32 = torch.empty((N,), dtype=torch.int32, device=dev)
        self.sample_seed = int(sample_seed)
        self.rollouts_done = 0
        self.fused = bool(fused)          # use the hand-written forward (make_rollout_forward) when the model has one
        self._fused_fwd = None
        # graph=True: the WHOLE rollout (reset, T x (forward, sample, step), bootstrap forward, weight
        # refresh) is captured once into a CUDA graph and replayed -- one launch per rollout instead of
        # ~35 per step, which is what matters when N is small and every kernel is launch-bound.  A
        # device-side epoch counter, bumped inside the graph, keeps sampler / dropout draws fresh.
        self.use_graph = bool(graph)
        self._graph = None
        self._graph_aux = None
        self._graph_key_captured = None
        self._epoch = torch.zeros(1, dtype=torch.int32, device=dev) if self.use_graph else None

    def _graph_key(self, model: nn.Module, autocast: bool):
        """Everything the captured graph bakes in besides the tensors it reads: the module object, train / eval
        mode, every Dropout2d probability, whether aux maps are produced, the autocast flag and the env's shape.
        A change re-captures (weights are NOT part of the key: the graph refreshes them in place every replay)."""
        drops = tuple(float(mod.p) for mod in model.modules() if isinstance(mod, (nn.Dropout, nn.Dropout2d)))
        return (id(model), bool(model.training), drops, self.aux_maps, bool(autocast), self.vec.num_envs, self.steps)

    @staticmethod
    def can_graph(model: nn.Module) -> bool:
        """graph=True needs a fused forward: a CNNResidualPolicy with 8 | channels-per-group, or a CNNPolicy with
        <= 16 input planes."""
        return supports_fused(model)

    @torch.no_grad()
    def collect(self, model: nn.Module, autocast: bool = True) -> Tuple[RolloutBuffer, Dict]:
        if not self.use_graph:
            return self._collect(model, autocast)
        if not (self.fused and autocast and supports_fused(model)):
            raise ValueError("graph=True needs the fused forward (CNNResidualPolicy or CNNPolicy, fused=True, CUDA autocast)")
        key = self._graph_key(model, autocast)
        if self._graph is None or self._graph_key_captured != key:
            side = torch.cuda.Stream(device=self.vec.device)
            side.wait_stream(torch.cuda.current_stream(self.vec.device))
            with torch.cuda.stream(side):                       # warm-up outside capture (cuDNN plans, lazy inits)
                self._collect(model, autocast)
            torch.cuda.current_stream(self.vec.device).wait_stream(side)
            torch.cuda.synchronize(self.vec.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._epoch.add_(1)
                _, aux = self._collect(model, autocast)
            self._graph, self._graph_aux, self._graph_key_captured = g, aux, key
        self._graph.replay()
        self.buffer._t = self.steps
        return self.buffer, dict(self._graph_aux)

    def _collect(self, model: nn.Module, autocast: bool = True) -> Tuple[RolloutBuffer, Dict]:
        vec, buf, T = self.vec, self.buffer, self.steps
        N, dev = vec.num_envs, vec.device
        def obs_slot(t):      # where the observation of time t lives (dense buffer slot or scratch)
            return buf.slot(t) if not self.compact else self._scratch[t & 1]

        vec.reset(out=obs_slot(0))                            # train_rl.py:163: every rollout starts fresh
        if self.compact:
            buf.snapshot(0)
        buf._t = 0
        ctx = (lambda: torch.autocast(device_type="cuda", dtype=torch.float16)) if autocast else nullcontext
        base_step = self.rollouts_done * (T + 1)
        fwd = model
        if self.fused and autocast and supports_fused(model):
            if self._fused_fwd is None or self._fused_fwd.model is not model:
                self._fused_fwd = make_rollout_forward(model, seed=self.sample_seed, sample_id_base=vec._desc.env_id_base)
                self._fused_fwd.epoch = self._epoch
            self._fused_fwd.refresh()                         # weights may have been updated since
            fwd, ctx = self._fused_fwd, nullcontext
        for t in range(T):
            cur = obs_slot(t)
            rows = slice(t * N, (t + 1) * N)
            with ctx():                                       # train_rl.py:222-227
                if self.aux_maps:
                    logits, values, _ = fwd(cur.obs, return_mine=True)
                else:
                    logits, values = fwd(cur.obs)
            masked_sample(logits, cur.action_mask, seed=self.sample_seed, step_index=base_step + t,
                          row_id_base=vec._desc.env_id_base, actions64=buf.actions[rows],
                          actions32=self.actions32, logp=buf.logp[rows], epoch=self._epoch)
            buf.values[rows] = values.float()                 # train_rl.py:256
            nxt = obs_slot(t + 1) if t + 1 < T else self.last
            vec.step(self.actions32, out=StepOut(obs=nxt.obs, action_mask=nxt.action_mask, rewards=buf.rewards[rows],
                                                 dones=buf.dones[rows], mine_labels=nxt.mine_labels,
                                                 mine_valid=nxt.mine_valid), want_infos=False)
            if self.compact and t + 1 < T:
                buf.snapshot(t + 1)
        buf._t = T
        with ctx():                                           # bootstrap value, train_rl.py:267-277
            if self.aux_maps:
                _, last_values, _ = fwd(self.last.obs, return_mine=True)
            else:
                _, last_values = fwd(self.last.obs)
        self.rollouts_done += 1
        return buf, {"last_values": last_values}


def collect_rollout(vec: VecMinesweeper, model: nn.Module, steps: int, device: torch.device,
                    aux_mine_weight: float = 0.0, aux_mine_calib_weight: float = 0.0,
                    collector: Optional[RolloutCollector] = None) -> Tuple[RolloutBuffer, Dict]:
    """Signature and return structure of train_rl.py:155-289: (buffer, {"last_values", "timings"}).
    `timings` reports device-side wall time of the whole rollout; the reference's per-bucket host
    timers (tensor_bridge / mine_label_copy) have nothing left to measure."""
    need_aux = (aux_mine_weight > 0) or (aux_mine_calib_weight > 0)       # train_rl.py:175-177
    if collector is None:
        collector = RolloutCollector(vec, steps, need_aux)
    t0 = time.perf_counter()
    buf, aux = collector.collect(model, autocast=torch.device(device).type == "cuda")
    torch.cuda.synchronize(vec.device)
    dt = time.perf_counter() - t0
    aux["timings"] = {
        "steps": steps, "rollout_total_s": dt, "rollout_per_step_ms": (dt / steps) * 1e3 if steps else 0.0,
        "tensor_bridge_total_s": 0.0, "mine_label_copy_total_s": 0.0,
    }
    return buf, aux
