"""Inference-only rollout forwards: `FusedRolloutForward` for `CNNResidualPolicy` and `FusedCnnForward` for the
three-convolution baseline `CNNPolicy` (build_model("cnn")); `make_rollout_forward` picks one.

`FusedRolloutForward` (SURVEY section 8, row f4): at the medium
config's shape (96 channels) and the package's default shape (128 channels) every convolution is a tcgen05 kernel with GroupNorm / ReLU / Dropout2d / the fp32 residual add
fused into its epilogue (msw_conv3x3_gn); other shapes use fp16 NHWC library convolutions with ONE fused kernel
(msw_gn_act) between them instead of the eager GroupNorm / ReLU / Dropout2d / residual-add / dtype-cast kernels.

Numerics follow the reference's fp16-autocast forward (train_rl.py:222-227 over
cnn_residual.py:83-96): convolutions and linears in fp16, GroupNorm statistics and arithmetic in
fp32, residual stream in fp32, activations rounded to fp16 exactly where autocast rounds them (at
the next convolution's input).  Dropout2d uses the package's counter-based RNG, not torch's stream.
The parameters are read from the live module, so training and rollouts share one set of weights.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
import torch.nn.functional as F

from . import _lib
from .policy import CNNPolicy, CNNResidualPolicy


def gn_act(x16: torch.Tensor, norm: torch.nn.GroupNorm, *, conv_bias: Optional[torch.Tensor] = None,
           res32: Optional[torch.Tensor] = None, relu: bool = True,
           drop_p: float = 0.0, want16: bool = True, want32: bool = False, seed: int = 0, call_id: int = 0,
           epoch: Optional[torch.Tensor] = None, pool32: Optional[torch.Tensor] = None, sample_id_base: int = 0
           ) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """x16: fp16 [N,C,H,W] in channels_last memory format (conv output, bias NOT applied when
    `conv_bias` -- fp32 [C] -- is given).  Returns (y16, y32) with the same logical shape / memory format;
    `pool32` (fp32 [N,C], optional) receives the spatial mean of the fp32 output."""
    L = _lib.load()
    if x16.dtype != torch.float16 or not x16.is_contiguous(memory_format=torch.channels_last):
        raise ValueError("gn_act: x must be fp16 channels_last")
    N, C, H, W = x16.shape
    dev = x16.device
    y16 = torch.empty_like(x16, memory_format=torch.channels_last) if want16 else None
    y32 = (torch.empty((N, C, H, W), dtype=torch.float32, device=dev, memory_format=torch.channels_last)
           if want32 else None)
    if pool32 is not None and (pool32.dtype != torch.float32 or tuple(pool32.shape) != (N, C) or not pool32.is_contiguous()):
        raise ValueError("gn_act: pool32 must be contiguous fp32 [N, C]")
    if res32 is not None and (res32.dtype != torch.float32 or tuple(res32.shape) != (N, C, H, W)
                              or not res32.is_contiguous(memory_format=torch.channels_last)):
        raise ValueError("gn_act: residual must be fp32 channels_last of the same shape")
    with torch.cuda.device(dev):
        rc = L.msw_gn_act(x16.data_ptr(), None if conv_bias is None else conv_bias.data_ptr(),
                          None if res32 is None else res32.data_ptr(), norm.weight.data_ptr(),
                          norm.bias.data_ptr(), None if y16 is None else y16.data_ptr(),
                          None if y32 is None else y32.data_ptr(), N, H * W, C, norm.num_groups, float(norm.eps),
                          int(relu), float(drop_p), int(seed) & 0xFFFFFFFFFFFFFFFF, int(call_id) & 0xFFFFFFFFFFFFFFFF,
                          None if epoch is None else epoch.data_ptr(), None, None, None,
                          None if pool32 is None else pool32.data_ptr(), int(sample_id_base),
                          torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "msw_gn_act")
    return y16, y32


def cell_heads(rows16: torch.Tensor, w1: torch.Tensor, b1: torch.Tensor, w2: torch.Tensor, b2: torch.Tensor
               ) -> Tuple[torch.Tensor, torch.Tensor]:
    """msw_cell_heads: rows16 fp16 [R, C] (NHWC activation viewed as rows) -> (policy logit, mine logit),
    fp16 [R] each; w1 [2C, C], b1 [2C], w2 [2C], b2 [2] fp16."""
    L = _lib.load()
    R, C = rows16.shape
    if rows16.dtype != torch.float16 or not rows16.is_contiguous():
        raise ValueError("cell_heads: rows must be contiguous fp16 [R, C]")
    dev = rows16.device
    out = torch.empty((2, R), dtype=torch.float16, device=dev)
    with torch.cuda.device(dev):
        rc = L.msw_cell_heads(rows16.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                              out[0].data_ptr(), out[1].data_ptr(), R, C, torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "msw_cell_heads")
    return out[0], out[1]


def conv3x3_taps(weight: torch.Tensor) -> torch.Tensor:
    """Conv2d weight [C_out, C_in, 3, 3] -> the fp16 [9, C_out, C_in] tap-major layout msw_conv3x3 reads."""
    co, ci = weight.shape[0], weight.shape[1]
    return weight.detach().permute(2, 3, 0, 1).to(torch.float16).reshape(9, co, ci).contiguous()


def conv3x3(x16: torch.Tensor, taps16: torch.Tensor) -> torch.Tensor:
    """msw_conv3x3: x16 fp16 [N,C,16,16] channels_last, taps16 from `conv3x3_taps` -> fp16 conv output
    (no bias), same shape / memory format."""
    L = _lib.load()
    N, Cin, H, W = x16.shape
    if x16.dtype != torch.float16 or not x16.is_contiguous(memory_format=torch.channels_last):
        raise ValueError("conv3x3: x must be fp16 channels_last")
    if taps16.dtype != torch.float16 or taps16.dim() != 3 or taps16.shape[0] != 9 or taps16.shape[2] != Cin or not taps16.is_contiguous():
        raise ValueError("conv3x3: taps must be contiguous fp16 [9, C_out, C_in]")
    C = taps16.shape[1]
    y = torch.empty((N, C, H, W), dtype=torch.float16, device=x16.device, memory_format=torch.channels_last)
    with torch.cuda.device(x16.device):
        rc = L.msw_conv3x3(x16.data_ptr(), taps16.data_ptr(), y.data_ptr(), N, H, W, Cin, C,
                           torch.cuda.current_stream(x16.device).cuda_stream)
    _lib.check(rc, "msw_conv3x3")
    return y


def to_p8(x: torch.Tensor) -> torch.Tensor:
    """fp32 [N, C, 16, 16] (C = 96 or 128, any memory format) -> the private "P8" order of the fused trunk's
    residual stream: [N][tile 2][32-channel slice C/32][8-channel chunk 4][pixel 128][8] (msw_conv_tc.cu; the
    slices are the epilogue's warpgroups).  Test / tooling helper."""
    n, c, h, w = x.shape
    assert c in (96, 128) and (h, w) == (16, 16)
    t = x.permute(0, 2, 3, 1).reshape(n, 2, 128, c // 32, 4, 8)    # [N][tile][pixel][slice][chunk][8]
    return t.permute(0, 1, 3, 4, 2, 5).contiguous()


def from_p8(t: torch.Tensor) -> torch.Tensor:
    """Inverse of `to_p8`: -> fp32 [N, C, 16, 16] (channels_last storage); C from the tensor's size."""
    n = t.shape[0]
    c = t.numel() // (n * 256)
    x = t.reshape(n, 2, c // 32, 4, 128, 8).permute(0, 1, 4, 2, 3, 5).reshape(n, 16, 16, c)
    return x.permute(0, 3, 1, 2)


def conv3x3_gn(x16: torch.Tensor, taps16: torch.Tensor, norm: torch.nn.GroupNorm, conv_bias: torch.Tensor, *,
               res32: Optional[torch.Tensor] = None, drop_p: float = 0.0, want32: bool = False, want_pool: bool = False,
               seed: int = 0, call_id: int = 0, epoch: Optional[torch.Tensor] = None,
               sample_id_base: int = 0) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """msw_conv3x3_gn: relu(GroupNorm(conv3x3(x16) + bias) [+ res32]) [* Dropout2d] in one launch.
    `res32` and the fp32 output are in the P8 order (`to_p8`); with `want_pool` the second result is instead
    the spatial mean of the fp32 output, fp32 [N, C] (the value head's AdaptiveAvgPool2d(1))."""
    L = _lib.load()
    N, Cin, H, W = x16.shape
    if x16.dtype != torch.float16 or not x16.is_contiguous(memory_format=torch.channels_last):
        raise ValueError("conv3x3_gn: x must be fp16 channels_last")
    if taps16.dtype != torch.float16 or taps16.dim() != 3 or taps16.shape[0] != 9 or taps16.shape[2] != Cin or not taps16.is_contiguous():
        raise ValueError("conv3x3_gn: taps must be contiguous fp16 [9, C_out, C_in]")
    C = taps16.shape[1]
    if res32 is not None and (res32.dtype != torch.float32 or res32.numel() != N * C * H * W or not res32.is_contiguous()):
        raise ValueError("conv3x3_gn: residual must be a contiguous fp32 tensor in P8 order")
    dev = x16.device
    y16 = torch.empty((N, C, H, W), dtype=torch.float16, device=dev, memory_format=torch.channels_last)
    y32 = torch.empty((N, 2, C // 32, 4, 128, 8), dtype=torch.float32, device=dev) if (want32 and not want_pool) else None
    # pooled partial sums: per row quarter (C = 96: one CTA per board), per tile and row quarter (C = 128: a CTA pair)
    pool4 = torch.empty((N, 8 if C == 128 else 4, C), dtype=torch.float32, device=dev) if want_pool else None
    with torch.cuda.device(dev):
        rc = L.msw_conv3x3_gn(x16.data_ptr(), taps16.data_ptr(), conv_bias.data_ptr(),
                              None if res32 is None else res32.data_ptr(), norm.weight.data_ptr(), norm.bias.data_ptr(),
                              y16.data_ptr(), None if y32 is None else y32.data_ptr(),
                              None if pool4 is None else pool4.data_ptr(), N, H, W, Cin, C, norm.num_groups,
                              float(norm.eps), float(drop_p), int(seed) & 0xFFFFFFFFFFFFFFFF,
                              int(call_id) & 0xFFFFFFFFFFFFFFFF, None if epoch is None else epoch.data_ptr(),
                              int(sample_id_base), torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "msw_conv3x3_gn")
    if want_pool:
        return y16, pool4.sum(dim=1) * (1.0 / (H * W))
    return y16, y32


class FusedRolloutForward:
    """Callable with the module's `(obs, return_mine)` signature, for use under torch.no_grad().

    Two shape classes, chosen once at construction (no run-time switches):
      * the medium config's shape (96 channels, 6 groups) and the package's default shape (128 channels, 8 groups;
        each convolution on a CTA pair), on 16x16 boards with <= 16 observation planes: every convolution runs on tcgen05 with GroupNorm / ReLU / Dropout2d / the fp32 residual add / the value head's
        average pool fused into its epilogue (msw_pack_obs16 -> 11 x msw_conv3x3_gn -> msw_cell_heads); the fp32
        residual stream lives in the kernels' private P8 order and no library convolution is on the path;
      * any other CNNResidualPolicy shape: library (cuDNN) fp16 NHWC convolutions with the fused GroupNorm kernel
        (msw_gn_act) between them.  Announced once, loudly, on stderr -- it is a different, slower path."""

    _warned = set()

    def __init__(self, model: CNNResidualPolicy, seed: int = 0, sample_id_base: int = 0):
        if not isinstance(model, CNNResidualPolicy):
            raise TypeError("FusedRolloutForward supports CNNResidualPolicy only")
        C = model.stem[0].out_channels
        G = model.stem[1].num_groups
        if C % 8 or (C // G) % 8:
            raise ValueError(f"fused forward needs C % 8 == 0 and (C/G) % 8 == 0, got C={C} G={G}")
        self.model, self.seed, self.calls = model, int(seed), 0
        self.sample_id_base = int(sample_id_base)     # global index of row 0 (env shard offset): keys the Dropout2d stream
        self.epoch: Optional[torch.Tensor] = None     # device uint32 counter mixed into the dropout RNG (graph replays)
        self.tc_trunk = (C, G) in ((96, 6), (128, 8)) and model.stem[0].in_channels <= 16 and len(model.residual_stack) >= 1
        self._w: List = []
        self.refresh()

    @staticmethod
    def supports(model) -> bool:
        if not isinstance(model, CNNResidualPolicy):
            return False
        C, G = model.stem[0].out_channels, model.stem[1].num_groups
        return C % 8 == 0 and (C // G) % 8 == 0

    @torch.no_grad()
    def refresh(self) -> None:
        """Re-cast the (possibly just updated) fp32 parameters into the fp16 copies the convs use.
        The copies are allocated once and updated IN PLACE, so their addresses are stable and the
        whole forward -- including this refresh -- can live inside a captured CUDA graph."""
        m = self.model
        p0, p2, q0, q2 = m.policy_head[0], m.policy_head[2], m.mine_head[0], m.mine_head[2]
        C = p0.out_channels
        if not self._w:
            def conv3(c):    # 3x3 conv: fp16 NHWC weight for the library path; the bias is folded into the GroupNorm step
                return (torch.empty_like(c.weight, dtype=torch.float16, memory_format=torch.channels_last),
                        torch.empty_like(c.bias, dtype=torch.float32))

            def lin(out_f, in_f, dev):
                return (torch.empty((out_f, in_f), dtype=torch.float16, device=dev),
                        torch.empty((out_f,), dtype=torch.float16, device=dev))

            dev = p0.weight.device
            self.stem = conv3(m.stem[0])
            cin = m.stem[0].in_channels
            # stem weight with the input channels padded to 16 (zeros): pairs with msw_pack_obs16
            self.stem16 = (torch.zeros((C, 16, 3, 3), dtype=torch.float16, device=dev).contiguous(memory_format=torch.channels_last)
                           if cin <= 16 else None)
            self.blocks = [(conv3(b.conv1), conv3(b.conv2)) for b in m.residual_stack]
            # tap-major fp16 copies of the weights for msw_conv3x3_gn (tcgen05)
            self.stem_taps = torch.zeros((9, C, 16), dtype=torch.float16, device=dev) if self.tc_trunk else None
            self.taps = ([(torch.empty((9, C, C), dtype=torch.float16, device=dev),
                           torch.empty((9, C, C), dtype=torch.float16, device=dev)) for _ in m.residual_stack]
                         if self.tc_trunk else None)
            # the two per-cell heads (1x1 -> ReLU -> 1x1) are row-wise linears on the NHWC activation:
            # one msw_cell_heads launch, the hidden layer never reaches HBM
            self.head1 = lin(2 * C, C, dev)
            self.head2 = (torch.empty((2 * C,), dtype=torch.float16, device=dev),       # policy w2 | mine w2
                          torch.empty((2,), dtype=torch.float16, device=dev))
            self.value = [lin(m.value_head[i].out_features, m.value_head[i].in_features, dev) for i in (2, 4, 6)]
            self._w = [self.stem]

        def put3(dst, c):
            dst[0].copy_(c.weight)
            dst[1].copy_(c.bias)

        put3(self.stem, m.stem[0])
        if self.stem16 is not None:
            self.stem16[:, :m.stem[0].in_channels].copy_(m.stem[0].weight)
        if self.stem_taps is not None:
            self.stem_taps[:, :, :m.stem[0].in_channels].copy_(m.stem[0].weight.permute(2, 3, 0, 1).reshape(9, C, -1))
        for (d1, d2), b in zip(self.blocks, m.residual_stack):
            put3(d1, b.conv1)
            put3(d2, b.conv2)
        if self.taps is not None:
            for (t1, t2), b in zip(self.taps, m.residual_stack):
                t1.copy_(b.conv1.weight.permute(2, 3, 0, 1).reshape(9, C, C))
                t2.copy_(b.conv2.weight.permute(2, 3, 0, 1).reshape(9, C, C))
        self.head1[0][:C].copy_(p0.weight.reshape(C, C)); self.head1[0][C:].copy_(q0.weight.reshape(C, C))
        self.head1[1][:C].copy_(p0.bias); self.head1[1][C:].copy_(q0.bias)
        self.head2[0][:C].copy_(p2.weight.reshape(-1)); self.head2[0][C:].copy_(q2.weight.reshape(-1))
        self.head2[1][0:1].copy_(p2.bias); self.head2[1][1:2].copy_(q2.bias)
        for dst, i in zip(self.value, (2, 4, 6)):
            dst[0].copy_(m.value_head[i].weight)
            dst[1].copy_(m.value_head[i].bias)

    def _drop_p(self, blk) -> float:
        return float(blk.dropout.p) if (self.model.training and isinstance(blk.dropout, torch.nn.Dropout2d)) else 0.0

    def _trunk_tc(self, obs: torch.Tensor, cid: int):
        """tcgen05 shapes: 1 + 2 * blocks msw_conv3x3_gn launches; returns (a16 NHWC, pooled fp32 [N, C])."""
        m = self.model
        base = self.sample_id_base
        nb, cin, hh, ww = obs.shape
        x = torch.empty((nb, 16, hh, ww), dtype=torch.float16, device=obs.device, memory_format=torch.channels_last)
        with torch.cuda.device(obs.device):
            _lib.check(_lib.load().msw_pack_obs16(obs.data_ptr(), x.data_ptr(), nb, cin, hh * ww,
                                                  torch.cuda.current_stream(obs.device).cuda_stream), "msw_pack_obs16")
        a16, a32 = conv3x3_gn(x, self.stem_taps, m.stem[1], self.stem[1], want32=True)   # stem conv + GN + ReLU
        last = len(self.blocks) - 1
        pooled = None
        for k, (blk, ((_, b1), (_, b2))) in enumerate(zip(m.residual_stack, self.blocks)):
            # conv1 + GroupNorm + ReLU + Dropout2d
            t16, _ = conv3x3_gn(a16, self.taps[k][0], blk.norm1, b1, drop_p=self._drop_p(blk), seed=self.seed,
                                call_id=cid + k, epoch=self.epoch, sample_id_base=base)
            # conv2 + GroupNorm + fp32 residual add + ReLU; the last block emits the value head's average pool
            # instead of a residual stream nobody reads
            if k == last:
                a16, pooled = conv3x3_gn(t16, self.taps[k][1], blk.norm2, b2, res32=a32, want_pool=True)
            else:
                a16, a32 = conv3x3_gn(t16, self.taps[k][1], blk.norm2, b2, res32=a32, want32=True)
        return a16, pooled

    def _heads(self, a16: torch.Tensor, pooled: torch.Tensor, return_mine: bool):
        n, c, h, w = a16.shape
        rows = a16.permute(0, 2, 3, 1).reshape(n * h * w, c)         # NHWC storage: a view, no copy
        if c in (32, 64, 96, 128):
            pol, mine = cell_heads(rows, self.head1[0], self.head1[1], self.head2[0], self.head2[1])
        else:                                                        # other widths: the same math as library GEMMs
            hid = F.relu_(F.linear(rows, *self.head1))               # [n*h*w, 2C]
            pol = F.linear(hid[:, :c], self.head2[0][None, :c], self.head2[1][0:1]).squeeze(-1)
            mine = F.linear(hid[:, c:], self.head2[0][None, c:], self.head2[1][1:2]).squeeze(-1)
        logits = pol.reshape(n, h * w)
        v = F.relu_(F.linear(pooled.to(torch.float16), *self.value[0]))
        v = F.relu_(F.linear(v, *self.value[1]))
        value = F.linear(v, *self.value[2]).squeeze(-1)
        if not return_mine:
            return logits, value
        return logits, value, mine.reshape(n, 1, h, w)

    def _trunk_library(self, obs: torch.Tensor, cid: int):
        """Any other shape: cuDNN fp16 NHWC convolutions with msw_gn_act between them."""
        m = self.model
        key = (m.stem[0].out_channels, m.stem[1].num_groups, tuple(obs.shape[1:]))
        if key not in FusedRolloutForward._warned:
            FusedRolloutForward._warned.add(key)
            import sys
            print(f"[minesweeper_ppo_b200] FusedRolloutForward: shape C={key[0]} G={key[1]} obs={key[2]} is outside the "
                  "tcgen05 trunk (96 channels and 6 groups or 128 channels and 8 groups, 16x16 boards): convolutions "
                  "run in cuDNN with the fused GroupNorm kernel between them", file=sys.stderr, flush=True)
        if self.stem16 is not None and obs.dtype == torch.float32 and obs.is_contiguous():
            nb, cin, hh, ww = obs.shape
            x = torch.empty((nb, 16, hh, ww), dtype=torch.float16, device=obs.device, memory_format=torch.channels_last)
            with torch.cuda.device(obs.device):
                _lib.check(_lib.load().msw_pack_obs16(obs.data_ptr(), x.data_ptr(), nb, cin, hh * ww,
                                                      torch.cuda.current_stream(obs.device).cuda_stream), "msw_pack_obs16")
            c0 = F.conv2d(x, self.stem16, None, padding=1)
        else:
            c0 = F.conv2d(obs.to(dtype=torch.float16, memory_format=torch.channels_last), self.stem[0], None, padding=1)
        a16, a32 = gn_act(c0, m.stem[1], conv_bias=self.stem[1], want32=True)
        last = len(self.blocks) - 1
        pooled = None
        for k, (blk, ((w1, b1), (w2, b2))) in enumerate(zip(m.residual_stack, self.blocks)):
            c1 = F.conv2d(a16, w1, None, padding=1)
            t16, _ = gn_act(c1, blk.norm1, conv_bias=b1, drop_p=self._drop_p(blk), seed=self.seed, call_id=cid + k,
                            epoch=self.epoch, sample_id_base=self.sample_id_base)
            if k == last:        # nothing reads the residual stream after the last block except the value head's pool
                pooled = torch.empty((a16.shape[0], a16.shape[1]), dtype=torch.float32, device=a16.device)
            c2 = F.conv2d(t16, w2, None, padding=1)
            a16, a32 = gn_act(c2, blk.norm2, conv_bias=b2, res32=a32, want32=k != last, pool32=pooled)
        if pooled is None:                                           # no residual blocks
            pooled = a32.mean(dim=(2, 3))                            # AdaptiveAvgPool2d(1) in fp32
        return a16, pooled

    @torch.no_grad()
    def __call__(self, obs: torch.Tensor, return_mine: bool = False):
        self.calls += 1
        cid = self.calls << 8
        if (self.tc_trunk and tuple(obs.shape[2:]) == (16, 16) and obs.dtype == torch.float32 and obs.is_contiguous()):
            a16, pooled = self._trunk_tc(obs, cid)
        else:
            a16, pooled = self._trunk_library(obs, cid)
        return self._heads(a16, pooled, return_mine)


def cnn_forward(x16: torch.Tensor, taps: Tuple[torch.Tensor, torch.Tensor, torch.Tensor], vecs: Tuple[torch.Tensor, ...],
                heads16: torch.Tensor, head_bias16: torch.Tensor, eps: Tuple[float, float]
                ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """msw_cnn_forward: x16 fp16 [N, 16, 16, 16] channels_last (msw_pack_obs16's layout); taps = the fp16 tap-major
    weights [9, 32, 16], [9, 64, 32], [9, 64, 64]; vecs = fp32 (b1, gamma1, beta1, b2, gamma2, beta2, b3);
    heads16 fp16 [2, 64] (policy, mine weights), head_bias16 fp16 [2].  Returns fp16 (logits [N, 256],
    mine [N, 256], pooled [N, 64])."""
    L = _lib.load()
    N, cin, H, W = x16.shape
    if x16.dtype != torch.float16 or not x16.is_contiguous(memory_format=torch.channels_last):
        raise ValueError("cnn_forward: x must be fp16 channels_last")
    dev = x16.device
    logits = torch.empty((N, H * W), dtype=torch.float16, device=dev)
    mine = torch.empty((N, H * W), dtype=torch.float16, device=dev)
    pooled = torch.empty((N, taps[2].shape[1]), dtype=torch.float16, device=dev)
    b1, g1, be1, b2, g2, be2, b3 = vecs
    with torch.cuda.device(dev):
        rc = L.msw_cnn_forward(x16.data_ptr(), taps[0].data_ptr(), b1.data_ptr(), g1.data_ptr(), be1.data_ptr(),
                               taps[1].data_ptr(), b2.data_ptr(), g2.data_ptr(), be2.data_ptr(), taps[2].data_ptr(),
                               b3.data_ptr(), heads16[0].data_ptr(), head_bias16[0:1].data_ptr(), heads16[1].data_ptr(),
                               head_bias16[1:2].data_ptr(), logits.data_ptr(), mine.data_ptr(), pooled.data_ptr(), N, H, W,
                               cin, taps[0].shape[1], 4, taps[1].shape[1], 8, taps[2].shape[1], float(eps[0]),
                               float(eps[1]), torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "msw_cnn_forward")
    return logits, mine, pooled


class FusedCnnForward:
    """Rollout forward of the three-convolution baseline `CNNPolicy` (build_model("cnn")), with the module's
    `(obs, return_mine)` signature, for use under torch.no_grad().

    On 16x16 boards with <= 16 observation planes (fp32, contiguous) the whole network up to the value MLP is one
    msw_cnn_forward launch after msw_pack_obs16: the three convolutions, both GroupNorms, the 1x1 policy / mine heads
    and the average pool, with the roundings of the fp16 autocast forward.  The value MLP (Linear -> ReLU -> Linear)
    runs in torch fp16 on the pooled features.  Any other input runs the module itself under fp16 autocast.

    The fp16 / fp32 parameter copies are allocated once and updated in place by `refresh()`, so their addresses are
    stable and the forward can be captured in a CUDA graph.  Conv and head biases are rounded to fp16 first, as
    autocast casts them.  `epoch` and `sample_id_base` are set by the collector like on `FusedRolloutForward`;
    this network has no dropout, so nothing reads them."""

    def __init__(self, model: CNNPolicy, seed: int = 0, sample_id_base: int = 0):
        if not isinstance(model, CNNPolicy):
            raise TypeError("FusedCnnForward supports CNNPolicy only")
        self.model, self.seed = model, int(seed)
        self.sample_id_base = int(sample_id_base)
        self.epoch: Optional[torch.Tensor] = None
        self.cin = model.backbone[0].in_channels
        self._w = None
        self.refresh()

    @staticmethod
    def supports(model) -> bool:
        return isinstance(model, CNNPolicy) and model.backbone[0].in_channels <= 16

    @torch.no_grad()
    def refresh(self) -> None:
        m = self.model
        conv = (m.backbone[0], m.backbone[3], m.backbone[6])
        norm = (m.backbone[2], m.backbone[5])
        if self._w is None:
            dev = conv[0].weight.device
            self.taps = tuple(torch.zeros((9, c.out_channels, 16 if k == 0 else c.in_channels), dtype=torch.float16, device=dev)
                              for k, c in enumerate(conv))
            self.vecs = tuple(torch.empty((n,), dtype=torch.float32, device=dev) for n in (32, 32, 32, 64, 64, 64, 64))
            self.heads16 = torch.empty((2, 64), dtype=torch.float16, device=dev)
            self.head_bias16 = torch.empty((2,), dtype=torch.float16, device=dev)
            v1, v2 = m.value_head[2], m.value_head[4]
            self.value = [(torch.empty_like(l.weight, dtype=torch.float16), torch.empty_like(l.bias, dtype=torch.float16))
                          for l in (v1, v2)]
            self._w = True
        for t, c in zip(self.taps, conv):
            t[:, :, :c.in_channels].copy_(c.weight.permute(2, 3, 0, 1).reshape(9, c.out_channels, c.in_channels))
        b1, g1, be1, b2, g2, be2, b3 = self.vecs
        for dst, c in ((b1, conv[0]), (b2, conv[1]), (b3, conv[2])):
            dst.copy_(c.bias.to(torch.float16))
        g1.copy_(norm[0].weight); be1.copy_(norm[0].bias)
        g2.copy_(norm[1].weight); be2.copy_(norm[1].bias)
        self.heads16[0].copy_(m.policy_head.weight.reshape(-1)); self.heads16[1].copy_(m.mine_head.weight.reshape(-1))
        self.head_bias16[0:1].copy_(m.policy_head.bias); self.head_bias16[1:2].copy_(m.mine_head.bias)
        for (w, b), l in zip(self.value, (m.value_head[2], m.value_head[4])):
            w.copy_(l.weight)
            b.copy_(l.bias)

    def fused_input(self, obs: torch.Tensor) -> bool:
        return (obs.is_cuda and obs.dim() == 4 and obs.dtype == torch.float32 and obs.is_contiguous()
                and obs.shape[1] == self.cin and tuple(obs.shape[2:]) == (16, 16))

    @torch.no_grad()
    def __call__(self, obs: torch.Tensor, return_mine: bool = False):
        if not self.fused_input(obs):
            with torch.autocast("cuda", dtype=torch.float16):
                return self.model(obs, return_mine=return_mine)
        nb, cin, hh, ww = obs.shape
        x = torch.empty((nb, 16, hh, ww), dtype=torch.float16, device=obs.device, memory_format=torch.channels_last)
        with torch.cuda.device(obs.device):
            _lib.check(_lib.load().msw_pack_obs16(obs.data_ptr(), x.data_ptr(), nb, cin, hh * ww,
                                                  torch.cuda.current_stream(obs.device).cuda_stream), "msw_pack_obs16")
        norm = (self.model.backbone[2], self.model.backbone[5])
        logits, mine, pooled = cnn_forward(x, self.taps, self.vecs, self.heads16, self.head_bias16,
                                           (norm[0].eps, norm[1].eps))
        v = F.relu_(F.linear(pooled, *self.value[0]))
        value = F.linear(v, *self.value[1]).squeeze(-1)
        if not return_mine:
            return logits, value
        return logits, value, mine.reshape(nb, 1, hh, ww)


def supports_fused(model) -> bool:
    """True when `make_rollout_forward` has a hand-written forward for `model` (the collector's fused path and
    graph capture)."""
    return FusedRolloutForward.supports(model) or FusedCnnForward.supports(model)


def make_rollout_forward(model, seed: int = 0, sample_id_base: int = 0):
    """The rollout forward for `model`: FusedCnnForward for a CNNPolicy, FusedRolloutForward otherwise."""
    if isinstance(model, CNNPolicy):
        return FusedCnnForward(model, seed=seed, sample_id_base=sample_id_base)
    return FusedRolloutForward(model, seed=seed, sample_id_base=sample_id_base)
