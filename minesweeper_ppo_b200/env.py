"""Device-resident vectorised Minesweeper environment with the reference's API.

Mirrors `minesweeper/env.py` of yakvrz/minesweeper-ppo for the rollout hot path:

    EnvConfig                      env.py:19-30
    VecMinesweeper(num_envs, cfg, seed=0, late_start_cfg=None, late_start_seed=None)
                                   env.py:382-403
      .reset() -> {"obs","action_mask"}                         env.py:468-477
      .step(actions) -> (batch, rewards, dones, infos)          env.py:479-511
      .envs[i].{revealed,flags,mine_mask,adjacent_counts,first_click_done,step_count,H,W,cfg}
                                   env.py:68-75 (read-only views, unpacked lazily)
      .num_envs, .cfg, .action_space(), .obs_channels()         env.py:391-392, 513-517

All state lives in HBM as bitboards and every call is one CUDA launch through the
C ABI of include/msw_b200.h.  Two calling conventions, chosen at construction:

  api="numpy"  (default -- what the reference's callers expect): NumPy in, NumPy
               out, list-of-dict `infos`; each call copies through pinned host
               memory (msw_step_host).
  api="torch"  native: CUDA tensors in and out, tensor-valued infos, optional
               `out=` buffers so the kernel writes straight into a rollout buffer.

There is no CPU implementation in this package: without the CUDA library / a CUDA
device the constructor raises.
"""
from __future__ import annotations

import ctypes as C
import os
from collections.abc import Sequence
from dataclasses import dataclass
from typing import Any, Dict, Optional, Tuple, Union

import numpy as np
import torch

from . import _lib

OBS_CHANNELS = _lib.OBS_CHANNELS
_OUTCOME_NAMES = (None, "win", "loss")
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
try:
    _libc = C.CDLL(None, use_errno=True)
    _libc.madvise
except Exception:                                             # pragma: no cover
    _libc = None


@dataclass
class EnvConfig:
    """Same fields and defaults as the reference EnvConfig (env.py:19-30)."""
    H: int = 8
    W: int = 8
    mine_count: int = 10
    guarantee_safe_neighborhood: bool = True
    use_pair_constraints: Optional[bool] = None  # deprecated in the reference, unused
    solver_preset: str = "zf"

    win_reward: float = 1.0
    loss_reward: float = -1.0
    step_penalty: float = 1e-4


def reward_constants(cfg) -> Tuple[np.float32, np.float32, np.float32]:
    """(step, loss, win) rewards rounded exactly as the reference does: accumulated in
    Python float64 (env.py:110,128,137,142) and stored into a float32 array (env.py:501)."""
    pen = float(cfg.step_penalty)
    step = np.float32(0.0 - pen)
    loss = np.float32((0.0 + float(cfg.loss_reward)) - pen)
    win = np.float32((0.0 + float(cfg.win_reward)) - pen)
    return step, loss, win


def pack_boards(cells: np.ndarray, HW: int) -> np.ndarray:
    """bool [n, HW] (or [n,H,W]) -> int32 [n, wpb] flat little-endian bitboards."""
    cells = np.asarray(cells).reshape(-1, HW).astype(np.uint8)
    wpb = (HW + 31) // 32
    packed = np.packbits(cells, axis=1, bitorder="little")
    out = np.zeros((cells.shape[0], wpb * 4), np.uint8)
    out[:, : packed.shape[1]] = packed
    return out.view("<u4").view(np.int32).reshape(cells.shape[0], wpb)


@dataclass
class StepOut:
    """Caller-owned destination tensors for `step(..., out=)` / `reset(out=)` (CUDA,
    contiguous).  Any of the optional members may be None."""
    obs: torch.Tensor                       # f32 [n,10,H,W]
    action_mask: torch.Tensor               # bool [n,HW]
    rewards: Optional[torch.Tensor] = None  # f32 [n]
    dones: Optional[torch.Tensor] = None    # bool [n]
    mine_labels: Optional[torch.Tensor] = None   # f32 [n,H,W]
    mine_valid: Optional[torch.Tensor] = None    # bool [n,H,W]


class _EnvView:
    """Read-only stand-in for `vec.envs[i]` (MinesweeperEnv attributes, env.py:41-75)."""

    def __init__(self, vec: "VecMinesweeper", i: int):
        self._vec, self._i = vec, i
        self.cfg = vec.cfg
        self.H, self.W = vec.H, vec.W
        self.cell_count = self.reveal_count = self.A = vec.HW

    def _cells(self, key: str) -> np.ndarray:
        return self._vec._unpacked()[key][self._i].reshape(self.H, self.W)

    @property
    def mine_mask(self) -> np.ndarray: return self._cells("mine").view(bool)
    @property
    def revealed(self) -> np.ndarray: return self._cells("revealed").view(bool)
    @property
    def flags(self) -> np.ndarray: return self._cells("flags").view(bool)
    @property
    def adjacent_counts(self) -> np.ndarray: return self._cells("counts")
    @property
    def first_click_done(self) -> bool: return bool(self._vec._unpacked()["meta"][self._i, 0])
    @property
    def step_count(self) -> int: return int(self._vec._unpacked()["meta"][self._i, 1])
    @property
    def _last_new_reveals(self) -> int: return int(self._vec._unpacked()["meta"][self._i, 3])
    @property
    def action_space(self) -> int: return self.A                  # env.py:154-156 (property)
    @property
    def obs_channels(self) -> int: return OBS_CHANNELS            # env.py:158-160 (property)


class _EnvList:
    def __init__(self, vec: "VecMinesweeper"):
        self._vec = vec

    def __len__(self) -> int: return self._vec.num_envs

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        return _EnvView(self._vec, i)

    def __iter__(self):
        return (self[i] for i in range(len(self)))


def _fastest_pinned(nbytes: int, dev_buf: torch.Tensor, to_host: bool, tries: int = 6) -> torch.Tensor:
    """A pinned uint8 [nbytes] buffer for the small per-step DMAs of msw_step_host.  Where a pinned allocation lands in
    host-physical memory decides how long a 256 KB DMA takes (17 us or 35 us for different 256 KB pieces of one
    allocation on the GPU boxes, stable over time: profiles/r02aj_pinned_probe.txt), and these buffers are on the
    critical path of every step, so `tries` candidates are allocated, one DMA is timed on each, and the fastest is kept
    (about a millisecond, once per env)."""
    import time
    if nbytes == 0 or tries <= 1:
        return torch.empty((nbytes,), dtype=torch.uint8).pin_memory()
    cands = [torch.empty((nbytes,), dtype=torch.uint8).pin_memory() for _ in range(tries)]
    stream = torch.cuda.current_stream(dev_buf.device)
    best, best_t = cands[0], float("inf")
    for c in cands:
        t = float("inf")
        for rep in range(4):
            stream.synchronize()
            t0 = time.perf_counter()
            if to_host:
                c.copy_(dev_buf, non_blocking=True)
            else:
                dev_buf.copy_(c, non_blocking=True)
            stream.synchronize()
            if rep:                                   # the first copy of a buffer warms its translations
                t = min(t, time.perf_counter() - t0)
        if t < best_t:
            best, best_t = c, t
    return best


class _LazyList(Sequence):
    """A read-only list whose items are made on access (the per-env `infos` lists of VecMinesweeper.step,
    env.py:485-505).  Compares equal to the list / tuple / sequence with the same items."""
    __slots__ = ("_n", "_item")

    def __init__(self, n: int, item):
        self._n, self._item = int(n), item

    def __len__(self) -> int:
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self._item(k) for k in range(*i.indices(self._n))]
        i = int(i)
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError("list index out of range")
        return self._item(i)

    def __iter__(self):
        return (self._item(k) for k in range(self._n))

    def __eq__(self, other):
        if not isinstance(other, (list, tuple, Sequence)) or isinstance(other, (str, bytes)):
            return NotImplemented
        return len(other) == self._n and all(a == b for a, b in zip(self, other))

    __hash__ = None

    def __repr__(self) -> str:
        return repr(list(self))

    def __reduce__(self):                    # pickles (and copies) as the plain list it stands for
        return (list, (list(self),))


def _madvise_hugepage(a: np.ndarray) -> None:
    """MADV_HUGEPAGE on the page-aligned interior of a large array (best effort; 2-3 % on the delta expansion where
    transparent huge pages are in `madvise` mode, profiles/r02s_host_obs_probe.txt)."""
    if a.nbytes < (4 << 20):
        return
    try:
        lo = (a.ctypes.data + 4095) & ~4095
        ln = (a.ctypes.data + a.nbytes - lo) & ~4095
        if _libc is not None and ln > 0:
            _libc.madvise(C.c_void_p(lo), C.c_size_t(ln), 14)             # MADV_HUGEPAGE
    except Exception:
        pass


class _ResultSet:
    """One recycled (obs, mask) pair of the NumPy calling convention with the shadow msw_step_host's delta
    expansion keeps for it.  obs is 64-byte aligned (one board row of a 16-wide plane = one cache line)."""
    __slots__ = ("raw", "obs", "mask", "shadow", "valid")

    def __init__(self, n: int, H: int, W: int, shadow_words: int):
        count = n * OBS_CHANNELS * H * W
        self.raw = np.empty((count + 16,), np.float32)
        off = ((-self.raw.ctypes.data) % 64) // 4
        self.obs = self.raw[off:off + count].reshape(n, OBS_CHANNELS, H, W)
        self.mask = np.empty((n, H * W), bool)
        self.shadow = np.empty((n, max(1, shadow_words)), np.uint64)
        self.valid = 0                     # 0: obs / mask hold garbage; 1: exactly what `shadow` describes
        for a in (self.raw, self.mask, self.shadow):       # scattered line updates: fewer TLB misses with huge pages
            _madvise_hugepage(a)


class VecMinesweeper:
    """Batched Minesweeper on one B200; API of the reference class (env.py:379-517)."""

    def __init__(
        self,
        num_envs: int,
        cfg: EnvConfig,
        seed: int = 0,
        late_start_cfg: Optional[Dict[str, Any]] = None,
        late_start_seed: Optional[int] = None,
        *,
        device: Union[str, torch.device, None] = None,
        api: str = "numpy",
        env_id_base: int = 0,
        aux_maps: bool = False,
    ):
        assert num_envs > 0                                           # env.py:390
        if api not in ("numpy", "torch"):
            raise ValueError("api must be 'numpy' or 'torch'")
        self._L = _lib.load()                                         # raises if the CUDA library is missing
        if not torch.cuda.is_available():
            raise RuntimeError("VecMinesweeper needs a CUDA device; this package has no CPU fallback")
        self.cfg = cfg
        self.num_envs = int(num_envs)
        self.api = api
        self.aux_maps = bool(aux_maps)
        self.seed = int(seed)
        self.H, self.W = int(cfg.H), int(cfg.W)
        self.HW = self.H * self.W
        self.wpb = self._L.msw_words_per_board(self.H, self.W)
        if self.wpb == 0:
            raise ValueError(f"unsupported board {self.H}x{self.W}: need 1<=W<=32 and H*W<={_lib.MAX_CELLS}")
        if not 0 <= int(cfg.mine_count) <= self.HW - 1:
            raise ValueError(f"mine_count {cfg.mine_count} out of range for {self.H}x{self.W}")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise RuntimeError("VecMinesweeper state lives in HBM; device must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())

        n, dev = self.num_envs, self.device
        self._mines = torch.zeros((n, self.wpb), dtype=torch.int32, device=dev)
        self._revealed = torch.zeros((n, self.wpb), dtype=torch.int32, device=dev)
        self._flags: Optional[torch.Tensor] = None                    # allocated only if flags are ever set
        self._meta = torch.zeros((n, 4), dtype=torch.int32, device=dev)

        rs, rl, rw = reward_constants(cfg)
        self.reward_constants = (rs, rl, rw)
        self._desc = _lib.EnvDesc(self.H, self.W, int(cfg.mine_count), int(bool(cfg.guarantee_safe_neighborhood)),
                                  float(rs), float(rl), float(rw), 0, self.seed & 0xFFFFFFFFFFFFFFFF, int(env_id_base))
        self._state = _lib.State()
        self._sync_state_struct()
        self._io = _lib.StepIO()
        self._inject: Optional[Tuple[torch.Tensor, torch.Tensor]] = None
        self._cache: Optional[Dict[str, np.ndarray]] = None
        self._pinned: Dict[str, torch.Tensor] = {}
        self._host_calls: Dict[Any, Any] = {}
        self._pinned_ok: set = set()
        self._result_pool: list = []
        self.host_delta = True       # NumPy convention: rewrite only what changed in a recycled result set (step_host)
        # host threads of the NumPy-result expansion: the CPUs this process may use, shared between the ranks
        # torchrun started on this node (one process per GPU)
        try:
            cpus = len(os.sched_getaffinity(0))
        except (AttributeError, OSError):
            cpus = os.cpu_count() or 1
        self.host_threads = max(1, cpus // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)))
        self._staging: Dict[str, torch.Tensor] = {}
        # late-start curriculum (env.py:397-403, 416-466): parameters normalised as the reference does
        self._late = None
        if late_start_cfg:
            lo = max(1, int(late_start_cfg.get("min_hidden", 5)))
            hi = max(lo, int(late_start_cfg.get("max_hidden", lo)))
            ls_seed = (int(late_start_seed) if late_start_seed is not None
                       else (self.seed * 0x9E3779B97F4A7C15 + 0x5DEECE66D)) & 0xFFFFFFFFFFFFFFFF
            self._late = (ls_seed, float(late_start_cfg.get("prob", 0.0)), lo, hi,
                          max(1, int(late_start_cfg.get("max_attempts", 3))),
                          max(1, int(late_start_cfg.get("max_extra_steps", self.HW))))
            if self._late[1] <= 0.0:
                self._late = None
        self.envs = _EnvList(self)
        self.mine_labels: Optional[torch.Tensor] = None               # aux maps of the last reset/step
        self.mine_valid: Optional[torch.Tensor] = None

    # ------------------------------------------------------------------ helpers
    def _sync_state_struct(self) -> None:
        s = self._state
        s.mines, s.revealed, s.meta = self._mines.data_ptr(), self._revealed.data_ptr(), self._meta.data_ptr()
        s.flags = self._flags.data_ptr() if self._flags is not None else None

    def _stream(self) -> int:
        """cudaStream_t of torch's current stream on the env's device (the raw getter skips building a Stream object:
        ~2 us per call, which is 1.5 % of a host-buffer step)."""
        if _raw_stream is not None:
            return _raw_stream(self.device.index)
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check(self, t: Optional[torch.Tensor], shape, dtype, name: str) -> Optional[int]:
        if t is None:
            return None
        if t.device != self.device or t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
            raise ValueError(f"{name}: need contiguous {dtype} {tuple(shape)} on {self.device}, "
                             f"got {t.dtype} {tuple(t.shape)} on {t.device}")
        return t.data_ptr()

    def _alloc_encode(self) -> StepOut:
        n, dev = self.num_envs, self.device
        return StepOut(
            obs=torch.empty((n, OBS_CHANNELS, self.H, self.W), dtype=torch.float32, device=dev),
            action_mask=torch.empty((n, self.HW), dtype=torch.bool, device=dev),
            mine_labels=torch.empty((n, self.H, self.W), dtype=torch.float32, device=dev) if self.aux_maps else None,
            mine_valid=torch.empty((n, self.H, self.W), dtype=torch.bool, device=dev) if self.aux_maps else None,
        )

    def _fill_encode(self, enc: _lib.EncodeOut, o: StepOut) -> None:
        n = self.num_envs
        enc.obs = self._check(o.obs, (n, OBS_CHANNELS, self.H, self.W), torch.float32, "obs")
        enc.mask = self._check(o.action_mask, (n, self.HW), torch.bool, "action_mask")
        enc.mine_labels = self._check(o.mine_labels, (n, self.H, self.W), torch.float32, "mine_labels")
        enc.mine_valid = self._check(o.mine_valid, (n, self.H, self.W), torch.bool, "mine_valid")

    def action_space(self) -> int:                                    # env.py:513-514
        return self.HW

    def obs_channels(self) -> int:                                    # env.py:516-517
        return OBS_CHANNELS

    # ------------------------------------------------------------------ reset
    def reset(self, out: Optional[StepOut] = None) -> Dict[str, Any]:
        """VecMinesweeper.reset (env.py:468-477)."""
        o = out if out is not None else self._alloc_encode()
        enc = _lib.EncodeOut()
        self._fill_encode(enc, o)
        with torch.cuda.device(self.device):
            if self._late is None:
                _lib.check(self._L.msw_reset(C.byref(self._desc), C.byref(self._state), self.num_envs,
                                             C.byref(enc), self._stream()), "msw_reset")
            else:                                  # env.py:406-414: reset, late start, then observe
                _lib.check(self._L.msw_reset(C.byref(self._desc), C.byref(self._state), self.num_envs,
                                             None, self._stream()), "msw_reset")
                self._apply_late(None, enc)
        self._cache = None
        self._inject = None
        self.mine_labels, self.mine_valid = o.mine_labels, o.mine_valid
        if self.api == "numpy":
            return {"obs": o.obs.cpu().numpy(), "action_mask": o.action_mask.cpu().numpy()}
        return {"obs": o.obs, "action_mask": o.action_mask}

    def _apply_late(self, sel_ptr: Optional[int], enc: _lib.EncodeOut) -> None:
        seed, prob, lo, hi, attempts, extra = self._late
        _lib.check(self._L.msw_late_start(C.byref(self._desc), C.byref(self._state), self.num_envs, sel_ptr, seed,
                                          prob, lo, hi, attempts, extra, self._stream()), "msw_late_start")
        _lib.check(self._L.msw_encode(C.byref(self._desc), C.byref(self._state), self.num_envs, C.byref(enc),
                                      self._stream()), "msw_encode")

    # ------------------------------------------------------------------ test / compat hooks
    def inject_layouts(self, mine: Union[np.ndarray, torch.Tensor], sel: Union[np.ndarray, torch.Tensor]) -> None:
        """Parity-harness hook (SURVEY 8c): envs with sel[i] that place their mines during the
        NEXT step take mine[i] (bool [n,HW] / [n,H,W]) instead of sampling."""
        if isinstance(mine, torch.Tensor):
            mine = mine.cpu().numpy()
        if isinstance(sel, torch.Tensor):
            sel = sel.cpu().numpy()
        bits = torch.from_numpy(pack_boards(mine, self.HW)).to(self.device)
        s = torch.from_numpy(np.ascontiguousarray(sel, dtype=np.uint8)).to(self.device)
        assert bits.shape == (self.num_envs, self.wpb) and s.shape == (self.num_envs,)
        self._inject = (bits, s)

    def set_state(self, *, mine=None, revealed=None, flags=None, first_click_done=None, step_count=None) -> None:
        """Overwrite parts of the device state from per-cell host arrays (tests, late-start tooling)."""
        n = self.num_envs
        if mine is not None:
            self._mines.copy_(torch.from_numpy(pack_boards(mine, self.HW)))
        if revealed is not None:
            self._revealed.copy_(torch.from_numpy(pack_boards(revealed, self.HW)))
        if flags is not None:
            if self._flags is None:
                self._flags = torch.zeros((n, self.wpb), dtype=torch.int32, device=self.device)
            self._flags.copy_(torch.from_numpy(pack_boards(flags, self.HW)))
        if first_click_done is not None:
            self._meta[:, 0] = torch.as_tensor(np.asarray(first_click_done, dtype=np.int32), device=self.device)
        if step_count is not None:
            self._meta[:, 1] = torch.as_tensor(np.asarray(step_count, dtype=np.int32), device=self.device)
        self._sync_state_struct()
        self._cache = None

    def encode(self, out: Optional[StepOut] = None) -> Dict[str, Any]:
        """Observation / mask (/aux maps) of the current state without stepping."""
        o = out if out is not None else self._alloc_encode()
        enc = _lib.EncodeOut()
        self._fill_encode(enc, o)
        with torch.cuda.device(self.device):
            _lib.check(self._L.msw_encode(C.byref(self._desc), C.byref(self._state), self.num_envs,
                                          C.byref(enc), self._stream()), "msw_encode")
        self.mine_labels, self.mine_valid = o.mine_labels, o.mine_valid
        if self.api == "numpy":
            return {"obs": o.obs.cpu().numpy(), "action_mask": o.action_mask.cpu().numpy()}
        return {"obs": o.obs, "action_mask": o.action_mask}

    def _unpacked(self) -> Dict[str, np.ndarray]:
        """Lazy device->host expansion of the bitboards for the `.envs[i]` views."""
        if self._cache is None:
            n, HW, dev = self.num_envs, self.HW, self.device
            bufs = [torch.empty((n, HW), dtype=torch.uint8, device=dev) for _ in range(4)]
            with torch.cuda.device(dev):
                _lib.check(self._L.msw_unpack_state(C.byref(self._desc), C.byref(self._state), n,
                                                    *[b.data_ptr() for b in bufs], self._stream()),
                           "msw_unpack_state")
            names = ("mine", "revealed", "flags", "counts")
            self._cache = {k: b.cpu().numpy() for k, b in zip(names, bufs)}
            self._cache["meta"] = self._meta.cpu().numpy()
        return self._cache

    def forced_subset(self) -> np.ndarray:
        """rules.analyze_forced_modules (rules.py:206-259) for every env in one launch: bool [n, HW]
        of "subset_reveal" cells (cached until the next step / reset)."""
        u = self._unpacked()
        if "subset" not in u:
            bits = torch.empty((self.num_envs, self.wpb), dtype=torch.int32, device=self.device)
            self._launch_forced_subset(bits)
            raw = bits.cpu().numpy().view(np.uint8).reshape(self.num_envs, -1)
            u["subset"] = np.unpackbits(raw, axis=1, count=self.HW, bitorder="little").astype(bool)
        return u["subset"]

    def avoidability(self, search_budget: int = 0) -> Dict[str, np.ndarray]:
        """avoidability.analyze_avoidability (avoidability.py:145-394) for every env in one launch, in the
        array form of msw_avoidability: {"safe": bool [n,HW], "comp_of_cell": i16 [n,HW], "comp_size": i16
        [n,HW], "flags": u8 [n]} (cached until the next step / reset)."""
        u = self._unpacked()
        if "avoid" not in u:
            n, HW, dev = self.num_envs, self.HW, self.device
            bits = torch.empty((n, self.wpb), dtype=torch.int32, device=dev)
            coc = torch.empty((n, HW), dtype=torch.int16, device=dev)
            cs = torch.empty((n, HW), dtype=torch.int16, device=dev)
            fl = torch.empty((n,), dtype=torch.uint8, device=dev)
            self._launch_avoidability(bits, coc, cs, fl, search_budget)
            raw = bits.cpu().numpy().view(np.uint8).reshape(n, -1)
            u["avoid"] = {"safe": np.unpackbits(raw, axis=1, count=HW, bitorder="little").astype(bool),
                          "comp_of_cell": coc.cpu().numpy(), "comp_size": cs.cpu().numpy(), "flags": fl.cpu().numpy()}
        return u["avoid"]

    # device halves of forced_subset() / avoidability(): fill caller-owned device buffers, no host copy, no cache
    def _launch_forced_subset(self, bits: torch.Tensor) -> None:
        """msw_forced_subset into int32 [n, wpb] `bits`."""
        self._check(bits, (self.num_envs, self.wpb), torch.int32, "subset bits")
        with torch.cuda.device(self.device):
            _lib.check(self._L.msw_forced_subset(C.byref(self._desc), C.byref(self._state), self.num_envs,
                                                 bits.data_ptr(), self._stream()), "msw_forced_subset")

    def _launch_avoidability(self, bits: torch.Tensor, coc: torch.Tensor, cs: torch.Tensor, fl: torch.Tensor,
                             search_budget: int = 0) -> None:
        """msw_avoidability into int32 [n, wpb] `bits`, int16 [n, HW] `coc` / `cs` and uint8 [n] `fl`."""
        n, HW = self.num_envs, self.HW
        self._check(bits, (n, self.wpb), torch.int32, "safe bits")
        self._check(coc, (n, HW), torch.int16, "comp_of_cell")
        self._check(cs, (n, HW), torch.int16, "comp_size")
        self._check(fl, (n,), torch.uint8, "avoid flags")
        with torch.cuda.device(self.device):
            _lib.check(self._L.msw_avoidability(C.byref(self._desc), C.byref(self._state), n, bits.data_ptr(),
                                                coc.data_ptr(), cs.data_ptr(), fl.data_ptr(),
                                                int(search_budget) & 0xFFFFFFFF, self._stream()), "msw_avoidability")

    def random_actions(self, step_index: int, valid_only: bool = True, seed: int = 1,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Synthetic action source (BASELINE.md section 4): uniformly random unrevealed cell
        (or any cell) per env, generated on device."""
        if out is None:
            out = torch.empty((self.num_envs,), dtype=torch.int32, device=self.device)
        a32 = out.data_ptr() if out.dtype == torch.int32 else None
        a64 = out.data_ptr() if out.dtype == torch.int64 else None
        if (a32 is None and a64 is None) or out.device != self.device or out.shape != (self.num_envs,):
            raise ValueError("random_actions: out must be int32/int64 [num_envs] on the env device")
        with torch.cuda.device(self.device):
            _lib.check(self._L.msw_random_actions(C.byref(self._desc), C.byref(self._state), self.num_envs,
                                                  int(seed) & 0xFFFFFFFFFFFFFFFF, int(step_index) & 0xFFFFFFFF,
                                                  int(valid_only), a32, a64, self._stream()),
                       "msw_random_actions")
        return out

    # ------------------------------------------------------------------ step
    def _info_tensors(self) -> Dict[str, torch.Tensor]:
        st = self._staging
        if "outcome" not in st:
            n, dev = self.num_envs, self.device
            st["outcome"] = torch.empty((n,), dtype=torch.int8, device=dev)
            st["new_reveals"] = torch.empty((n,), dtype=torch.int32, device=dev)
            st["step"] = torch.empty((n,), dtype=torch.int32, device=dev)
            st["revealed_count"] = torch.empty((n,), dtype=torch.int32, device=dev)
        return st

    def step_random(self, step_index: int, valid_only: bool = True, seed: int = 1, out: Optional[StepOut] = None,
                    actions_out: Optional[torch.Tensor] = None, want_infos: bool = False):
        """Env-only throughput mode (BASELINE.md section 4): one launch that draws the synthetic
        action -- exactly what `random_actions(step_index, valid_only, seed)` returns -- and steps."""
        if self.api != "torch":
            raise ValueError("step_random needs api='torch'")
        return self._step_device(None, out, want_infos, (1 if valid_only else 2, int(step_index), int(seed), actions_out))

    def step(self, actions, out: Optional[StepOut] = None, want_infos: bool = True):
        """VecMinesweeper.step (env.py:479-511).  Returns (batch, rewards, dones, infos)."""
        if self.api == "numpy":
            return self._step_numpy(actions)
        return self._step_device(actions, out, want_infos, None)

    def _step_device(self, actions, out: Optional[StepOut], want_infos: bool, _rand):
        """One msw_step launch on device tensors; `_rand` = (mode, step_index, seed, actions_out) selects
        the built-in synthetic policy instead of `actions`."""
        n, dev = self.num_envs, self.device
        if _rand is None:
            if not isinstance(actions, torch.Tensor):
                actions = torch.as_tensor(np.asarray(actions))
            assert tuple(actions.shape) == (n,)                       # env.py:480
            if actions.dtype not in (torch.int32, torch.int64):
                actions = actions.to(torch.int64)
            actions = actions.to(dev).contiguous()
        o = out if out is not None else self._alloc_encode()
        rewards = o.rewards if o.rewards is not None else torch.empty((n,), dtype=torch.float32, device=dev)
        dones = o.dones if o.dones is not None else torch.empty((n,), dtype=torch.bool, device=dev)
        io = self._io
        if _rand is None:
            io.actions32 = actions.data_ptr() if actions.dtype == torch.int32 else None
            io.actions64 = actions.data_ptr() if actions.dtype == torch.int64 else None
            io.rand_mode, io.actions_out32 = 0, None
        else:
            mode, step_index, seed, a_out = _rand
            io.actions32 = io.actions64 = None
            io.rand_mode, io.rand_step, io.rand_seed = mode, step_index & 0xFFFFFFFF, seed & 0xFFFFFFFFFFFFFFFF
            io.actions_out32 = self._check(a_out, (n,), torch.int32, "actions_out")
        io.inject_bits, io.inject_sel = ((self._inject[0].data_ptr(), self._inject[1].data_ptr())
                                         if self._inject is not None else (None, None))
        io.reward = self._check(rewards, (n,), torch.float32, "rewards")
        io.done = self._check(dones, (n,), torch.bool, "dones")
        infos: Dict[str, Any] = {}
        if want_infos:
            it = self._info_tensors()
            io.outcome, io.new_reveals = it["outcome"].data_ptr(), it["new_reveals"].data_ptr()
            io.step, io.revealed_count = it["step"].data_ptr(), it["revealed_count"].data_ptr()
            infos = {"outcome_code": it["outcome"], "last_new_reveals": it["new_reveals"], "step": it["step"],
                     "revealed_count": it["revealed_count"], "done": dones}
        else:
            io.outcome = io.new_reveals = io.step = io.revealed_count = None
        self._fill_encode(io.enc, o)
        with torch.cuda.device(dev):
            if self._late is None:
                _lib.check(self._L.msw_step(C.byref(self._desc), C.byref(self._state), C.byref(io), n,
                                            self._stream()), "msw_step")
            else:        # step without observing, late-start the envs that just finished, then observe
                enc = _lib.EncodeOut(io.enc.obs, io.enc.mask, io.enc.mine_labels, io.enc.mine_valid)
                io.enc.obs = io.enc.mask = io.enc.mine_labels = io.enc.mine_valid = None
                _lib.check(self._L.msw_step(C.byref(self._desc), C.byref(self._state), C.byref(io), n,
                                            self._stream()), "msw_step")
                self._apply_late(io.done, enc)
        self._inject = None
        self._cache = None
        self.mine_labels, self.mine_valid = o.mine_labels, o.mine_valid
        return {"obs": o.obs, "action_mask": o.action_mask}, rewards, dones, infos

    # reference calling convention: NumPy in / NumPy out (msw_step_host)
    def _host_buffers(self) -> Tuple[Dict[str, torch.Tensor], Dict[str, torch.Tensor]]:
        if not self._pinned:
            n, dev = self.num_envs, self.device
            spec = {
                "actions": ((n,), torch.int32), "reward": ((n,), torch.float32), "done": ((n,), torch.bool),
                "outcome": ((n,), torch.int8), "new_reveals": ((n,), torch.int32), "step": ((n,), torch.int32),
                "revealed_count": ((n,), torch.int32),
            }
            # The per-env scalars sit back to back (reward | done | outcome | pad | new_reveals | step |
            # revealed_count) in ONE pinned and ONE device allocation, in the order msw_step_host queues
            # its copies, so they travel as a single DMA.
            scalars = ("reward", "done", "outcome", "new_reveals", "step", "revealed_count")
            offs, off = {}, 0
            for k in scalars:
                shape, dt = spec[k]
                off = (off + dt.itemsize - 1) // dt.itemsize * dt.itemsize
                offs[k] = off
                off += n * dt.itemsize
            dev_blob = torch.empty((off,), dtype=torch.uint8, device=dev)
            pin_blob = _fastest_pinned(off, dev_blob, to_host=True)
            for k, (shape, dt) in spec.items():
                if k in offs:
                    nb = n * dt.itemsize
                    self._pinned[k] = pin_blob[offs[k]:offs[k] + nb].view(dt)
                    self._staging["h_" + k] = dev_blob[offs[k]:offs[k] + nb].view(dt)
                else:
                    self._staging["h_" + k] = torch.empty(shape, dtype=dt, device=dev)
                    self._pinned[k] = _fastest_pinned(n * dt.itemsize, self._staging["h_" + k].view(torch.uint8),
                                                      to_host=False).view(dt)
            # packed post-step state (mines | revealed | meta): what obs / mask are expanded from on the host
            self._pinned["stage"] = torch.empty((n * (2 * self.wpb + 4),), dtype=torch.int32).pin_memory()
        return self._pinned, self._staging

    @staticmethod
    def host_obs_d2h_bytes(H: int, W: int, n: int) -> int:
        """Device->host bytes per step of the reference calling convention: packed state + reward + done
        (the fp32 planes are expanded on the host, they do not cross PCIe)."""
        wpb = (H * W + 31) // 32
        return n * (2 * wpb * 4 + 5)

    def _result_arrays(self) -> "_ResultSet":
        """(obs f32 [n,10,H,W], mask bool [n,HW]) for the next result.  The reference returns fresh arrays every
        call (np.stack, env.py:507-510); fresh 688 MB allocations would cost more in page faults than the whole
        step, so arrays are recycled from a small pool -- but ONLY when nobody else references them any more
        (any view / torch.from_numpy alias keeps a reference to the array or to its base), otherwise a new set is
        made.  A pooled set carries a `shadow` (the bit planes the arrays hold, include/msw_b200.h), so
        msw_step_host rewrites only the cache lines that changed since the set was last filled."""
        import sys
        for e in self._result_pool:
            # e.obs: slot + argument; e.raw: slot + obs.base + argument; e.mask: slot + argument
            if sys.getrefcount(e.obs) <= 2 and sys.getrefcount(e.raw) <= 3 and sys.getrefcount(e.mask) <= 2:
                return e
        e = _ResultSet(self.num_envs, self.H, self.W, self._L.msw_shadow_words(self.H, self.W))
        if len(self._result_pool) < 4:
            self._result_pool.append(e)
        return e

    def step_host(self, actions_pinned: torch.Tensor, *, copy_obs: bool = True, copy_infos: bool = True,
                  out: Optional[Tuple[np.ndarray, np.ndarray]] = None, threads: int = 0) -> Dict[str, Any]:
        """msw_step_host: pinned int32 actions in; per-env scalars back in pinned buffers.  With copy_obs the
        reference-shaped obs / mask NumPy arrays ("obs", "mask" of the result: `out` if given, else recycled
        arrays) are filled by the host-side expansion of the packed state; without it the kernel writes obs / mask
        into device tensors ("obs_device", "mask_device") for a device-resident consumer.  Synchronises the current
        stream.  The returned pinned tensors are valid until the next call."""
        n = self.num_envs
        pin, st = self._host_buffers()
        ap = actions_pinned.data_ptr()
        if ap not in self._pinned_ok:                          # is_pinned() is a driver query: ask once per ALLOCATION
            base = actions_pinned.untyped_storage().data_ptr()
            if not (actions_pinned.dtype == torch.int32 and tuple(actions_pinned.shape) == (n,) and
                    actions_pinned.is_contiguous() and (base in self._pinned_ok or actions_pinned.is_pinned())):
                raise ValueError("step_host: actions must be a pinned contiguous int32 [num_envs] CPU tensor")
            if len(self._pinned_ok) < 65536:
                self._pinned_ok.add(ap)
                self._pinned_ok.add(base)
        key = (copy_obs, copy_infos, self.aux_maps)
        prepared = self._host_calls.get(key)
        if prepared is None:                                   # struct filling is per-configuration, not per step
            io = _lib.StepIO()
            io.actions32, io.actions64 = st["h_actions"].data_ptr(), None
            io.rand_mode, io.actions_out32 = 0, None
            io.reward, io.done = st["h_reward"].data_ptr(), st["h_done"].data_ptr()
            io.outcome, io.new_reveals = st["h_outcome"].data_ptr(), st["h_new_reveals"].data_ptr()
            io.step, io.revealed_count = st["h_step"].data_ptr(), st["h_revealed_count"].data_ptr()
            if copy_obs:                                       # the planes are made on the host: no device-side encode
                io.enc.obs = io.enc.mask = None
            else:                                              # device consumer (the policy): obs / mask written to HBM
                if "h_obs" not in st:
                    st["h_obs"] = torch.empty((n, OBS_CHANNELS, self.H, self.W), dtype=torch.float32, device=self.device)
                    st["h_mask"] = torch.empty((n, self.HW), dtype=torch.bool, device=self.device)
                io.enc.obs, io.enc.mask = st["h_obs"].data_ptr(), st["h_mask"].data_ptr()
            if self.aux_maps:                                  # device-resident aux maps for a device consumer
                if "h_labels" not in st:
                    st["h_labels"] = torch.empty((n, self.H, self.W), dtype=torch.float32, device=self.device)
                    st["h_valid"] = torch.empty((n, self.H, self.W), dtype=torch.bool, device=self.device)
                io.enc.mine_labels, io.enc.mine_valid = st["h_labels"].data_ptr(), st["h_valid"].data_ptr()
            else:
                io.enc.mine_labels = io.enc.mine_valid = None
            h = _lib.HostOut()
            h.reward, h.done = pin["reward"].data_ptr(), pin["done"].data_ptr()
            if copy_infos:
                h.outcome, h.new_reveals = pin["outcome"].data_ptr(), pin["new_reveals"].data_ptr()
                h.step, h.revealed_count = pin["step"].data_ptr(), pin["revealed_count"].data_ptr()
            h.stage = pin["stage"].data_ptr()
            prepared = self._host_calls[key] = (io, h, C.byref(self._desc), C.byref(self._state), C.byref(io),
                                                C.byref(h))
        io, h, r_desc, r_state, r_io, r_h = prepared
        res: Dict[str, Any] = dict(pin)
        if not copy_obs:
            res["obs_device"], res["mask_device"] = st["h_obs"], st["h_mask"]
        rset = None
        if copy_obs:
            if out is not None:
                obs, mask = out
            else:
                rset = self._result_arrays()
                obs, mask = rset.obs, rset.mask
            if (obs.dtype != np.float32 or obs.shape != (n, OBS_CHANNELS, self.H, self.W) or not obs.flags.c_contiguous
                    or mask.dtype != np.bool_ or mask.shape != (n, self.HW) or not mask.flags.c_contiguous):
                raise ValueError("step_host: out must be (float32 [n,10,H,W], bool [n,HW]) C-contiguous arrays")
            h.obs, h.mask = obs.ctypes.data, mask.ctypes.data
            res["obs"], res["mask"] = obs, mask
        else:
            h.obs = h.mask = None
        use_shadow = rset is not None and self.host_delta
        if use_shadow:                                         # delta mode: only what changed since this set was filled
            h.shadow, h.shadow_valid = rset.shadow.ctypes.data, rset.valid
        else:
            h.shadow, h.shadow_valid = None, 0
        if rset is not None:
            rset.valid = 0                                     # until a call has succeeded WITH the shadow kept up to date
        h.threads = int(threads) if threads else self.host_threads
        io.inject_bits, io.inject_sel = ((self._inject[0].data_ptr(), self._inject[1].data_ptr())
                                         if self._inject is not None else (None, None))
        if torch.cuda.current_device() == self.device.index:
            rc = self._L.msw_step_host(r_desc, r_state, r_io, ap, r_h, n, self._stream())
        else:
            with torch.cuda.device(self.device):
                rc = self._L.msw_step_host(r_desc, r_state, r_io, ap, r_h, n, self._stream())
        if rc:
            _lib.check(rc, "msw_step_host")
        if use_shadow:
            rset.valid = 1
        self._inject = None
        self._cache = None
        if self.aux_maps:
            self.mine_labels, self.mine_valid = st["h_labels"], st["h_valid"]
        return res

    def _step_numpy(self, actions) -> Tuple[Dict[str, np.ndarray], np.ndarray, np.ndarray, Dict[str, Any]]:
        n = self.num_envs
        actions = np.asarray(actions)
        assert actions.shape == (n,)                                  # env.py:480
        if self._late is not None:               # three launches: go through the device-tensor path
            a = np.mod(actions.astype(np.int64, copy=False), self.HW)
            self.api = "torch"
            try:
                b, r, d, info = self.step(torch.from_numpy(a))
            finally:
                self.api = "numpy"
            dones = d.cpu().numpy()
            outcome, newr = info["outcome_code"].cpu().numpy(), info["last_new_reveals"].cpu().numpy()
            step, rc = info["step"].cpu().numpy(), info["revealed_count"].cpu().numpy()
            batch = {"obs": b["obs"].cpu().numpy(), "action_mask": b["action_mask"].cpu().numpy()}
            rewards = r.cpu().numpy()
        else:
            pin, _ = self._host_buffers()
            if actions.dtype.kind in "iu" and (actions.dtype.itemsize < 4 or actions.dtype == np.int32):
                pin["actions"].numpy()[:] = actions               # fits int32 as it is: one conversion pass
            else:
                a = actions.astype(np.int64, copy=False)
                # int(actions[i]) % (H*W) with Python semantics (env.py:104-106) for values beyond int32
                if a.size and (a.max() > 2**31 - 1 or a.min() < -2**31):
                    a = np.mod(a, self.HW)
                pin["actions"].numpy()[:] = a
            res = self.step_host(pin["actions"])
            rewards = pin["reward"].numpy().copy()
            dones = pin["done"].numpy().copy()
            outcome, newr = pin["outcome"].numpy(), pin["new_reveals"].numpy()
            step, rc = pin["step"].numpy(), pin["revealed_count"].numpy()
            batch = {"obs": res["obs"], "action_mask": res["mask"]}
            del res
        # env.py:485-505: per-env Python lists.  Building N dicts costs more than the whole step at large N and
        # train_rl.py:242 never looks at them, so the lists are lazy sequences over copies of the scalar arrays:
        # same indexing / len / iteration / equality as the reference's lists, items made on access.
        hw = max(1, self.HW)
        step, newr, rc, outcome, done_i = step.copy(), newr.copy(), rc.copy(), outcome.copy(), dones.copy()
        infos = {
            "aux": _LazyList(n, lambda i: {"step": int(step[i]), "last_new_reveals": int(newr[i]),
                                           "revealed_frac": int(rc[i]) / hw}),
            "outcome": _LazyList(n, lambda i: _OUTCOME_NAMES[outcome[i]]),
            "done": _LazyList(n, lambda i: bool(done_i[i])),
        }
        return batch, rewards, dones, infos

    # ------------------------------------------------------------------ raw state (native API)
    @property
    def state_tensors(self) -> Dict[str, Optional[torch.Tensor]]:
        """Bitboard state in HBM: int32 [n, wpb] boards and int32 [n,4] meta."""
        return {"mines": self._mines, "revealed": self._revealed, "flags": self._flags, "meta": self._meta}
