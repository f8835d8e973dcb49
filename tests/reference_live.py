"""Import the UNMODIFIED reference (yakvrz/minesweeper-ppo) as installed under baseline/_ref/.

`tools/install_reference.sh` copies the reference tree verbatim into baseline/_ref/ (git-ignored,
travels to the GPU box with the working tree).  This helper puts it on sys.path with numba's cache
redirected to a writable temp dir (`@njit(cache=True)`, env_numba.py:16) and offers the two wrappers
the live parity tests need:

  LayoutRecorder   wraps -- does not edit -- MinesweeperEnv._place_mines_safe (env.py:280-312) and
                   logs every mine layout the reference draws, so the CUDA env can be fed the same
                   boards through `inject_layouts` (SURVEY 8c "How layouts are shared").
  InjectingVec     minesweeper_ppo_b200.VecMinesweeper in the reference calling convention that
                   replays recorded layouts by (env index, episode number); the stand-in the
                   unmodified eval.evaluate_vec is pointed at.

Test infrastructure only.  Nothing here reads /root/reference: the GPU box does not have it.
"""
from __future__ import annotations

import os
import sys
import tempfile
from typing import Dict, List, Optional

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.environ.get("MSW_REFERENCE", os.path.join(ROOT, "baseline", "_ref"))

_mods: Optional[Dict[str, object]] = None


def available() -> bool:
    return os.path.isfile(os.path.join(REF_DIR, "minesweeper", "env.py"))


SKIP_REASON = (f"the reference is not installed at {REF_DIR} (tools/install_reference.sh <checkout>); "
               "it is not part of this repository")


def require():
    if not available():
        raise RuntimeError(f"{REF_DIR} is missing: install the reference with tools/install_reference.sh <checkout>")


def load() -> Dict[str, object]:
    """Import the reference's modules.  Returns {"env", "env_numba", "buffers", "rules", "avoidability",
    "models", "eval"} (eval imported lazily by `load_eval`)."""
    global _mods
    if _mods is not None:
        return _mods
    require()
    os.environ.setdefault("NUMBA_CACHE_DIR", tempfile.mkdtemp(prefix="msw_numba_cache_"))
    sys.dont_write_bytecode = True
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import minesweeper.env as ref_env
    import minesweeper.env_numba as ref_env_numba
    import minesweeper.buffers as ref_buffers
    import minesweeper.rules as ref_rules
    import minesweeper.avoidability as ref_avoid
    import minesweeper.models as ref_models
    assert os.path.realpath(ref_env.__file__).startswith(os.path.realpath(REF_DIR)), ref_env.__file__
    assert ref_env_numba.HAS_ENV_NUMBA, "the reference must run its numba flood fill (env_numba.py)"
    _mods = dict(env=ref_env, env_numba=ref_env_numba, buffers=ref_buffers, rules=ref_rules,
                 avoidability=ref_avoid, models=ref_models)
    return _mods


def load_eval():
    """The reference's eval.py (module name `eval`), unmodified."""
    load()
    import importlib
    mod = importlib.import_module("eval")
    assert os.path.realpath(mod.__file__).startswith(os.path.realpath(REF_DIR)), mod.__file__
    return mod


class LayoutRecorder:
    """Context manager: logs (env object, mine_mask copy) for every _place_mines_safe call."""

    def __init__(self):
        self.env_mod = load()["env"]
        self.log: List = []
        self._orig = self.env_mod.MinesweeperEnv._place_mines_safe

    def __enter__(self):
        rec, orig = self, self._orig

        def wrapped(env, first_click_rc):
            orig(env, first_click_rc)
            rec.log.append((env, env.mine_mask.copy()))

        self.env_mod.MinesweeperEnv._place_mines_safe = wrapped
        return self

    def __exit__(self, *exc):
        self.env_mod.MinesweeperEnv._place_mines_safe = self._orig

    def drain(self, index_of: Dict[int, int]):
        """-> list of (env index, bool [H,W]) placed since the last drain."""
        out = [(index_of[id(e)], m) for e, m in self.log]
        self.log = []
        return out


def make_injecting_vec(layouts_by_env: Dict[int, List[np.ndarray]]):
    """Class with the reference constructor signature `VecMinesweeper(num_envs, cfg, seed)` backed by the
    CUDA env (api="numpy"); env i's k-th episode uses layouts_by_env[i][k]."""
    import minesweeper_ppo_b200 as m

    class InjectingVec(m.VecMinesweeper):
        def __init__(self, num_envs, cfg, seed=0, late_start_cfg=None, late_start_seed=None):
            ec = m.EnvConfig(H=cfg.H, W=cfg.W, mine_count=cfg.mine_count,
                             guarantee_safe_neighborhood=cfg.guarantee_safe_neighborhood,
                             win_reward=cfg.win_reward, loss_reward=cfg.loss_reward, step_penalty=cfg.step_penalty)
            super().__init__(num_envs, ec, seed, late_start_cfg, late_start_seed, api="numpy")
            self._fresh = np.ones(num_envs, bool)
            self._episode = np.zeros(num_envs, np.int64)
            self.injected = 0

        def reset(self, *a, **k):
            self._fresh[:] = True
            return super().reset(*a, **k)

        def step(self, actions, *a, **k):
            n, HW = self.num_envs, self.HW
            sel = self._fresh.copy()
            mine = np.zeros((n, HW), bool)
            for i in np.nonzero(sel)[0]:
                mine[i] = layouts_by_env[int(i)][int(self._episode[i])].reshape(-1)
            self.inject_layouts(mine, sel)
            self.injected += int(sel.sum())
            out = super().step(actions, *a, **k)
            dones = np.asarray(out[2], bool)
            self._episode[sel] += 1              # a click on a fresh board always places the mines
            self._fresh = dones.copy()           # done -> auto-reset -> fresh board
            return out

    return InjectingVec
