"""-m gpu: the CUDA env against the REAL reference at scale.

1. `test_cuda_matches_reference_trace`: replays tests/golden/trace_*.npz (4,096 envs x 256 steps of the
   live reference, recorded as SHA-256 digests) through the C ABI -- needs nothing but the fixtures.
2. `test_lockstep_with_live_reference`: imports the unmodified reference from baseline/_ref ON THIS BOX
   and steps it side by side with the CUDA env (BASELINE.md section 4, C2 parity sub-run: N=4,096,
   256 steps, 16x16x40, layouts injected from the reference), comparing every output and the per-env
   state of every step array against array.
3. `test_unmodified_evaluate_vec_on_cuda_env`: BASELINE configs[0] (C1) -- the reference's own
   eval.evaluate_vec (eval.py:265-511), unmodified, run once on the reference numba env and once with
   `eval.VecMinesweeper` pointed at the CUDA env (reference calling convention, `vec.envs[i]` views,
   list-of-dict infos; rules.analyze_forced_modules / avoidability.analyze_avoidability are the
   reference's own, reading the CUDA env's state views); the metric dicts must be equal.

2, 3 and the live collector test skip when the reference is not installed (tools/install_reference.sh puts it
in baseline/_ref); 1, test_gpu_rollout's C1 test and test_gpu_gae's rollout-fixture test hold the same comparisons
against recorded reference outputs.
"""
import math

import numpy as np
import pytest

import parity as P
import reference_live as RL
import trace as TR

pytestmark = pytest.mark.gpu

N, T = 4096, 256
needs_reference = pytest.mark.skipif(not RL.available(), reason=RL.SKIP_REASON)


def _make_cuda(cfg, n):
    return P.CudaAdapter(cfg, n)


@pytest.mark.parametrize("series", ["A", "B", "C"])
def test_cuda_matches_reference_trace(series):
    stats = TR.replay_trace(series, N, T, TR.trace_cfg(), _make_cuda)
    assert stats["layouts_placed"] > 20000
    if series == "C":
        assert stats["wins"] > 5000


@needs_reference
@pytest.mark.parametrize("series,steps,env_seed", [("A", 256, 7), ("B", 64, 8), ("C", 256, 9)])
def test_lockstep_with_live_reference(series, steps, env_seed):
    # seeds differ from the recorded traces', so this is fresh ground every time the reference is present
    stats = TR.lockstep_live(series, N, steps, TR.trace_cfg(), _make_cuda, env_seed=env_seed, action_seed=env_seed + 100)
    print(f"lock-step series {series}: {N}x{steps} env-steps, {stats}")
    assert stats["layouts_placed"] > 0
    if series == "C":
        assert stats["wins"] > 1000


@needs_reference
def test_lockstep_expert_board_live_reference():
    """C4's board (H=16, W=30, 99 mines) and its transpose (H=30, W=16), 512 envs x 96 steps each."""
    for H, W in ((16, 30), (30, 16)):
        TR.lockstep_live("C", 512, 96, TR.trace_cfg(H, W, 99), _make_cuda, env_seed=3, action_seed=4)
        TR.lockstep_live("A", 512, 32, TR.trace_cfg(H, W, 99), _make_cuda, env_seed=5, action_seed=6)


def _metrics_equal(a, b):
    assert a.keys() == b.keys()
    for k in a:
        x, y = float(a[k]), float(b[k])
        assert (math.isnan(x) and math.isnan(y)) or x == y, (k, x, y)


def _run_eval_both(model, episodes, num_envs, seed):
    """Unmodified eval.evaluate_vec on (1) the reference env, recording the layouts it draws per (env,
    episode), (2) the CUDA env replaying exactly those layouts."""
    import torch
    ev = RL.load_eval()
    E = RL.load()["env"]
    env_cfg = E.EnvConfig(H=16, W=16, mine_count=40, guarantee_safe_neighborhood=True, step_penalty=1e-4)
    layouts, made = {}, []
    orig_vec = ev.VecMinesweeper

    class RecordingVec(orig_vec):                  # subclass only to learn each env object's index
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            made.append(self)

    with RL.LayoutRecorder() as rec:
        ev.VecMinesweeper = RecordingVec
        try:
            want = ev.evaluate_vec(model, env_cfg, episodes=episodes, seed=seed, num_envs=num_envs)
        finally:
            ev.VecMinesweeper = orig_vec
        index_of = {id(e): i for i, e in enumerate(made[0].envs)}
        for i, m in rec.drain(index_of):
            layouts.setdefault(i, []).append(m)
    cuda_vec = []
    Inj = RL.make_injecting_vec(layouts)

    class Tracked(Inj):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            cuda_vec.append(self)

    ev.VecMinesweeper = Tracked
    try:
        got = ev.evaluate_vec(model, env_cfg, episodes=episodes, seed=seed, num_envs=num_envs)
    finally:
        ev.VecMinesweeper = orig_vec
    assert cuda_vec and cuda_vec[0].injected == sum(len(v) for v in layouts.values())
    torch.cuda.synchronize()
    return want, got


@needs_reference
def test_unmodified_evaluate_vec_on_cuda_env():
    import torch
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    # (i) BASELINE configs[0]: 64 envs, 256 episodes, random-init medium cnn_residual built by the reference
    models = RL.load()["models"]
    torch.manual_seed(0)
    model = models.build_model("cnn_residual", obs_shape=(10, 16, 16),
                               model_cfg=dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256)).cuda()
    want, got = _run_eval_both(model, 256, 64, 0)
    _metrics_equal(want, got)
    assert want["episodes"] == 256.0
    # (ii) a scripted policy with exact integer logits that plays long games (hundreds of analytics calls,
    # forced-guess / safe-option branches, wins)
    pol = P.scripted_policy(16, 16).cuda()
    want2, got2 = _run_eval_both(pol, 96, 32, 1)
    _metrics_equal(want2, got2)
    assert want2["avg_steps"] > 3.0
    print("C1 (random-init medium policy):", got)
    print("C1 (scripted policy):", got2)


@needs_reference
def test_live_collect_rollout_buffer_and_gae():
    """The reference's REAL collector (train_rl.collect_rollout, train_rl.py:155-289) run live on this box --
    reference numba env on the host, the reference's medium cnn_residual on the GPU under fp16 autocast, torch's
    Categorical sampling, aux maps on -- at 1,024 envs x 64 steps, then RolloutBuffer.compute_gae on the GPU with
    the fp16 bootstrap value autocast produces (train_rl.py:272-277).  The CUDA env, fed the same actions and the
    reference's mine layouts through the direct-write buffer protocol (slot t+1 gets obs / mask / labels / valid,
    slot t gets reward / done), must rebuild the reference's buffer bit for bit, and msw_gae must reproduce its
    advantages / returns bit for bit from the reference's values."""
    import torch
    import minesweeper_ppo_b200 as m
    mods = RL.load()
    import importlib
    train_rl = importlib.import_module("train_rl")
    E = mods["env"]
    N, T, H, W = 1024, 64, 16, 16
    HW = H * W
    cfg = E.EnvConfig(H=H, W=W, mine_count=40, guarantee_safe_neighborhood=True, step_penalty=1e-4)
    torch.manual_seed(0)
    model = mods["models"].build_model("cnn_residual", obs_shape=(10, H, W),
                                       model_cfg=dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256)).cuda()
    dev = torch.device("cuda")
    with RL.LayoutRecorder() as rec:
        vec = E.VecMinesweeper(N, cfg, seed=21)
        index_of = {id(e): i for i, e in enumerate(vec.envs)}
        placed = []                       # (step, env, layout)
        tcount = [0]
        orig_step = vec.step

        def step_logged(actions):
            r = orig_step(actions)
            for i, mm in rec.drain(index_of):
                placed.append((tcount[0], i, mm.reshape(-1)))
            tcount[0] += 1
            return r

        vec.step = step_logged
        buf, aux = train_rl.collect_rollout(vec, model, T, dev, aux_mine_weight=0.05, aux_mine_calib_weight=0.01)
    last_values = aux["last_values"].detach()
    assert last_values.dtype == torch.float16, "autocast bootstrap value (train_rl.py:272-277)"
    buf.compute_gae(last_values, gamma=0.995, lam=0.95)
    assert int(buf.dones.sum()) > 1000 and len(placed) > 1000

    v = m.VecMinesweeper(N, m.EnvConfig(H=H, W=W, mine_count=40, step_penalty=1e-4), api="torch", aux_maps=True)
    mine = m.RolloutBuffer(N, T, (10, H, W), HW, v.device, aux_maps=True)
    scratch = v._alloc_encode()
    v.reset(out=mine.slot(0))
    by_step = {}
    for t, i, mm in placed:
        by_step.setdefault(t, []).append((i, mm))
    ref_actions = buf.actions.view(T, N)
    for t in range(T):
        sel = np.zeros(N, bool)
        lay = np.zeros((N, HW), bool)
        for i, mm in by_step.get(t, ()):
            sel[i], lay[i] = True, mm
        v.inject_layouts(lay, sel)
        nxt = mine.slot(t + 1) if t + 1 < T else scratch
        cur = mine.slot(t)
        v.step(ref_actions[t].to(v.device), out=m.StepOut(obs=nxt.obs, action_mask=nxt.action_mask, rewards=cur.rewards,
                                                          dones=cur.dones, mine_labels=nxt.mine_labels,
                                                          mine_valid=nxt.mine_valid), want_infos=False)
    mine.values.copy_(buf.values)
    mine.compute_gae(last_values, 0.995, 0.95)
    torch.cuda.synchronize()
    for name in ("obs", "action_mask", "rewards", "dones", "mine_labels", "mine_valid", "advantages", "returns"):
        a, b = getattr(mine, name), getattr(buf, name)
        assert a.dtype == b.dtype and a.shape == b.shape, name
        if a.dtype.is_floating_point:
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), name      # bit patterns
        else:
            assert torch.equal(a, b), name
