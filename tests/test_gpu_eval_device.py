"""Device-resident greedy evaluator (evaluate.evaluate_vec_device, DESIGN.md section 4.9): the metric dict
against the reference's own recorded dict and against evaluate_vec, msw_masked_argmax against torch, canary
windows around every output of the new kernels.  Needs a B200."""
import json
import math
from collections import deque

import numpy as np
import pytest

import parity as P

pytestmark = pytest.mark.gpu
PAD = 4096          # canary bytes on each side of a window


def _assert_same_dict(got, want, belief_tol=0.0):
    assert set(got) == set(want), set(got) ^ set(want)
    for k, w in want.items():
        v = got[k]
        if isinstance(w, float) and math.isnan(w):
            assert math.isnan(v), (k, v)
        elif k == "avg_progress":                   # float64 summation order (DESIGN.md section 4.9)
            assert abs(v - w) <= 1e-12 * abs(w), (k, v, w)
        elif k.startswith("belief_"):
            assert abs(v - w) <= belief_tol, (k, v, w)
        else:
            assert v == w, (k, v, w)


@pytest.mark.parametrize("name", ["8x8x10", "16x16x40"])
def test_device_eval_matches_reference_metrics(name):
    """tests/golden/c1_eval.npz: the dict the unmodified reference eval.evaluate_vec produced with the scripted
    policy, and every layout its envs drew; replayed through evaluate_vec_device on the torch API."""
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.evaluate import evaluate_vec_device
    g = P.load("c1_eval")
    H, W, M, num_envs, episodes, seed, pol_seed = (int(x) for x in g[f"{name}_cfg"])
    want = json.loads(str(g[f"{name}_metrics"]))
    queues = [deque() for _ in range(num_envs)]
    for i, bits in zip(g[f"{name}_layout_env"], P.unpack(g[f"{name}_layout_bits"], H * W)):
        queues[int(i)].append(bits)

    class ReplayVec(m.VecMinesweeper):
        def step(self, actions, out=None, want_infos=True):
            fresh = self._meta[:, 0].cpu().numpy() == 0
            mine = np.zeros((self.num_envs, self.HW), bool)
            for i in np.flatnonzero(fresh):
                mine[i] = queues[i].popleft()
            self.inject_layouts(mine, fresh)
            return super().step(actions, out=out, want_infos=want_infos)

    cfg = m.EnvConfig(H=H, W=W, mine_count=M, step_penalty=1e-4)
    model = P.scripted_policy(H, W, seed=pol_seed).cuda()
    got = evaluate_vec_device(model, cfg, episodes=episodes, seed=seed, num_envs=num_envs, vec_factory=ReplayVec)
    assert all(len(q) == 0 for q in queues), "the replay must consume exactly the layouts the reference drew"
    # the reference dict has no subset-rule keys; belief_* to 1e-6: CPU vs GPU sigmoid differ in the last ulp
    _assert_same_dict({k: got[k] for k in want}, want, belief_tol=1e-6)


@pytest.mark.parametrize("H,W,M,num_envs,episodes,max_steps", [
    (16, 16, 40, 1024, 4096, 512),
    (16, 30, 99, 512, 512, 512),
    (9, 9, 10, 64, 150, 8),                 # partial last batch (150 = 2 x 64 + 22) and the step cutoff
])
def test_device_eval_equals_host_eval(H, W, M, num_envs, episodes, max_steps):
    """Same seed, no injection: both evaluators draw the same Philox boards and must return the same dict."""
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.evaluate import evaluate_vec, evaluate_vec_device
    cfg = m.EnvConfig(H=H, W=W, mine_count=M, step_penalty=1e-4)
    model = P.scripted_policy(H, W, seed=3).cuda()
    kw = dict(episodes=episodes, seed=11, num_envs=num_envs, max_steps_per_episode=max_steps)
    want = evaluate_vec(model, cfg, **kw)
    got = evaluate_vec_device(model, cfg, **kw)
    _assert_same_dict(got, want)
    assert got["episodes"] == episodes and got["avg_steps"] > 1.0


def test_device_eval_equals_host_eval_cnn():
    """The random-init medium CNN in fp32 with deterministic cuDNN: the same logits feed both argmaxes."""
    import torch
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.evaluate import evaluate_vec, evaluate_vec_device
    torch.manual_seed(0)
    model = m.build_model("cnn_residual", obs_shape=(10, 16, 16),
                          model_cfg=dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256)).cuda()
    cfg = m.EnvConfig(H=16, W=16, mine_count=40, step_penalty=1e-4)
    det, bench = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        want = evaluate_vec(model, cfg, episodes=512, seed=2, num_envs=256)
        got = evaluate_vec_device(model, cfg, episodes=512, seed=2, num_envs=256)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = det, bench
    _assert_same_dict(got, want)
    assert model.training                                   # restored after the evaluation


def test_device_eval_reproducible_and_budget_error():
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.evaluate import evaluate_vec_device
    cfg = m.EnvConfig(H=16, W=16, mine_count=40, step_penalty=1e-4)
    model = P.scripted_policy(16, 16, seed=1).cuda()
    a = evaluate_vec_device(model, cfg, episodes=700, seed=5, num_envs=256)
    b = evaluate_vec_device(model, cfg, episodes=700, seed=5, num_envs=256)
    _assert_same_dict(a, b)
    assert a["forced_guess_rate"] > 0.0                      # the exact search ran on some analysed state
    with pytest.raises(RuntimeError, match="exceeded its step budget"):
        evaluate_vec_device(model, cfg, episodes=700, seed=5, num_envs=256, search_budget=1)


@pytest.mark.parametrize("A", [64, 81, 256, 480, 1024])
def test_masked_argmax_matches_torch(A):
    import torch
    from minesweeper_ppo_b200.evaluate import masked_argmax
    g = torch.Generator(device="cuda").manual_seed(A)
    n = 1001
    logits = torch.randint(-4, 4, (n, A), device="cuda", generator=g).float()      # many ties
    mask = torch.rand((n, A), device="cuda", generator=g) < 0.3
    logits[10, 7] = float("nan"); logits[10, A - 2] = float("nan"); mask[10, 7] = mask[10, A - 2] = True
    logits[11, 3] = float("nan"); mask[11, 3] = False                               # masked NaN is filled, loses
    logits[12] = -3e9; mask[12, :A // 2] = True; mask[12, A // 2:] = False           # legal below -1e9: masked wins
    logits[13] = float("-inf"); mask[13] = True                                     # all -inf: first index
    mask[14] = False; mask[n - 1] = False                                           # all-masked: the guard
    logits[15] = float("nan"); mask[15] = False                                     # all-masked NaN row
    logits[16, 0] = -0.0; logits[16, 1] = 0.0; logits[16, 2:] = -5; mask[16] = True  # -0 == +0: first index
    ref_mask = mask.clone()
    ref_mask[~ref_mask.any(dim=1)] = True
    want = logits.masked_fill(~ref_mask, -1e9).argmax(dim=-1)
    got = masked_argmax(logits, mask)
    assert got.dtype == torch.int32
    assert torch.equal(got.long(), want), torch.nonzero(got.long() != want)[:5].tolist()
    assert torch.equal(mask, ref_mask), "the empty-row guard must be written back to the mask"
    assert int(got[10]) == 7 and int(got[12]) == A // 2 and int(got[13]) == 0 and int(got[16]) == 0


def _window(torch, shape, dtype, fill=0x5A):
    nb = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    raw = torch.full((PAD + nb + PAD,), fill, dtype=torch.uint8, device="cuda")
    return raw, raw[PAD:PAD + nb].view(dtype).view(*shape), nb


def _intact(raw, nb, fill=0x5A):
    return bool((raw[:PAD] == fill).all()) and bool((raw[PAD + nb:] == fill).all())


@pytest.mark.parametrize("H,W,M,n", [(16, 16, 40, 37), (16, 30, 99, 19), (5, 7, 6, 33), (32, 32, 200, 5)])
def test_eval_kernel_outputs_stay_inside_their_windows(H, W, M, n):
    """Every buffer msw_masked_argmax / msw_eval_pre_step / msw_eval_post_step write is a window in a
    canary-filled allocation; a short evaluation runs on them and the canaries must be untouched."""
    import torch
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200 import _lib
    from minesweeper_ppo_b200.evaluate import _DeviceEvaluator, _INT64_MAX, _K, masked_argmax
    cfg = m.EnvConfig(H=H, W=W, mine_count=M, step_penalty=1e-4)
    vec = m.VecMinesweeper(n, cfg, seed=3, api="torch")
    model = P.scripted_policy(H, W, seed=0).cuda()
    ev = _DeviceEvaluator(model, vec, search_budget=0, max_steps=6)
    wins = {}
    for name in ("actions", "sel", "counted", "ep_unavoidable", "step_counter", "counters", "finished"):
        t = getattr(ev, name)
        wins[name] = _window(torch, tuple(t.shape), t.dtype)
        wins[name][1].copy_(t)
        setattr(ev, name, wins[name][1])
    ev.counters[_K["error_key"]] = _INT64_MAX
    remaining = 2 * n - 3
    while remaining > 0:
        bs = min(n, remaining)
        ev.new_batch()
        while ev.run_step(bs) < bs:
            pass
        remaining -= bs
    ev.check_budget()
    torch.cuda.synchronize()
    for k, (raw, view, nb) in wins.items():
        assert _intact(raw, nb), f"{k} window overrun at {H}x{W} n={n}"
    c = dict(zip(_lib.EVAL_COUNTERS, ev.counters.cpu().tolist()))
    assert c["total_steps"] > 0 and c["guess_attempts"] + c["forced_steps"] > 0
    # msw_masked_argmax with an odd A and a ragged n
    A = H * W
    ra, a, na = _window(torch, (n,), torch.int32)
    rm, mk, nm = _window(torch, (n, A), torch.bool)
    mk.copy_(torch.rand((n, A), device="cuda") < 0.5)
    masked_argmax(torch.randn((n, A), device="cuda"), mk, out=a)
    torch.cuda.synchronize()
    assert _intact(ra, na) and _intact(rm, nm)
    assert int(a.min()) >= 0 and int(a.max()) < A
