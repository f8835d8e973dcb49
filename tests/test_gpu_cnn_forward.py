"""The baseline policy's rollout forward (msw_cnn_fwd.cu: cnn_fwd_kernel, msw_cnn_forward) and
fused_forward.FusedCnnForward on build_model("cnn").  Needs a B200."""
import os

import numpy as np
import pytest

import parity as P

pytestmark = pytest.mark.gpu
PAD = 4096          # canary bytes on each side of an output window


def _params(torch, seed):
    """Random fp16 tap-major weights, fp16-valued biases (as autocast casts them) and GroupNorm affines."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    taps = []
    for cout, cin in ((32, 16), (64, 32), (64, 64)):
        taps.append((torch.randn((9, cout, cin), device="cuda", generator=g) / (9 * cin) ** 0.5).half())
    r = lambda n, s: (s * torch.randn((n,), device="cuda", generator=g)).half().float()
    u = lambda n, lo, hi: lo + (hi - lo) * torch.rand((n,), device="cuda", generator=g)
    vecs = (r(32, 0.2), u(32, 0.5, 1.5), u(32, -0.3, 0.3), r(64, 0.2), u(64, 0.5, 1.5), u(64, -0.3, 0.3), r(64, 0.2))
    heads = (torch.randn((2, 64), device="cuda", generator=g) / 8).half()
    hb = (0.1 * torch.randn((2,), device="cuda", generator=g)).half()
    return taps, vecs, heads, hb


def _restated(torch, x16, taps, vecs, heads, hb, eps=(1e-5, 1e-5)):
    """The kernel's formula in plain torch fp32 with the same fp16 rounding points."""
    import torch.nn.functional as F
    b1, g1, be1, b2, g2, be2, b3 = vecs
    w = lambda t: t.float().reshape(3, 3, t.shape[1], t.shape[2]).permute(2, 3, 0, 1)
    col = lambda v: v.view(1, -1, 1, 1)
    c1 = (F.conv2d(x16.float(), w(taps[0]), padding=1) + col(b1)).half()
    a1 = F.group_norm(torch.relu(c1).float(), 4, g1, be1, eps[0]).half()
    c2 = (F.conv2d(a1.float(), w(taps[1]), padding=1) + col(b2)).half()
    a2 = F.group_norm(torch.relu(c2).float(), 8, g2, be2, eps[1]).half()
    f = torch.relu((F.conv2d(a2.float(), w(taps[2]), padding=1) + col(b3)).half())
    n = x16.shape[0]
    pol = (torch.einsum("nchw,c->nhw", f.float(), heads[0].float()) + hb[0].float()).half().reshape(n, 256)
    mine = (torch.einsum("nchw,c->nhw", f.float(), heads[1].float()) + hb[1].float()).half().reshape(n, 256)
    pooled = f.float().mean(dim=(2, 3)).half()
    return pol, mine, pooled


def _x16(torch, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn((n, 16, 16, 16), device="cuda", generator=g).half().contiguous(memory_format=torch.channels_last)


def _close(got, want, what):
    # fp32 accumulation in a different order flips an fp16 rounding now and then (one ulp at that point); the flip
    # passes through GroupNorm and the next convolutions, so the outputs differ by a few fp16 ulps of their scale
    # at a few positions, and by far less on average.
    scale = float(want.float().abs().max()) + 1e-3
    d = (got.float() - want.float()).abs()
    assert float(d.max()) <= 1e-2 * scale, (what, float(d.max()), scale)
    assert float(d.mean()) <= 5e-4 * scale, (what, float(d.mean()), scale)


@pytest.mark.parametrize("n", [1, 3, 149, 301])
def test_cnn_forward_matches_torch_fp32(n):
    """msw_cnn_forward on random fp16 inputs vs the torch fp32 restatement of its formula; n = 301 is more boards
    than CTAs, n = 3 leaves a CTA's second slot idle.  Bitwise reproducible."""
    import torch
    from minesweeper_ppo_b200.fused_forward import cnn_forward
    torch.backends.cudnn.allow_tf32 = False
    x = _x16(torch, n, n)
    taps, vecs, heads, hb = _params(torch, 7)
    got = cnn_forward(x, taps, vecs, heads, hb, (1e-5, 1e-5))
    again = cnn_forward(x, taps, vecs, heads, hb, (1e-5, 1e-5))
    assert all(torch.equal(a, b) for a, b in zip(got, again)), "bitwise reproducible"
    want = _restated(torch, x, taps, vecs, heads, hb)
    for a, b, what in zip(got, want, ("logits", "mine", "pooled")):
        assert a.shape == b.shape and a.dtype == torch.float16, what
        _close(a, b, what)


@pytest.mark.parametrize("layer", [0, 1, 2])
def test_cnn_forward_one_hot_taps(layer):
    """Each tap of each layer alone, as one-hot weights (output channel co reads input channel co % Cin), the other
    layers random: checks the shifted descriptors, the edge masks at x = 0 / 15 and the zero halo rows at y = 0 / 15
    of that layer's operand."""
    import torch
    from minesweeper_ppo_b200.fused_forward import cnn_forward
    torch.backends.cudnn.allow_tf32 = False
    n = 5
    x = _x16(torch, n, 11)
    taps, vecs, heads, hb = _params(torch, 3)
    cout, cin = taps[layer].shape[1], taps[layer].shape[2]
    for k in range(9):
        t = list(taps)
        one = torch.zeros_like(taps[layer])
        one[k, torch.arange(cout), torch.arange(cout) % cin] = 1.0
        t[layer] = one
        got = cnn_forward(x, t, vecs, heads, hb, (1e-5, 1e-5))
        want = _restated(torch, x, t, vecs, heads, hb)
        for a, b, what in zip(got, want, ("logits", "mine", "pooled")):
            _close(a, b, f"layer {layer} tap {k} {what}")


def _observations(torch, m, n, seed, steps=8):
    """Observations and action masks of real VecMinesweeper states after a few random moves."""
    cfg = m.EnvConfig(H=16, W=16, mine_count=40, step_penalty=1e-4)
    vec = m.VecMinesweeper(n, cfg, seed=seed, api="torch")
    o = vec._alloc_encode()
    vec.reset(out=o)
    for t in range(steps):
        vec.step(vec.random_actions(t), out=o, want_infos=False)
    return o.obs.clone(), o.action_mask.clone()


@pytest.mark.parametrize("hidden", [64, 256])
def test_fused_cnn_forward_matches_autocast_module(hidden):
    """FusedCnnForward vs build_model("cnn") under fp16 autocast on real env states, at n in {1, 3, 148, 149, 8192}
    (one board, fewer boards than CTAs, a full wave, a partial second wave, many boards per CTA)."""
    import torch
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.fused_forward import FusedCnnForward
    torch.manual_seed(hidden)
    net = m.build_model("cnn", obs_shape=(10, 16, 16), model_cfg={"hidden": hidden}).cuda().eval()
    with torch.no_grad():                                    # non-trivial GroupNorm affines
        for mod in net.modules():
            if isinstance(mod, torch.nn.GroupNorm):
                mod.weight.uniform_(0.5, 1.5); mod.bias.uniform_(-0.3, 0.3)
    ff = FusedCnnForward(net)
    obs_all, mask_all = _observations(torch, m, 8192, seed=hidden)
    for n in (1, 3, 148, 149, 8192):
        obs, mask = obs_all[:n].contiguous(), mask_all[:n]
        assert ff.fused_input(obs)
        got = ff(obs, return_mine=True)
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            ref = net(obs, return_mine=True)
        for a, b, name in zip(got, ref, ("logits", "value", "mine")):
            assert a.shape == b.shape and a.dtype == b.dtype == torch.float16, (n, name, a.shape, b.shape, a.dtype)
            # cuDNN and the kernel sum in different orders and round at the same points: a few fp16 ulps of the
            # output's scale (the tolerance test_gpu_conv128 uses for the residual model against autocast)
            err = float((a.float() - b.float()).abs().max())
            scale = float(b.float().abs().max()) + 1e-3
            assert err <= 2e-2 * scale, (n, name, err, scale)
        # the greedy action over the masked logits: rows whose top two legal logits are within a rounding of each
        # other may pick differently; allow 0.5 % of rows (at least one)
        fill = torch.finfo(torch.float16).min
        ga = got[0].masked_fill(~mask, fill).argmax(dim=1)
        gb = ref[0].masked_fill(~mask, fill).argmax(dim=1)
        assert int((ga != gb).sum()) <= max(1, n // 200), (n, int((ga != gb).sum()))


def test_fused_cnn_forward_bitwise_and_independent_of_n():
    """Two calls give identical bytes; a board's outputs do not depend on how many boards are in the call or on
    which CTA / slot ran it."""
    import torch
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.fused_forward import FusedCnnForward
    torch.manual_seed(1)
    net = m.build_model("cnn", obs_shape=(10, 16, 16)).cuda().eval()
    ff = FusedCnnForward(net)
    obs, _ = _observations(torch, m, 1000, seed=5)
    full = ff(obs, return_mine=True)
    again = ff(obs, return_mine=True)
    assert all(torch.equal(a, b) for a, b in zip(full, again))
    for lo, hi in ((0, 1), (7, 10), (148, 300), (999, 1000)):
        part = ff(obs[lo:hi].contiguous(), return_mine=True)
        for a, b in zip(part, full):
            assert torch.equal(a, b[lo:hi]), (lo, hi)


def test_fused_cnn_forward_other_inputs_run_the_autocast_module():
    """Non-16x16 boards (and non-fp32 / non-contiguous observations) run the module under fp16 autocast."""
    import torch
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.fused_forward import FusedCnnForward
    torch.manual_seed(2)
    net = m.build_model("cnn", obs_shape=(10, 16, 30)).cuda().eval()
    ff = FusedCnnForward(net)
    obs = (torch.rand((4, 10, 16, 30), device="cuda") < 0.3).float()
    assert not ff.fused_input(obs)
    got = ff(obs, return_mine=True)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        ref = net(obs, return_mine=True)
    assert all(torch.equal(a, b) for a, b in zip(got, ref))
    half = (torch.rand((4, 10, 16, 16), device="cuda") < 0.3).half()
    assert not ff.fused_input(half)


def test_graph_captured_rollout_cnn(oracle):
    """RolloutCollector(graph=True) with build_model("cnn") captures and replays; replaying the recorded actions
    through the oracle reproduces every env-written buffer field bit for bit."""
    import torch
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.fused_forward import FusedCnnForward
    torch.manual_seed(0)
    N, T = 128, 16
    cfg = m.EnvConfig(H=16, W=16, mine_count=40, step_penalty=1e-4)
    vec = m.VecMinesweeper(N, cfg, seed=2, api="torch")
    model = m.build_model("cnn", obs_shape=(10, 16, 16)).cuda()
    assert m.RolloutCollector.can_graph(model)
    col = m.RolloutCollector(vec, T, aux_maps=True, sample_seed=3, graph=True)
    b1, _ = col.collect(model)
    torch.cuda.synchronize()
    assert isinstance(col._fused_fwd, FusedCnnForward)
    a1, v1 = b1.actions.clone(), b1.values.clone()
    ep = vec.state_tensors["meta"][:, 2].cpu().numpy().astype(np.uint32)
    with torch.no_grad():
        for p_ in model.parameters():
            p_.mul_(1.01)
    b2, aux = col.collect(model)
    torch.cuda.synchronize()
    assert not torch.equal(a1, b2.actions) and not torch.equal(v1, b2.values)
    c = lambda t_: t_.cpu().numpy()
    ref = oracle.OracleVecEnv(N, cfg, seed=2, nthreads=os.cpu_count() or 1, aux_maps=True)
    ref.episode_idx[:] = ep
    b = ref.reset()
    obs, mask, lab = b["obs"], b["action_mask"], ref.mine_labels
    acts = c(b2.actions).reshape(T, N)
    for t in range(T):
        s = slice(t * N, (t + 1) * N)
        P.assert_bits_equal(c(b2.obs[s]), obs, f"slot {t} obs")
        P.assert_bits_equal(c(b2.action_mask[s]), mask, f"slot {t} mask")
        P.assert_bits_equal(c(b2.mine_labels[s]), lab, f"slot {t} labels")
        assert mask[np.arange(N), acts[t]].all()
        bb, r, d, _ = ref.step(acts[t], tensor_infos=True)
        P.assert_bits_equal(c(b2.rewards[s]), r, f"slot {t} rewards")
        P.assert_bits_equal(c(b2.dones[s]), d, f"slot {t} dones")
        obs, mask, lab = bb["obs"], bb["action_mask"], ref.mine_labels
    assert aux["last_values"].shape == (N,)


@pytest.mark.parametrize("graph", [False, True])
def test_expert_board_cnn_rollout_runs_through_the_module(graph):
    """A 16x30 cnn rollout still runs (the autocast module inside FusedCnnForward), with and without capture."""
    import torch
    import minesweeper_ppo_b200 as m
    torch.manual_seed(0)
    N, T = 64, 6
    cfg = m.EnvConfig(H=16, W=30, mine_count=99, step_penalty=1e-4)
    vec = m.VecMinesweeper(N, cfg, seed=4, api="torch")
    model = m.build_model("cnn", obs_shape=(10, 16, 30)).cuda()
    col = m.RolloutCollector(vec, T, aux_maps=True, sample_seed=1, graph=graph)
    buf, aux = col.collect(model)
    buf, aux = col.collect(model)
    torch.cuda.synchronize()
    assert aux["last_values"].shape == (N,) and bool(torch.isfinite(buf.values).all())
    acts = buf.actions.view(T, N)
    assert bool((acts >= 0).all()) and bool((acts < 16 * 30).all())


def _window(torch, shape, dtype, fill=0x5A):
    nbytes = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    raw = torch.full((PAD + nbytes + PAD,), fill, dtype=torch.uint8, device="cuda")
    return raw, raw[PAD:PAD + nbytes].view(dtype).view(*shape), nbytes


def _intact(raw, nbytes, fill=0x5A):
    return bool((raw[:PAD] == fill).all()) and bool((raw[PAD + nbytes:] == fill).all())


def _call(L, torch, x, taps, vecs, heads, hb, lg, mn, pl, n, H=16, W=16, cin=16, c1=32, g1=4, c2=64, g2=8, c3=64):
    b1, g1v, be1, b2, g2v, be2, b3 = vecs
    return L.msw_cnn_forward(x.data_ptr(), taps[0].data_ptr(), b1.data_ptr(), g1v.data_ptr(), be1.data_ptr(),
                             taps[1].data_ptr(), b2.data_ptr(), g2v.data_ptr(), be2.data_ptr(), taps[2].data_ptr(),
                             b3.data_ptr(), heads[0].data_ptr(), hb[0:1].data_ptr(), heads[1].data_ptr(),
                             hb[1:2].data_ptr(), lg, mn, pl, n, H, W, cin, c1, g1, c2, g2, c3, 1e-5, 1e-5,
                             torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("n", [1, 37, 149])
def test_cnn_forward_outputs_stay_inside_their_windows(n):
    import torch
    from minesweeper_ppo_b200 import _lib
    L = _lib.load()
    x = _x16(torch, n, n)
    taps, vecs, heads, hb = _params(torch, 1)
    rl, lg, nl = _window(torch, (n, 256), torch.float16)
    rm, mn, nm = _window(torch, (n, 256), torch.float16)
    rp, pl, npl = _window(torch, (n, 64), torch.float16)
    assert _call(L, torch, x, taps, vecs, heads, hb, lg.data_ptr(), mn.data_ptr(), pl.data_ptr(), n) == 0
    torch.cuda.synchronize()
    assert _intact(rl, nl) and _intact(rm, nm) and _intact(rp, npl)
    assert bool(torch.isfinite(lg).all()) and bool(torch.isfinite(mn).all()) and bool(torch.isfinite(pl).all())


def test_cnn_forward_shape_errors():
    """Every shape but 16x16, Cin 16, widths 32 / 64 / 64 and groups 4 / 8 is MSW_ERR_BAD_SHAPE (1) with a message."""
    import torch
    from minesweeper_ppo_b200 import _lib
    L = _lib.load()
    n = 2
    x = _x16(torch, n, 0)
    taps, vecs, heads, hb = _params(torch, 0)
    out = torch.zeros((3, n, 256), dtype=torch.float16, device="cuda")
    ptrs = (out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr())
    for bad in (dict(H=8), dict(W=30), dict(cin=10), dict(c1=64), dict(g1=8), dict(c2=128), dict(g2=4), dict(c3=32)):
        assert _call(L, torch, x, taps, vecs, heads, hb, *ptrs, n, **bad) == 1, bad
        assert b"msw_cnn_forward" in L.msw_last_error(), bad
    assert _call(L, torch, x, taps, vecs, heads, hb, *ptrs, -1) == 1
    assert _call(L, torch, x, taps, vecs, heads, hb, *ptrs, n) == 0
    torch.cuda.synchronize()
