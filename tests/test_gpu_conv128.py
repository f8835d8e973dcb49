"""The 128-channel tcgen05 trunk (msw_conv_tc.cu, conv3x3_pair_kernel: one board per 2-CTA cluster) -- the shape of
the package's default residual model, build_model("cnn_residual") -- and FusedRolloutForward on that model.
Needs a B200."""
import os

import numpy as np
import pytest

import parity as P

pytestmark = pytest.mark.gpu
C = 128
PAD = 4096          # canary bytes on each side of an output window


@pytest.mark.parametrize("n,cin", [(1, 128), (5, 128), (301, 128), (1, 16), (5, 16), (301, 16)])
def test_conv3x3_c128_matches_cudnn(n, cin):
    """msw_conv3x3 at C = 128 vs cuDNN (both fp32 accumulation, one fp16 rounding), every tap alone with one-hot
    weights (exact: catches a wrong descriptor, shift or mask of either CTA of the pair), bitwise reproducible.
    n = 301 is more boards than there are clusters."""
    import torch
    import torch.nn.functional as F
    from minesweeper_ppo_b200.fused_forward import conv3x3, conv3x3_taps
    g = torch.Generator(device="cuda").manual_seed(n + cin)
    x = torch.randn((n, cin, 16, 16), device="cuda", generator=g).half().contiguous(memory_format=torch.channels_last)
    w = (torch.randn((C, cin, 3, 3), device="cuda", generator=g) / (9 * cin) ** 0.5).half()
    got = conv3x3(x, conv3x3_taps(w))
    again = conv3x3(x, conv3x3_taps(w))
    assert torch.equal(got, again)
    want = F.conv2d(x, w.contiguous(memory_format=torch.channels_last), None, padding=1)
    exact = F.conv2d(x.float(), w.float(), None, padding=1)
    err, ref_err = float((got.float() - exact).abs().max()), float((want.float() - exact).abs().max())
    assert got.shape == want.shape and got.dtype == torch.float16
    assert err <= max(2 * ref_err, 4e-3), (err, ref_err)            # as close to the fp32 result as cuDNN is
    for ky in range(3):
        for kx in range(3):
            w1 = torch.zeros((C, cin, 3, 3), device="cuda", dtype=torch.float16)
            # output channel co reads input channel co % cin: every output channel of both weight halves is used
            w1[torch.arange(C), torch.arange(C) % cin, ky, kx] = 1.0
            one = conv3x3(x, conv3x3_taps(w1))
            ref = F.conv2d(x, w1.contiguous(memory_format=torch.channels_last), None, padding=1)
            assert torch.equal(one, ref), (ky, kx)


@pytest.mark.parametrize("n,cin,res,drop,pool", [(3, 128, False, 0.0, False), (300, 128, False, 0.25, False),
                                                 (149, 128, True, 0.0, False), (7, 128, True, 0.0, False),
                                                 (5, 128, True, 0.0, True), (301, 128, True, 0.0, True),
                                                 (37, 16, False, 0.0, False)])
def test_conv3x3_gn_c128_matches_torch_fp32(n, cin, res, drop, pool):
    """msw_conv3x3_gn at C = 128, G = 8 in every epilogue mode (stem, no residual, no residual + Dropout2d,
    residual -> y32, residual -> pool) vs the torch fp32 expression and vs msw_conv3x3 -> msw_gn_act, with the
    tolerances of test_gpu_rollout.test_conv3x3_gn_matches_torch_fp32."""
    import torch
    import torch.nn.functional as F
    from minesweeper_ppo_b200.fused_forward import conv3x3, conv3x3_gn, conv3x3_taps, from_p8, gn_act, to_p8
    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator(device="cuda").manual_seed(n + cin)
    x = torch.randn((n, cin, 16, 16), device="cuda", generator=g).half().contiguous(memory_format=torch.channels_last)
    w = (torch.randn((C, cin, 3, 3), device="cuda", generator=g) / (9 * cin) ** 0.5).half()
    bias = 0.2 * torch.randn((C,), device="cuda", generator=g)
    norm = torch.nn.GroupNorm(8, C).cuda()
    with torch.no_grad():
        norm.weight.uniform_(0.5, 1.5); norm.bias.uniform_(-0.3, 0.3)
    r = torch.randn((n, C, 16, 16), device="cuda", generator=g) if res else None
    r_p8 = to_p8(r) if res else None
    assert not res or torch.equal(from_p8(r_p8), r)
    taps = conv3x3_taps(w)
    kw = dict(res32=r_p8, drop_p=drop, seed=5, call_id=77, sample_id_base=1000)
    got16, got2 = conv3x3_gn(x, taps, norm, bias, want32=not pool, want_pool=pool, **kw)
    again16, again2 = conv3x3_gn(x, taps, norm, bias, want32=not pool, want_pool=pool, **kw)
    assert torch.equal(got16, again16) and torch.equal(got2, again2), "bitwise reproducible"
    with torch.no_grad():
        conv16 = F.conv2d(x.float(), w.float(), None, padding=1).half()
        z = F.group_norm(conv16.float() + bias.view(1, C, 1, 1), 8, norm.weight, norm.bias, norm.eps)
        want32 = torch.relu(z + r if res else z)
    scale = float(want32.abs().max()) + 1.0
    if drop > 0:
        got32 = from_p8(got2)
        dropped = got32.abs().sum(dim=(2, 3)) == 0
        frac = float((dropped & (want32.abs().sum(dim=(2, 3)) > 0)).float().mean())
        assert 0.18 < frac < 0.32, frac
        want32 = torch.where(dropped[:, :, None, None], torch.zeros_like(want32), want32 / (1.0 - drop))
        scale = float(want32.abs().max()) + 1.0
    if pool:
        assert got2.shape == (n, C)
        assert float((got2 - want32.mean(dim=(2, 3))).abs().max()) <= 1e-3 * scale
    else:
        got32 = from_p8(got2)
        assert float((got32 - want32).abs().max()) <= 4e-3 * scale
        assert float((got32 - want32).abs().mean()) <= 2e-5 * scale
        assert torch.equal(got16, got32.half().contiguous(memory_format=torch.channels_last))
    assert float((got16.float() - want32).abs().max()) <= 5e-3 * scale
    # the unfused pair: the same fp16 conv output bit for bit, only the statistics' reduction order differs
    u16, u32 = gn_act(conv3x3(x, taps), norm, conv_bias=bias,
                      res32=(r.contiguous(memory_format=torch.channels_last) if res else None),
                      drop_p=drop, want32=True, seed=5, call_id=77, sample_id_base=1000)
    uscale = float(u32.abs().max()) + 1.0
    if pool:
        assert float((got2 - u32.mean(dim=(2, 3))).abs().max()) <= 2e-5 * uscale
    else:
        assert float((from_p8(got2) - u32).abs().max()) <= 2e-5 * uscale
        if drop > 0:
            assert torch.equal(from_p8(got2).abs().sum(dim=(2, 3)) == 0, u32.abs().sum(dim=(2, 3)) == 0)
    assert float((got16.float() - u16.float()).abs().max()) <= 2e-3 * uscale


def test_dropout_stream_c128_is_keyed_by_global_sample():
    import torch
    from minesweeper_ppo_b200.fused_forward import conv3x3_gn, conv3x3_taps
    g = torch.Generator(device="cuda").manual_seed(0)
    n = 64
    x = torch.randn((n, C, 16, 16), device="cuda", generator=g).half().contiguous(memory_format=torch.channels_last)
    w = (torch.randn((C, C, 3, 3), device="cuda", generator=g) / (9 * C) ** 0.5).half()
    bias = torch.zeros((C,), device="cuda")
    norm = torch.nn.GroupNorm(8, C).cuda()
    taps = conv3x3_taps(w)
    tail = x[40:].contiguous(memory_format=torch.channels_last)
    full, _ = conv3x3_gn(x, taps, norm, bias, drop_p=0.3, seed=1, call_id=2, sample_id_base=0)
    part, _ = conv3x3_gn(tail, taps, norm, bias, drop_p=0.3, seed=1, call_id=2, sample_id_base=40)
    assert torch.equal(full[40:], part)
    other, _ = conv3x3_gn(tail, taps, norm, bias, drop_p=0.3, seed=1, call_id=2, sample_id_base=0)
    assert not torch.equal(full[40:], other)


def _default_model(torch, m):
    torch.manual_seed(3)
    net = m.build_model("cnn_residual", obs_shape=(10, 16, 16)).cuda()
    with torch.no_grad():                                    # non-trivial affine parameters
        for mod in net.modules():
            if isinstance(mod, torch.nn.GroupNorm):
                mod.weight.uniform_(0.5, 1.5); mod.bias.uniform_(-0.3, 0.3)
    return net


def test_fused_forward_default_model(capfd):
    """FusedRolloutForward on build_model("cnn_residual") (128 channels, 8 groups, 6 blocks) takes the tcgen05
    trunk silently, matches the module under fp16 autocast and the library trunk, and is bitwise reproducible."""
    import torch
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.fused_forward import FusedRolloutForward
    net = _default_model(torch, m).eval()
    assert net.stem[0].out_channels == 128 and net.stem[1].num_groups == 8
    x = (torch.rand(300, 10, 16, 16, device="cuda") < 0.3).float()
    ff = FusedRolloutForward(net)
    assert ff.tc_trunk
    capfd.readouterr()
    got = ff(x, return_mine=True)
    again = ff(x, return_mine=True)
    torch.cuda.synchronize()
    assert capfd.readouterr().err == "", "the 128-channel shape must not be announced as a fallback"
    assert all(torch.equal(u, v) for u, v in zip(got, again)), "bitwise reproducible"
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        ref = net(x, return_mine=True)
    lib = ff._heads(*ff._trunk_library(x, 1 << 8), True)
    for a, b, c, name in zip(got, ref, lib, ("logits", "value", "mine")):
        assert a.shape == b.shape and a.dtype == torch.float16, name
        for other, what in ((b, "autocast"), (c, "library trunk")):
            err = float((a.float() - other.float()).abs().max())
            scale = float(other.float().abs().max()) + 1e-3
            assert err <= 2e-2 * scale, (name, what, err, scale)
    # with Dropout2d on (train mode) both trunks draw the same channels from the same stream
    net.train()
    ff2 = FusedRolloutForward(net, seed=4)
    _, pooled = ff2._trunk_tc(x, 5 << 8)
    _, bpooled = ff2._trunk_library(x, 5 << 8)
    assert float((pooled - bpooled).abs().max()) <= 2e-2 * (float(bpooled.abs().max()) + 1e-3)


def test_graph_captured_rollout_default_model(oracle):
    """RolloutCollector(graph=True) with the default model (whose forward is the 128-channel tcgen05 trunk):
    replaying the recorded actions through the oracle reproduces every env-written buffer field bit for bit."""
    import torch
    import minesweeper_ppo_b200 as m
    torch.manual_seed(0)
    N, T = 128, 16
    cfg = m.EnvConfig(H=16, W=16, mine_count=40, step_penalty=1e-4)
    vec = m.VecMinesweeper(N, cfg, seed=2, api="torch")
    model = m.build_model("cnn_residual", obs_shape=(10, 16, 16)).cuda()
    col = m.RolloutCollector(vec, T, aux_maps=True, sample_seed=3, graph=True)
    b1, _ = col.collect(model)
    torch.cuda.synchronize()
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


def _window(torch, shape, dtype, fill=0x5A):
    nbytes = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    raw = torch.full((PAD + nbytes + PAD,), fill, dtype=torch.uint8, device="cuda")
    return raw, raw[PAD:PAD + nbytes].view(dtype).view(*shape), nbytes


def _intact(raw, nbytes, fill=0x5A):
    return bool((raw[:PAD] == fill).all()) and bool((raw[PAD + nbytes:] == fill).all())


@pytest.mark.parametrize("n", [1, 37, 149])
def test_conv3x3_gn_c128_outputs_stay_inside_their_windows(n):
    import torch
    from minesweeper_ppo_b200 import _lib
    from minesweeper_ppo_b200.fused_forward import conv3x3_taps
    L = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cuda").manual_seed(n)
    x = torch.randn((n, C, 16, 16), device="cuda", generator=g).half().contiguous(memory_format=torch.channels_last)
    taps = conv3x3_taps((torch.randn((C, C, 3, 3), device="cuda", generator=g) / (9 * C) ** 0.5).half())
    bias = torch.zeros((C,), device="cuda")
    norm = torch.nn.GroupNorm(8, C).cuda()
    res = torch.randn((n * C * 256,), device="cuda", generator=g)
    ry16, y16, ny16 = _window(torch, (n, 16, 16, C), torch.float16)
    ry32, y32, ny32 = _window(torch, (n * C * 256,), torch.float32)
    rpl, pool, npl = _window(torch, (n, 8, C), torch.float32)

    def call(res32, y32p, poolp, drop):
        return L.msw_conv3x3_gn(x.data_ptr(), taps.data_ptr(), bias.data_ptr(), res32, norm.weight.data_ptr(),
                                norm.bias.data_ptr(), y16.data_ptr(), y32p, poolp, n, 16, 16, C, C, 8, 1e-5, drop,
                                1, 2, None, 0, 0, st)

    assert call(None, y32.data_ptr(), None, 0.2) == 0                  # EPI 0 with Dropout2d, y32 out
    assert call(res.data_ptr(), y32.data_ptr(), None, 0.0) == 0        # EPI 1
    assert call(res.data_ptr(), None, pool.data_ptr(), 0.0) == 0       # EPI 2
    torch.cuda.synchronize()
    assert _intact(ry16, ny16) and _intact(ry32, ny32) and _intact(rpl, npl)
    assert bool(torch.isfinite(pool).all()) and bool(torch.isfinite(y32).all())


def test_conv3x3_c128_shape_errors():
    """G != 8 at C = 128, Cin = 96 into C = 128 and H != 16 are MSW_ERR_BAD_SHAPE (1)."""
    import torch
    from minesweeper_ppo_b200 import _lib
    L = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    n = 2
    x = torch.zeros((n * 256 * C,), dtype=torch.float16, device="cuda")
    taps = torch.zeros((9 * C * C,), dtype=torch.float16, device="cuda")
    y = torch.zeros((n * 256 * C,), dtype=torch.float16, device="cuda")
    v = torch.ones((C,), device="cuda")

    def gn(H, cin, G):
        return L.msw_conv3x3_gn(x.data_ptr(), taps.data_ptr(), v.data_ptr(), None, v.data_ptr(), v.data_ptr(),
                                y.data_ptr(), None, None, n, H, 16, cin, C, G, 1e-5, 0.0, 0, 0, None, 0, 0, st)

    assert gn(16, C, 6) == 1
    assert gn(16, 96, 8) == 1
    assert gn(8, C, 8) == 1
    assert L.msw_conv3x3(x.data_ptr(), taps.data_ptr(), y.data_ptr(), n, 16, 16, 96, C, st) == 1
    assert L.msw_conv3x3(x.data_ptr(), taps.data_ptr(), y.data_ptr(), n, 16, 8, C, C, st) == 1
    assert gn(16, C, 8) == 0
    torch.cuda.synchronize()
