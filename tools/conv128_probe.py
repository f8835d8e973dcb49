"""The 128-channel tcgen05 trunk (conv3x3_pair_kernel) against the library trunk (cuDNN fp16 NHWC convolution +
msw_gn_act), at the size of a C3 rollout forward (8,192 boards), for the default residual model
(build_model("cnn_residual"): 128 channels, 8 groups, 6 blocks).

    python tools/conv128_probe.py [--out PATH] [--boards 8192] [--reps 20] [--rollout-steps 128]

Prints and writes one JSON document:
  * per layer kind (stem, EPI 0 = no residual + Dropout2d, EPI 1 = residual in + fp32 out, EPI 2 = residual in +
    pooled out): microseconds per launch of both paths, inputs alternating between two sets larger than L2, and
    the achieved rate against the larger of FLOP / 2,250 TFLOP/s and bytes / 7.7 TB/s (B200 data-sheet dense
    fp16 rate and HBM bandwidth; algorithmic bytes, counted below);
  * the whole forward (13 convolutions + heads) of both trunks, with their outputs compared at that size;
  * RolloutCollector(graph=True) frames/s at boards x rollout-steps with both trunks;
  * the GPU's name, power limit and max SM clock, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

PEAK_FLOPS, PEAK_BW = 2250e12, 7.7e12


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return {"query": q, "nvidia_smi": r.stdout.strip().splitlines()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--boards", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rollout-steps", type=int, default=128)
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.fused_forward import FusedRolloutForward, conv3x3_gn, conv3x3_taps, gn_act

    torch.backends.cudnn.benchmark = True
    n, C, reps = args.boards, 128, args.reps
    res = {"gpu": gpu_info(), "boards": n}

    def timed(fn):
        for i in range(4):
            fn(i & 1)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(i & 1)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / reps

    # ---- per layer
    g = torch.Generator(device="cuda").manual_seed(0)
    cl = torch.channels_last
    x16 = [torch.randn((n, C, 16, 16), device="cuda", generator=g).half().contiguous(memory_format=cl) for _ in range(2)]
    obs16 = [torch.randn((n, 16, 16, 16), device="cuda", generator=g).half().contiguous(memory_format=cl) for _ in range(2)]
    r_p8 = [torch.randn((n * C * 256,), device="cuda", generator=g) for _ in range(2)]
    r_nhwc = [torch.randn((n, C, 16, 16), device="cuda", generator=g).contiguous(memory_format=cl) for _ in range(2)]
    w = (torch.randn((C, C, 3, 3), device="cuda", generator=g) / (9 * C) ** 0.5).half()
    w_stem = (torch.randn((C, 16, 3, 3), device="cuda", generator=g) / (9 * 16) ** 0.5).half()
    taps, taps_stem = conv3x3_taps(w), conv3x3_taps(w_stem)
    w_cl, ws_cl = w.contiguous(memory_format=cl), w_stem.contiguous(memory_format=cl)
    bias = 0.1 * torch.randn((C,), device="cuda", generator=g)
    norm = torch.nn.GroupNorm(8, C).cuda()
    pool = torch.empty((n, C), device="cuda")
    act16, act32 = n * 256 * C * 2, n * 256 * C * 4
    flop_layer, flop_stem = 2.0 * n * 256 * C * C * 9, 2.0 * n * 256 * C * 16 * 9
    layers = [
        # name, FLOP, algorithmic HBM bytes, tcgen05 path, library path
        ("stem", flop_stem, n * 256 * 16 * 2 + act16 + act32,
         lambda i: conv3x3_gn(obs16[i], taps_stem, norm, bias, want32=True),
         lambda i: gn_act(F.conv2d(obs16[i], ws_cl, None, padding=1), norm, conv_bias=bias, want32=True)),
        ("epi0", flop_layer, 2 * act16,
         lambda i: conv3x3_gn(x16[i], taps, norm, bias, drop_p=0.05, seed=1, call_id=i),
         lambda i: gn_act(F.conv2d(x16[i], w_cl, None, padding=1), norm, conv_bias=bias, drop_p=0.05, seed=1, call_id=i)),
        ("epi1", flop_layer, 2 * act16 + 2 * act32,
         lambda i: conv3x3_gn(x16[i], taps, norm, bias, res32=r_p8[i], want32=True),
         lambda i: gn_act(F.conv2d(x16[i], w_cl, None, padding=1), norm, conv_bias=bias, res32=r_nhwc[i], want32=True)),
        ("epi2", flop_layer, 2 * act16 + act32,
         lambda i: conv3x3_gn(x16[i], taps, norm, bias, res32=r_p8[i], want_pool=True),
         lambda i: gn_act(F.conv2d(x16[i], w_cl, None, padding=1), norm, conv_bias=bias, res32=r_nhwc[i], want32=False,
                          pool32=pool)),
    ]
    res["layers"] = {}
    for name, flop, nbytes, tc, lib in layers:
        bound_us = max(flop / PEAK_FLOPS, nbytes / PEAK_BW) * 1e6
        row = {"flop": flop, "hbm_bytes": nbytes, "bound_us": bound_us,
               "bound_by": "tensor rate" if flop / PEAK_FLOPS > nbytes / PEAK_BW else "HBM bandwidth"}
        for kind, fn in (("tcgen05", tc), ("library", lib)):
            us = timed(fn)
            row[kind] = {"us": us, "tflops": flop / us / 1e6, "gb_per_s": nbytes / us / 1e3, "share_of_bound": bound_us / us}
        res["layers"][name] = row
        print(name, json.dumps(row), flush=True)
    del x16, obs16, r_p8, r_nhwc
    torch.cuda.empty_cache()

    # ---- whole forward of the default model
    torch.manual_seed(0)
    model = m.build_model("cnn_residual", obs_shape=(10, 16, 16)).cuda().eval()
    ff = FusedRolloutForward(model)
    assert ff.tc_trunk
    obs = [(torch.rand((n, 10, 16, 16), device="cuda", generator=g) < 0.3).float() for _ in range(2)]
    with torch.no_grad():
        tc_fwd = lambda i: ff._heads(*ff._trunk_tc(obs[i], 1 << 8), True)
        lib_fwd = lambda i: ff._heads(*ff._trunk_library(obs[i], 1 << 8), True)
        a, b = tc_fwd(0), lib_fwd(0)
        cmp = {}
        for u, v, name in zip(a, b, ("logits", "value", "mine")):
            cmp[name] = {"max_abs_diff": float((u.float() - v.float()).abs().max()), "scale": float(v.float().abs().max())}
        n_conv = 1 + 2 * len(model.residual_stack)
        flop_fwd = flop_stem + (n_conv - 1) * flop_layer
        res["forward"] = {"convolutions": n_conv, "conv_flop": flop_fwd, "tcgen05_ms": timed(tc_fwd) / 1e3,
                          "library_ms": timed(lib_fwd) / 1e3, "outputs_tcgen05_vs_library": cmp}
    print("forward", json.dumps(res["forward"]), flush=True)
    del ff, obs, model
    torch.cuda.empty_cache()

    # ---- rollout: RolloutCollector(graph=True) with the default model, both trunks
    T = args.rollout_steps
    cfg = m.EnvConfig(H=16, W=16, mine_count=40, guarantee_safe_neighborhood=True, step_penalty=1e-4)
    res["rollout"] = {"envs": n, "steps": T}
    for kind in ("tcgen05", "library"):
        torch.manual_seed(0)
        vec = m.VecMinesweeper(n, cfg, seed=0, api="torch")
        model = m.build_model("cnn_residual", obs_shape=(10, 16, 16)).cuda()
        col = m.RolloutCollector(vec, T, aux_maps=True, graph=True)
        fwd = FusedRolloutForward(model, seed=col.sample_seed, sample_id_base=vec._desc.env_id_base)
        fwd.epoch = col._epoch
        fwd.tc_trunk = kind == "tcgen05"
        col._fused_fwd = fwd
        times = []
        for i in range(3):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            col.collect(model)
            e1.record()
            torch.cuda.synchronize()
            if i >= 1:
                times.append(e0.elapsed_time(e1))
        ms = sum(times) / len(times)
        res["rollout"][kind] = {"ms_rollout": ms, "frames_per_s": n * T / (ms / 1e3)}
        print("rollout", kind, json.dumps(res["rollout"][kind]), flush=True)
        del col, vec, model, fwd
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
