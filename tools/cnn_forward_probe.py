"""The baseline policy's rollout forward (build_model("cnn"): msw_pack_obs16 -> msw_cnn_forward -> value MLP in
torch fp16) against the module under fp16 autocast, and the rollout collector with both.

    python tools/cnn_forward_probe.py [--out PATH] [--boards 8192,65536] [--reps 20]

Prints and writes one JSON document:
  * per board count: microseconds of the msw_cnn_forward kernel alone (pre-packed input), of the whole fused
    forward (pack + kernel + value MLP) and of the autocast module on the same observations, the two forwards
    alternating in rounds within this process; two input sets alternate, each larger than the 126 MB L2 at 8,192
    boards; the kernel's achieved FLOP/s from the shape-derived count and its share of the larger of FLOP /
    2,250 TFLOP/s and bytes / 7.7 TB/s (B200 data-sheet dense fp16 rate and HBM bandwidth);
  * the fused outputs against the module's at that size;
  * RolloutCollector frames/s: graph=True (fused forward) against the eager module (fused=False, graph=False), at
    8,192 envs x 128 steps and 128 envs x 64 steps;
  * the GPU's name, power limit and max SM clock, read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

PEAK_FLOPS, PEAK_BW = 2250e12, 7.7e12
# per board: three 3x3 convolutions (conv1 at K = 16, the packed input) and the two 1x1 heads, 2 FLOP per MAC
FLOP_PER_BOARD = 2 * 256 * 9 * (16 * 32 + 32 * 64 + 64 * 64) + 2 * 2 * 256 * 64
# per board: the fp16 16-channel input in; fp16 logits, mine logits and pooled features out
BYTES_PER_BOARD = 256 * 16 * 2 + 2 * 256 * 2 + 64 * 2


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return {"query": q, "nvidia_smi": r.stdout.strip().splitlines()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--boards", default="8192,65536")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import minesweeper_ppo_b200 as m
    from minesweeper_ppo_b200.fused_forward import FusedCnnForward, cnn_forward

    torch.backends.cudnn.benchmark = True
    res = {"gpu": gpu_info(), "flop_per_board": FLOP_PER_BOARD, "hbm_bytes_per_board": BYTES_PER_BOARD, "forward": {}}

    def timed(fn, reps):
        for i in range(3):
            fn(i & 1)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(i & 1)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / reps

    torch.manual_seed(0)
    net = m.build_model("cnn", obs_shape=(10, 16, 16)).cuda().eval()
    ff = FusedCnnForward(net)
    eps = (net.backbone[2].eps, net.backbone[5].eps)
    g = torch.Generator(device="cuda").manual_seed(0)
    for n in (int(b) for b in args.boards.split(",")):
        obs = [(torch.rand((n, 10, 16, 16), device="cuda", generator=g) < 0.3).float() for _ in range(2)]
        x16 = [torch.zeros((n, 16, 16, 16), dtype=torch.float16, device="cuda").contiguous(memory_format=torch.channels_last)
               for _ in range(2)]
        for o, x in zip(obs, x16):
            x[:, :10].copy_(o)
        reps = max(3, args.reps * 8192 // n)
        with torch.no_grad():
            kern = lambda i: cnn_forward(x16[i], ff.taps, ff.vecs, ff.heads16, ff.head_bias16, eps)
            fused = lambda i: ff(obs[i], return_mine=True)

            def module(i):
                with torch.autocast("cuda", dtype=torch.float16):
                    return net(obs[i], return_mine=True)

            rounds = {"kernel_us": [], "fused_forward_us": [], "autocast_module_us": []}
            for _ in range(args.rounds):
                rounds["kernel_us"].append(timed(kern, reps))
                rounds["fused_forward_us"].append(timed(fused, reps))
                rounds["autocast_module_us"].append(timed(module, reps))
            a, b = fused(0), module(0)
            cmp = {name: {"max_abs_diff": float((u.float() - v.float()).abs().max()), "scale": float(v.float().abs().max())}
                   for u, v, name in zip(a, b, ("logits", "value", "mine"))}
        med = {k: statistics.median(v) for k, v in rounds.items()}
        flop, nbytes = n * FLOP_PER_BOARD, n * BYTES_PER_BOARD
        bound_us = max(flop / PEAK_FLOPS, nbytes / PEAK_BW) * 1e6
        row = {"boards": n, "reps": reps, "rounds": rounds, "median": med,
               "kernel_tflops": flop / med["kernel_us"] / 1e6, "kernel_gb_per_s": nbytes / med["kernel_us"] / 1e3,
               "bound_us": bound_us, "bound_by": "tensor rate" if flop / PEAK_FLOPS > nbytes / PEAK_BW else "HBM bandwidth",
               "kernel_share_of_bound": bound_us / med["kernel_us"],
               "speedup_fused_vs_module": med["autocast_module_us"] / med["fused_forward_us"], "outputs_fused_vs_module": cmp}
        res["forward"][str(n)] = row
        print("forward", json.dumps(row), flush=True)
        del obs, x16
        torch.cuda.empty_cache()

    # ---- rollouts: graph-captured fused forward against the eager autocast module
    cfg = m.EnvConfig(H=16, W=16, mine_count=40, guarantee_safe_neighborhood=True, step_penalty=1e-4)
    res["rollout"] = []
    for envs, T in ((8192, 128), (128, 64)):
        row = {"envs": envs, "steps": T}
        for kind in ("graph_fused", "eager_module"):
            torch.manual_seed(0)
            vec = m.VecMinesweeper(envs, cfg, seed=0, api="torch")
            model = m.build_model("cnn", obs_shape=(10, 16, 16)).cuda()
            col = (m.RolloutCollector(vec, T, aux_maps=True, graph=True) if kind == "graph_fused"
                   else m.RolloutCollector(vec, T, aux_maps=True, fused=False, graph=False))
            times = []
            for i in range(4):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                col.collect(model)
                e1.record()
                torch.cuda.synchronize()
                if i >= 1:
                    times.append(e0.elapsed_time(e1))
            ms = statistics.median(times)
            row[kind] = {"ms_rollout": ms, "frames_per_s": envs * T / (ms / 1e3), "ms_each": times}
            del col, vec, model
            torch.cuda.empty_cache()
        row["speedup"] = row["graph_fused"]["frames_per_s"] / row["eager_module"]["frames_per_s"]
        res["rollout"].append(row)
        print("rollout", json.dumps(row), flush=True)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
