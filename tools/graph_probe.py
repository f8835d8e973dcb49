"""Development: rollout wall time with and without CUDA-graph capture at small N (launch-bound regime;
the reference's default training config is 128 envs x 64 steps)."""
import os, sys, json, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import minesweeper_ppo_b200 as m

out = {}
for N in [int(a) for a in sys.argv[1:]] or (128, 1024, 8192):
    T = 64
    cfg = m.EnvConfig(H=16, W=16, mine_count=40, step_penalty=1e-4)
    torch.manual_seed(0)
    model = m.build_model("cnn_residual", obs_shape=(10, 16, 16),
                          model_cfg=dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256)).cuda()
    res = {}
    all_modes = (("stock_module", dict(fused=False)), ("fused", dict(fused=True)), ("fused_graph", dict(fused=True, graph=True)))
    want = os.environ.get("MODES")
    for mode, kw in [mk for mk in all_modes if not want or mk[0] in want.split(",")]:
        print("mode", mode, "N", N, file=sys.stderr, flush=True)
        vec = m.VecMinesweeper(N, cfg, seed=0, api="torch")
        col = m.RolloutCollector(vec, T, aux_maps=True, **kw)
        for i in range(2):
            col.collect(model)
            torch.cuda.synchronize()
            print("  warm", i, file=sys.stderr, flush=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 5
        for _ in range(reps):
            col.collect(model)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        res[mode] = {"ms_per_rollout": dt * 1e3, "frames_per_s": N * T / dt}
        del col, vec
        torch.cuda.empty_cache()
    out[f"N={N},T={T}"] = res
print(json.dumps(out, indent=1))
