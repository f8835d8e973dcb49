"""Development: time the fused rollout forward at C3 size and list its kernels (torch profiler)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import minesweeper_ppo_b200 as m
from minesweeper_ppo_b200.fused_forward import FusedRolloutForward
from torch.profiler import profile, ProfilerActivity

N = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
torch.backends.cudnn.benchmark = os.environ.get("CUDNN_BENCHMARK", "0") == "1"
model = m.build_model("cnn_residual", obs_shape=(10, 16, 16),
                      model_cfg=dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256)).cuda()
x = (torch.rand(N, 10, 16, 16, device="cuda") < 0.3).float()
ff = FusedRolloutForward(model)
for _ in range(3):
    ff(x, return_mine=True)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(10):
    ff(x, return_mine=True)
b.record(); torch.cuda.synchronize()
print(f"fused forward: {a.elapsed_time(b)/10:.3f} ms / forward of {N} boards")
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    ff(x, return_mine=True)
    torch.cuda.synchronize()
print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=14, max_name_column_width=90))
