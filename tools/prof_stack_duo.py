"""Three launches of the two-tiles-per-pair C = 128 residual stack at the pipeline's bap shape (6 x 6000 frames, 10 blocks)
for a kernel profiler (144 CTAs fit the device; the launch is cooperative, which kernel replay cannot re-launch)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from ensemble_svs_with_interactions_b200 import ops  # noqa: E402
from ensemble_svs_with_interactions_b200.diffsinger import DiffNet, GaussianDiffusion  # noqa: E402

B, T = 6, 6000
torch.manual_seed(0)
m = GaussianDiffusion(128, 5, DiffNet(5, 128, 10, 128, 4), K_step=100).to("cuda").eval()
plan = m.denoise_fn.bf16_plan()
table = m._step_table()
cond = torch.randn(B, T, plan.H, device="cuda").to(torch.bfloat16)
xb0 = torch.randn(B, T, plan.C, device="cuda").to(torch.bfloat16)
e0, e1 = torch.empty_like(xb0), torch.empty_like(xb0)
skip = torch.empty(B, T, plan.C, device="cuda")
flags = torch.empty((B * 2 * ((T + 255) // 256),), device="cuda", dtype=torch.int32)
assert ops.diffnet_stack_fits(B, T, plan.C, plan.H)
for _ in range(3):
    ops.diffnet_stack_bf16(xb0, e0, e1, skip, cond, plan.w1p_all, plan.woutp_all, table[:, 50:51], plan.bout_all, flags,
                           plan.dilations, stepbias_batch_stride=0, stepbias_layer_stride=table.stride(0))
torch.cuda.synchronize()
print("done", bool(torch.isfinite(skip).all()))
