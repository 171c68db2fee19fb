"""Timing of the one-launch residual stack at the BASELINE config-2 shape (A/B aid for the stack kernel)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from ensemble_svs_with_interactions_b200 import ops  # noqa: E402

B, T = bench.B, bench.T
if len(sys.argv) > 2:
    B, T = int(sys.argv[1]), int(sys.argv[2])
if os.environ.get("SVSK_STACK_BENCH_MODEL"):   # "M,H,L,C", e.g. 5,128,10,128 = the pipeline's bap model
    from ensemble_svs_with_interactions_b200.diffsinger import DiffNet, GaussianDiffusion
    M_, H_, L_, C_ = (int(v) for v in os.environ["SVSK_STACK_BENCH_MODEL"].split(","))
    torch.manual_seed(0)
    m = GaussianDiffusion(H_, M_, DiffNet(M_, H_, L_, C_, 4), K_step=100).to("cuda").eval()
else:
    m = bench.build_model().to("cuda")
plan = m.denoise_fn.bf16_plan()
cond = torch.randn(B, T, plan.H, device="cuda").to(torch.bfloat16)
table = m._step_table()
xb0 = torch.randn(B, T, plan.C, device="cuda").to(torch.bfloat16)
e0b, e1b = torch.empty_like(xb0), torch.empty_like(xb0)
skip32 = torch.zeros(B, T, plan.C, device="cuda")
flags = torch.empty((B * 2 * ((T + 255) // 256),), device="cuda", dtype=torch.int32)
assert ops.diffnet_stack_fits(B, T, plan.C, plan.H)
# SVSK_STACK_BENCH_PCOND=1: with the conditioner projection precomputed (what a sampling run does), else inside the GEMM
pcond = None
if os.environ.get("SVSK_STACK_BENCH_PCOND"):
    ta, tb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m.denoise_fn.cond_projection_bf16(cond, plan)
    ta.record()
    pcond = m.denoise_fn.cond_projection_bf16(cond, plan)
    tb.record(); tb.synchronize()
    assert pcond is not None
    print(f"conditioner projection of all layers, once per run: {ta.elapsed_time(tb) * 1e3:.0f} us", flush=True)


def launch():
    ops.diffnet_stack_bf16(xb0, e0b, e1b, skip32, cond, plan.w1p_all, plan.woutp_all, table[:, 50:51], plan.bout_all, flags,
                           plan.dilations, stepbias_batch_stride=0, stepbias_layer_stride=table.stride(0), pcond=pcond)


for _ in range(3):
    launch()
torch.cuda.synchronize()
if os.environ.get("SVSK_PROFILE_RANGE"):
    torch.cuda.profiler.start()
    launch()
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
    sys.exit(0)
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(20):
    launch()
b.record(); b.synchronize()
us = a.elapsed_time(b) * 1e3 / 20
flops = 2.0 * B * T * (2 * plan.C * (3 * plan.C + plan.H) + 2 * plan.C * plan.C) * plan.L
print(f"B={B} T={T}: stack of {plan.L} blocks {us:8.1f} us/launch = {us / plan.L:6.2f} us/layer, {flops / us / 1e6:7.1f} TFLOP/s", flush=True)
