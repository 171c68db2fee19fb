"""Times WaveNet autoregressive sampling on one GPU: WaveNet.inference on the device (svsk_wavenet_ar_f32, one launch
for all steps, plus the conditioning GEMM and torch.rand) against the per-step host loop of the reference
(incremental_logits, softmax, OneHotCategorical: nnsvs/wavenet/wavenet.py:89-149), rebuilt here.

    python tools/bench_wavenet_ar.py --out DIR [--host-steps 100]

Device path: CUDA events over repeated whole inference() calls, after one warm-up call, for at least --min-seconds.
Host loop: --host-steps steps per (config, B) after 10 warm-up steps (it is the same per-step work at every length).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ensemble_svs_with_interactions_b200.wavenet import WaveNet  # noqa: E402

CONFIGS = {
    "default": dict(in_dim=334, out_dim=206, layers=10),        # WaveNet() of the reference
    "test_shape": dict(in_dim=300, out_dim=206, layers=2),      # the reference's test (tests/test_wavenet.py)
}


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unavailable"
    except (OSError, subprocess.TimeoutExpired):
        info["power_limit_and_max_sm_clock"] = "unavailable"
    return info


def time_device(m, c, steps, min_seconds):
    m.inference(c, steps)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    m.inference(c, steps)
    e1.record()
    torch.cuda.synchronize()
    reps = max(2, math.ceil(min_seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(reps):
        m.inference(c, steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return ms * 1e3 / (reps * steps), reps, ms / 1e3


@torch.no_grad()
def host_loop(m, c, steps):
    B = c.shape[0]
    m.clear_buffer()
    current = torch.zeros(B, 1, m.out_dim, device=c.device)
    for t in range(steps):
        x = m.incremental_logits(current, c[:, t, :].unsqueeze(1))
        probs = F.softmax(x.view(B, -1), dim=1)
        current = torch.distributions.OneHotCategorical(probs).sample().view(B, 1, -1)
    m.clear_buffer()


def time_host(m, c, steps):
    host_loop(m, c, 10)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    host_loop(m, c, steps)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e6 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_wavenet_ar.json")
    ap.add_argument("--batches", default="1,8,64")
    ap.add_argument("--steps", default="200,2000")
    ap.add_argument("--host-steps", type=int, default=100)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wavenet_ar: needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    info = device_info()
    print(json.dumps(info))
    rows = []
    for name, cfg in CONFIGS.items():
        torch.manual_seed(0)
        m = WaveNet(**cfg).cuda().eval()
        for B in [int(x) for x in a.batches.split(",")]:
            T = max(int(x) for x in a.steps.split(","))
            c = torch.randn(B, T, cfg["in_dim"], device="cuda")
            host_us = time_host(m, c, a.host_steps)
            for steps in [int(x) for x in a.steps.split(",")]:
                us, reps, secs = time_device(m, c, steps, a.min_seconds)
                row = dict(config=name, B=B, steps=steps, device_us_per_step=round(us, 3), device_reps=reps,
                           device_seconds=round(secs, 3), host_loop_us_per_step=round(host_us, 1),
                           host_loop_steps=a.host_steps, speedup=round(host_us / us, 1))
                print(json.dumps(row), flush=True)
                rows.append(row)
    with open(os.path.join(a.out, "bench_wavenet_ar.json"), "w") as f:
        json.dump(dict(info, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
