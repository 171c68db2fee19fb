"""Times one WaveNet training step on one GPU: forward + cross-entropy + backward (no optimizer), WaveNet.forward in
training mode on libsvsk kernels (wavenet/training.py) against the reference's modules under autograd.

    python tools/bench_wavenet_train.py --out DIR [--min-seconds 1]

Reference arm: the unmodified nnsvs WaveNet (oracle/ref_shim.py) with the same parameters when its tree is present,
otherwise the oracle port (oracle.wavenet_forward: the same convolutions as differentiable torch ops), labelled as such.
Timing: CUDA events over repeated steps after 3 warm-up steps, for at least --min-seconds per point.  Launches per step:
CUDA kernels of one step in a separate torch.profiler run, whose per-kernel breakdown is written too.
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ensemble_svs_with_interactions_b200 import _lib  # noqa: E402
from ensemble_svs_with_interactions_b200.wavenet import WaveNet  # noqa: E402
from oracle import ref_shim  # noqa: E402
from oracle import svs_oracle as O  # noqa: E402

SHAPES = [
    ("test_shape", dict(in_dim=300, out_dim=206, layers=2), 2, 200),     # the reference's test (tests/test_wavenet.py)
    ("default", dict(in_dim=334, out_dim=206, layers=10), 8, 1000),      # WaveNet() of the reference
]


def device_info():
    info = {"device": torch.cuda.get_device_name(0), "cudnn_allow_tf32": torch.backends.cudnn.allow_tf32,
            "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unavailable"
    except (OSError, subprocess.TimeoutExpired):
        info["power_limit_and_max_sm_clock"] = "unavailable"
    return info


def reference_step_fn(m, cfg):
    """(step function, label) of the reference arm with m's parameters."""
    if ref_shim.reference_available():
        ref = ref_shim.load_reference().WaveNet(**cfg).cuda().train()
        ref.load_state_dict(m.state_dict())
        params = list(ref.parameters())
        return (lambda c, x: ref(c, x)), params, "reference nnsvs WaveNet under autograd"
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in m.named_parameters()}
    layers = cfg["layers"]
    return (lambda c, x: O.wavenet_forward(sd, c, x, layers, 1)), list(sd.values()), \
        "oracle port (oracle.wavenet_forward) under autograd: the reference tree is not present"


def make_step(fwd, params, c, x, target, out_dim):
    def step():
        for p in params:
            p.grad = None
        loss = F.cross_entropy(fwd(c, x).reshape(-1, out_dim), target.reshape(-1))
        loss.backward()
    return step


def time_step(step, min_seconds):
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    step()
    e1.record()
    torch.cuda.synchronize()
    reps = max(10, math.ceil(min_seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(reps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return ms * 1e3 / reps, reps, ms / 1e3


def profile_step(step, top=25):
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    kern = {}
    n = 0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in e.name.lower() and "memset" not in e.name.lower():
            n += 1
            d = kern.setdefault(e.name, [0, 0.0])
            d[0] += 1
            d[1] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    rows = sorted(({"kernel": k[:120], "calls": v[0], "us": round(v[1], 1)} for k, v in kern.items()), key=lambda r: -r["us"])
    return n, rows[:top]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_wavenet_train.json")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wavenet_train: needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    info = device_info()
    print(json.dumps(info))
    rows = []
    for name, cfg, B, T in SHAPES:
        torch.manual_seed(0)
        m = WaveNet(**cfg).cuda().train()
        c = torch.randn(B, T, cfg["in_dim"], device="cuda")
        x = torch.randn(B, T, cfg["out_dim"], device="cuda")
        target = torch.randint(0, cfg["out_dim"], (B, T), device="cuda")
        ours = make_step(m, list(m.parameters()), c, x, target, cfg["out_dim"])
        rfwd, rparams, label = reference_step_fn(m, cfg)
        ref = make_step(rfwd, rparams, c, x, target, cfg["out_dim"])
        n0 = _lib.launch_count
        ours()
        svsk_launches = _lib.launch_count - n0
        us, reps, secs = time_step(ours, a.min_seconds)
        rus, rreps, rsecs = time_step(ref, a.min_seconds)
        kern, kern_rows = profile_step(ours)
        rkern, rkern_rows = profile_step(ref)
        row = dict(shape=name, B=B, T=T, layers=cfg["layers"], svsk_us_per_step=round(us, 1), svsk_reps=reps,
                   svsk_seconds=round(secs, 3), svsk_libsvsk_launches_per_step=svsk_launches, svsk_cuda_kernels_per_step=kern,
                   reference_arm=label, reference_us_per_step=round(rus, 1), reference_reps=rreps,
                   reference_seconds=round(rsecs, 3), reference_cuda_kernels_per_step=rkern, speedup=round(rus / us, 2),
                   svsk_kernels=kern_rows, reference_kernels=rkern_rows)
        print(json.dumps({k: v for k, v in row.items() if not k.endswith("_kernels")}), flush=True)
        rows.append(row)
    with open(os.path.join(a.out, "bench_wavenet_train.json"), "w") as f:
        json.dump(dict(info, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
