#!/usr/bin/env python
"""One FFConvLSTM training step (forward, MSE, backward) on libsvsk kernels (FFConvLSTM(..., backward_kernels=True)) at
the recipe's per-GPU batch of config 5 (B 6 x T 1000), for the recipe's mgc and bap encoders, against a stock-PyTorch
module with the same state_dict (nn.Linear / Conv1d / BatchNorm1d / nn.LSTM over pack_padded_sequence, cuDNN) under
autograd on the same GPU; plus a GaussianDiffusion training step with and without the encoder.  Device-event timings
after warm-up; the card's name and power limit are read in the same run; a torch.profiler per-kernel breakdown of one
libsvsk step comes from a separate pass.

  python tools/bench_encoder_train.py [--steps 20] [--warmup 5] [--out profiles/r05_bench_encoder_train.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from torch import nn  # noqa: E402

from ensemble_svs_with_interactions_b200.diffsinger import DiffNet, GaussianDiffusion  # noqa: E402
from ensemble_svs_with_interactions_b200.model import FFConvLSTM  # noqa: E402

SIZES = {  # conf/train_acoustic/model/multitrack_acoustic_nnsvs_world_multi_ar_f0_diff_mgcbap.yaml:104-116,146-158
    "recipe": dict(in_dim=87, ff_hidden_dim=512, conv_hidden_dim=256, lstm_hidden_dim=128, out_dim=256, in_ph_start_idx=3,
                   in_ph_end_idx=50, embed_dim=256),
    "recipe_bap": dict(in_dim=87, ff_hidden_dim=256, conv_hidden_dim=128, lstm_hidden_dim=64, out_dim=128, in_ph_start_idx=3,
                       in_ph_end_idx=50, embed_dim=256),
}


class StockFFConvLSTM(nn.Module):
    """nnsvs.model.FFConvLSTM (embed_dim set, dropout 0) in stock PyTorch modules, with the same state_dict keys."""

    def __init__(self, in_dim, ff_hidden_dim, conv_hidden_dim, lstm_hidden_dim, out_dim, in_ph_start_idx, in_ph_end_idx, embed_dim):
        super().__init__()
        self.s, self.e = in_ph_start_idx, in_ph_end_idx
        V = in_ph_end_idx - in_ph_start_idx
        self.emb = nn.Embedding(V, embed_dim)
        self.fc_in = nn.Linear(in_dim - V, embed_dim)
        self.ff = nn.Sequential(nn.Linear(embed_dim, ff_hidden_dim), nn.ReLU(), nn.Linear(ff_hidden_dim, ff_hidden_dim), nn.ReLU(),
                                nn.Linear(ff_hidden_dim, ff_hidden_dim), nn.ReLU())
        layers, c = [], ff_hidden_dim
        for _ in range(3):
            layers += [nn.ReflectionPad1d(3), nn.Conv1d(c, conv_hidden_dim, 7), nn.BatchNorm1d(conv_hidden_dim), nn.ReLU()]
            c = conv_hidden_dim
        self.conv = nn.Sequential(*layers)
        self.lstm = nn.LSTM(conv_hidden_dim, lstm_hidden_dim, 2, bidirectional=True, batch_first=True)
        self.fc = nn.Linear(2 * lstm_hidden_dim, out_dim)

    def forward(self, x, lengths):
        ph = torch.argmax(x[..., self.s:self.e], dim=-1)
        h = self.emb(ph) + self.fc_in(torch.cat([x[..., :self.s], x[..., self.e:]], dim=-1))
        h = self.conv(self.ff(h).transpose(1, 2)).transpose(1, 2)
        packed = nn.utils.rnn.pack_padded_sequence(h, lengths, batch_first=True, enforce_sorted=False)
        out, _ = self.lstm(packed)
        out, _ = nn.utils.rnn.pad_packed_sequence(out, batch_first=True)
        return self.fc(out)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name()


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--tracks", type=int, default=6)
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_encoder_train.py measures the GPU: no CUDA device")
    dev = "cuda"
    torch.backends.cudnn.benchmark = True
    B, T = a.tracks, a.frames
    lengths = [T - 37 * i for i in range(B)]
    res = {"card": card(), "B": B, "T": T, "lengths": lengths, "steps": a.steps, "warmup": a.warmup,
           "cudnn": torch.backends.cudnn.version(), "allow_tf32_cudnn": torch.backends.cudnn.allow_tf32, "encoders": {}}
    g = torch.Generator().manual_seed(0)
    for name, cfg in SIZES.items():
        torch.manual_seed(1)
        m = FFConvLSTM(**cfg, backward_kernels=True).to(dev).train()
        stock = StockFFConvLSTM(**cfg).to(dev).train()
        stock.load_state_dict(m.state_dict())
        x = torch.randn(B, T, cfg["in_dim"], generator=g).to(dev)
        tgt = torch.randn(B, T, cfg["out_dim"], generator=g).to(dev)

        def step(mod):
            mod.zero_grad(set_to_none=True)
            loss = ((mod(x, lengths) - tgt) ** 2).mean()
            loss.backward()
            return loss

        ours, ref = timed(lambda: step(m), a.steps, a.warmup), timed(lambda: step(stock), a.steps, a.warmup)
        ours2 = timed(lambda: step(m), a.steps, a.warmup)           # alternate the arms once to see the spread
        res["encoders"][name] = {"svsk_ms": [round(ours, 3), round(ours2, 3)], "stock_pytorch_ms": round(ref, 3)}
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            step(m)
            torch.cuda.synchronize()
        ka = prof.key_averages()
        rows = sorted(((e.key, e.device_time_total / 1e3, e.count) for e in ka if e.device_time_total > 0), key=lambda r: -r[1])
        res["encoders"][name]["kernels_ms"] = [{"name": k[:90], "ms": round(t, 4), "calls": c} for k, t, c in rows[:25]]
        res["encoders"][name]["kernels_total_ms"] = round(sum(r[1] for r in rows), 3)
        print(json.dumps({name: {k: v for k, v in res["encoders"][name].items() if k != "kernels_ms"}}), flush=True)
        for r in rows[:8]:
            print(f"  {r[1]:8.3f} ms  x{r[2]:<4d} {r[0][:100]}", flush=True)
    # GaussianDiffusion training step (mgc stream) with and without the encoder
    torch.manual_seed(2)
    cfg = SIZES["recipe"]
    x = torch.randn(B, T, cfg["in_dim"], generator=g).to(dev)
    cond = torch.randn(B, T, 256, generator=g).to(dev)
    y = torch.randn(B, T, 60, generator=g).to(dev)
    with_enc = GaussianDiffusion(87, 60, DiffNet(60, 256, 20, 256, 4), encoder=FFConvLSTM(**cfg, backward_kernels=True),
                                 K_step=100).to(dev).train()
    without = GaussianDiffusion(256, 60, DiffNet(60, 256, 20, 256, 4), K_step=100).to(dev).train()

    def dstep(model, c):
        model.zero_grad(set_to_none=True)
        n, eps = model(c, lengths, y)
        (n - eps).abs().mean().backward()

    res["diffusion_step_ms"] = {"with_encoder": round(timed(lambda: dstep(with_enc, x), a.steps, a.warmup), 3),
                                "without_encoder": round(timed(lambda: dstep(without, cond), a.steps, a.warmup), 3)}
    print(json.dumps({"diffusion_step_ms": res["diffusion_step_ms"], "card": res["card"]}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
