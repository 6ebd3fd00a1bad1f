"""Training-step timing of FNO2d(12, 12, 32) at the cfg2 shape (batch 64, 3 x 128 x 128 in, 32 channels) with a block norm,
three arms on the same parameters and inputs:

  none      norm=None: the FNOStackFn path the benchmark runs
  native    norm="group_norm": the norm applied to the kept-mode spectrum inside FNOStackFn (b2no_spec_norm_fwd / _bwd)
  composed  what convert_ left for a reference model with normed blocks before the native norm: the native spectral conv
            (SpectralBlockFn, bias in its epilogue), then in torch the 1x1 skip (cuDNN), GroupNorm, the add and the GELU

One activation is 134 MB, larger than the 126 MB L2.  A step is forward + backward with every parameter gradient; CUDA events
around --iters steps, the arms alternated --reps times.  Prints the card's name and power limit, one JSON line per arm and
repetition, then (a separate profiled run) the per-kernel device time per step of the none and native arms."""
import argparse
import json
import os
import re
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def composed_forward(m, x):
    """FNO.forward with each block as convert_ composed it: native conv, torch skip / norm / add / GELU."""
    blocks = m.fno_blocks
    h = m.lifting(x)
    for l in range(m.n_layers):
        y = blocks.norm[l](blocks.convs(h, l)) + F.conv2d(h, blocks.fno_skips[l].weight)
        h = F.gelu(y) if l < m.n_layers - l else y
    return m.projection(h)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import pde_policylearning_b200 as P
    dev = torch.device("cuda", 0)
    print(json.dumps({"gpu": card()}), flush=True)
    torch.manual_seed(0)
    plain = P.FNO2d(12, 12, 32, in_channels=3, out_channels=1).to(dev)
    normed = P.FNO2d(12, 12, 32, in_channels=3, out_channels=1, norm="group_norm").to(dev)
    normed.load_state_dict(plain.state_dict(), strict=False)
    x = torch.randn(64, 3, 128, 128, device=dev)
    g = torch.randn(64, 1, 128, 128, device=dev)
    p_plain, p_normed = list(plain.parameters()), list(normed.parameters())
    fns = {"none": lambda: torch.autograd.grad(plain(x), p_plain, g),
           "native": lambda: torch.autograd.grad(normed(x), p_normed, g),
           "composed": lambda: torch.autograd.grad(composed_forward(normed, x), p_normed, g)}
    with torch.no_grad():
        a, b = normed(x), composed_forward(normed, x)
        print(json.dumps({"native_vs_composed_rel_l2": float((a - b).norm() / b.norm())}), flush=True)
    for _ in range(args.reps):
        for arm, fn in fns.items():
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.iters):
                fn()
            t1.record()
            torch.cuda.synchronize()
            print(json.dumps({"arm": arm, "ms_per_step": round(t0.elapsed_time(t1) / args.iters, 3)}), flush=True)
    # per-kernel split (a separate, profiled run): device time per step of every kernel, none against native
    from torch.profiler import ProfilerActivity, profile
    split = {}
    for arm in ("none", "native"):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.iters):
                fns[arm]()
            torch.cuda.synchronize()
        for e in prof.key_averages():
            if e.device_time_total > 0:
                m = re.search(r"\b(k_\w+|\w*[Kk]ernel\w*)", e.key)
                name = m.group(1) if m else e.key[:60]
                d = split.setdefault(name, {"none": 0.0, "native": 0.0, "calls_native": 0})
                d[arm] += e.device_time_total / args.iters / 1000.0
                if arm == "native":
                    d["calls_native"] += e.count // args.iters
    total = {arm: round(sum(d[arm] for d in split.values()), 4) for arm in ("none", "native")}
    print(json.dumps({"kernel_ms_per_step_total": total}), flush=True)
    for name, d in sorted(split.items(), key=lambda kv: -abs(kv[1]["native"] - kv[1]["none"])):
        if abs(d["native"] - d["none"]) >= 0.001:
            print(json.dumps({"kernel": name, "none_ms": round(d["none"], 4), "native_ms": round(d["native"], 4),
                              "native_calls_per_step": d["calls_native"]}), flush=True)


if __name__ == "__main__":
    main()
