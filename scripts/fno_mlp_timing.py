"""Timing of the channel-MLP FNO block (FNOBlocks(use_mlp=True)) on the GPU.

  python scripts/fno_mlp_timing.py [--reps 20] [--rounds 3]

1. One cfg2-shape training step (batch 64, 128 x 128) of FNO2d(12, 12, 32) with FNOBlocks(use_mlp=True) as its blocks: the
   channel-MLP kernels (functional.ChannelMlpFn) against the composed fallback (two native pointwise convs writing the hidden tensor and the MLP
   output, then the gating as a two-operand pointwise conv), the two arms alternated, CUDA-event times.
2. The two new kernels alone at that shape (C = 32, H = 16): CUDA events around each op over many launches, the bytes the
   algorithm moves computed from the shapes, and the achieved GB/s.  The activations (134 MB each) exceed the 126 MB L2.
The card's name and power limit are read in the same run and printed with the numbers."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name(0)} (power limit not read: {e})"
    return q


def time_ms(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops
    assert torch.cuda.is_available(), "this script measures on the GPU"
    dev = torch.device("cuda", 0)
    print("card:", card())

    # ---- 1. training step, fused against composed ----
    torch.manual_seed(0)
    m = P.FNO2d(12, 12, 32, in_channels=3, out_channels=1)
    m.fno_blocks = P.FNOBlocks(32, 32, (12, 12), n_layers=4, use_mlp=True)
    m = m.to(dev)
    x = torch.randn(64, 3, 128, 128, device=dev)
    t = torch.randn(64, 1, 128, 128, device=dev)
    params = list(m.parameters())
    supported = ops.channel_mlp_supported

    def step():
        loss = P.rel_l2_loss(m(x), t, size_average=False)
        torch.autograd.grad(loss, params)

    arms = {"fused": supported, "composed": lambda u, c, h: False}
    res = {k: [] for k in arms}
    for _ in range(args.rounds):
        for name, sup in arms.items():
            ops.channel_mlp_supported = sup
            try:
                res[name].append(time_ms(step, args.reps))
            finally:
                ops.channel_mlp_supported = supported
    for name, v in res.items():
        print(f"training step, {name}: " + " / ".join(f"{a:.3f}" for a in v) + " ms")

    # ---- 2. the kernels alone ----
    B, C, H, N = 64, 32, 16, 128
    Pn = N * N
    g = lambda *s: torch.randn(*s, device=dev)
    u, xs, gy = g(B, C, N, N), g(B, C, N, N), g(B, C, N, N)
    w1, b1, w2, b2, gv = g(H, C) * C ** -0.5, g(H), g(C, H) * H ** -0.5, g(C), g(C)
    act = "gelu"
    _, pre = ops.channel_mlp_fwd(u, xs, w1, b1, w2, b2, gv, act, want_pre=True)
    f4 = 4 * B * Pn
    cases = {
        # read u, x; write y (+ pre when training)
        "fwd (inference)": (lambda: ops.channel_mlp_fwd(u, xs, w1, b1, w2, b2, gv, act, want_pre=False), 3 * C * f4),
        "fwd (training, writes pre)": (lambda: ops.channel_mlp_fwd(u, xs, w1, b1, w2, b2, gv, act, want_pre=True), 4 * C * f4),
        # read u, x, pre, gy; write du, dx, d2 (C channels) and h, d1 (H channels); + the dg reduction (negligible)
        "bwd": (lambda: ops.channel_mlp_bwd(u, xs, pre, gy, w1, b1, w2, b2, gv, act), (7 * C + 2 * H) * f4),
    }
    for name, (fn, nbytes) in cases.items():
        ts = [time_ms(fn, 4 * args.reps) for _ in range(args.rounds)]
        best = min(ts)
        print(f"kernel {name}: " + " / ".join(f"{a * 1e3:.1f}" for a in ts) + f" us; {nbytes / 1e6:.0f} MB algorithmic, "
              f"{nbytes / (best * 1e-3) / 1e9:.0f} GB/s at the best time")
    print("card:", card())


if __name__ == "__main__":
    main()
