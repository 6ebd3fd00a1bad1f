"""Per-call timing of the FNO dx pass with the 1x1 weight gradient fused into it (b2no_dft_inverse_wgrad) against the two
calls it replaces (b2no_dft_inverse + b2no_pw_wgrad), at the cfg2 layer shape (batch 64, 32 channels, 128 x 128, modes 12),
for the dx pass without activation (k_pw_tc<1>; the one that multiplies by GELU'(z) keeps the two calls).

CUDA events around --iters calls; each call takes the next of --sets input sets (g and x together > L2), so g and x come
from HBM as in a training step.  Prints one JSON line per variant and repetition: microseconds per call and GB/s over the
algorithmic bytes (read g, x; write dx)."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--width", type=int, default=32)
    ap.add_argument("--grid", type=int, default=128)
    ap.add_argument("--modes", type=int, default=12)
    ap.add_argument("--sets", type=int, default=3)
    ap.add_argument("--iters", type=int, default=60)
    args = ap.parse_args()
    from pde_policylearning_b200 import ops
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    B, C, N = args.batch, args.width, args.grid
    plan = ops.get_plan(ops.SpecGeom(nin=(N, N), half=(args.modes, args.modes)), dev)
    w = torch.randn(C, C, device=dev) / C ** 0.5
    sets = []
    for _ in range(args.sets):
        sets.append(dict(gxh=torch.randn(plan.spec_shape(B, C), dtype=torch.cfloat, device=dev),
                         g=torch.randn(B, C, N, N, device=dev), x=torch.randn(B, C, N, N, device=dev)))
    tensor_bytes = B * C * N * N * 4
    def epi(s):
        return ops.make_epilogue(pw_w=w, pw_x=s["g"], pw_transposed=True)

    def fused(s):
        r = ops.dft_inverse_wgrad(plan, 1, s["gxh"], epi(s), s["x"], need_bias=True)
        assert r is not None, "fused pass not eligible at this shape"

    def unfused(s):
        ops.dft_inverse(plan, 1, s["gxh"], epi(s))
        ops.pw_wgrad(s["g"], s["x"], need_bias=True)

    for name, fn in (("unfused", unfused), ("fused", fused), ("unfused", unfused), ("fused", fused)):
        for i in range(2 * args.sets):
            fn(sets[i % args.sets])
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(args.iters):
            fn(sets[i % args.sets])
        t1.record()
        torch.cuda.synchronize()
        us = t0.elapsed_time(t1) * 1e3 / args.iters
        print(json.dumps({"variant": name, "us_per_call": round(us, 1), "algorithmic_GBps": round(3 * tensor_bytes / us / 1e3, 1),
                          "gpu": torch.cuda.get_device_name(0)}), flush=True)


if __name__ == "__main__":
    main()
