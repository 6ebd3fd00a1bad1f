"""Forward + backward timing of a projection head with several outputs: the fused multi-output head (functional.mlp_head ->
MlpHeadMultiFn: b2no_mlp_head_fwd_multi, b2no_mlp_head_bwd_multi, b2no_pw_wgrad) against the composed path it replaces (two
pointwise convs, the hidden tensor and its pre-activation written in the forward and read in the backward), at two shapes:

  fullfield  PINObserverFullField's tail at the cfg4 grid: batch 4, 64 channels, 64 x 64 x 73 (padded), fc_dim 128,
             3 outputs (plane_num 3), the Reynolds term as a per-sample bias (fused) / a 1-channel map (composed)
  fno2d      the FNO2d head at the cfg2 shape with 2 outputs: batch 64, 32 channels, 128 x 128, 256 hidden

The input of each shape is larger than the 126 MB L2.  CUDA events around --iters steps (forward, backward with every
parameter gradient); the arms alternate (composed, fused, composed, fused).  Prints the card's name and power limit, then
one JSON line per arm and repetition."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def shapes(dev):
    torch.manual_seed(0)
    B, C, H = 4, 64, 128
    x = torch.randn(B, C, 64, 64, 73, device=dev, requires_grad=True)
    re = torch.linspace(0.1, 0.5, B, device=dev).reshape(B, 1)
    ff = dict(x=x, re=re, re_map=re.reshape(B, 1, 1, 1, 1).expand(B, 1, 64, 64, 73).contiguous(),
              w1=(torch.randn(H, C, device=dev) / C ** 0.5).requires_grad_(True),
              wre=torch.randn(H, 1, device=dev).requires_grad_(True), b1=torch.randn(H, device=dev).requires_grad_(True),
              w2=(torch.randn(3, H, device=dev) / H ** 0.5).requires_grad_(True), b2=torch.randn(3, device=dev).requires_grad_(True),
              g=torch.randn(B, 3, 64, 64, 73, device=dev))
    B, C, H = 64, 32, 256
    fno = dict(x=torch.randn(B, C, 128, 128, device=dev, requires_grad=True),
               w1=(torch.randn(H, C, 1, 1, device=dev) / C ** 0.5).requires_grad_(True),
               b1=torch.randn(H, device=dev).requires_grad_(True),
               w2=(torch.randn(2, H, 1, 1, device=dev) / H ** 0.5).requires_grad_(True),
               b2=torch.randn(2, device=dev).requires_grad_(True), g=torch.randn(B, 2, 128, 128, device=dev))
    return {"fullfield": ff, "fno2d": fno}


def arms(name, s):
    import pde_policylearning_b200.functional as Fn
    if name == "fullfield":
        leaves = [s[k] for k in ("x", "w1", "wre", "b1", "w2", "b2")]

        def fused():
            return Fn.mlp_head(s["x"], s["w1"], s["b1"][None, :] + s["re"] @ s["wre"].t(), s["w2"], s["b2"], "gelu")

        def composed():
            t = Fn.pointwise_conv2(s["x"], s["w1"], s["b1"], "gelu", s["re_map"], s["wre"])
            return Fn.pointwise_conv(t, s["w2"], s["b2"], None)
        assert Fn.mlp_head_fused_available(s["x"], s["w1"], s["w2"], None, True)
    else:
        leaves = [s[k] for k in ("x", "w1", "b1", "w2", "b2")]

        def fused():
            return Fn.mlp_head(s["x"], s["w1"], s["b1"], s["w2"], s["b2"], "gelu")

        def composed():
            return Fn.pointwise_conv(Fn.pointwise_conv(s["x"], s["w1"], s["b1"], "gelu"), s["w2"], s["b2"], None)
        assert Fn.mlp_head_fused_available(s["x"], s["w1"], s["w2"], s["b1"], True)

    def step(fn):
        def run():
            torch.autograd.grad(fn(), leaves, s["g"])
        return run
    return {"composed": step(composed), "fused": step(fused)}, (fused, composed)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    from pde_policylearning_b200 import ops
    dev = torch.device("cuda", 0)
    print(json.dumps({"gpu": card()}), flush=True)
    for name, s in shapes(dev).items():
        fns, (fused, composed) = arms(name, s)
        with torch.no_grad():
            d = (fused() - composed()).norm() / composed().norm()
        print(json.dumps({"shape": name, "fused_vs_composed_rel_l2": float(d)}), flush=True)
        for _ in range(args.reps):
            for arm in ("composed", "fused"):
                fn = fns[arm]
                for _ in range(3):
                    fn()
                torch.cuda.synchronize()
                n0 = ops.tensor_core_launches()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(args.iters):
                    fn()
                t1.record()
                torch.cuda.synchronize()
                print(json.dumps({"shape": name, "arm": arm, "ms_per_fwd_bwd": round(t0.elapsed_time(t1) / args.iters, 3),
                                  "tc_launches_per_step": (ops.tensor_core_launches() - n0) / args.iters}), flush=True)
        del fns, fused, composed, s
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
