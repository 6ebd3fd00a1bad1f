#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: FNO fwd+bwd samples/s (+ SpectralConv roofline fraction).

Workload at every N (weak scaling): BASELINE config 2 -- FNO2dObserver(12,12,32) == FNO2d base_fno.yaml,
4 Fourier layers, 128x128 synthetic vorticity-like fields, batch 64 PER GPU, fp32.  One step = forward,
relative-L2 loss (run_pde_observers.py:138,188-193), backward, (N>1: one NCCL gradient all-reduce), Adam.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = device-timed throughput of K steps with inputs resident in HBM; `e2e` =
the same through the public module API with pinned HOST inputs (H2D + loss D2H inside the timed region).
`--impl reference` times the reference's CPU algorithm (the oracle port, or the unmodified reference where
B2NO_REFERENCE_ROOT names a checkout of it) on the host cores with all threads, on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step computed as .npy files (dump_outputs()).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import warnings  # noqa: E402

import torch  # noqa: E402

warnings.filterwarnings("ignore")

METRIC = "fno2d_fwd_bwd_samples_per_s"
UNIT = "samples/s"
GRID = 128
MODES = 12
WIDTH = 32
BATCH = 64
LAYERS = 4


def config_dict(n_gpus):
    return {"workload": "FNO2d base_fno.yaml (FNO2dObserver modes 12, width 32, 4 layers, proj 256) on synthetic "
                        "128x128 fields, batch 64 per GPU, fp32, step = fwd + rel-L2 loss + bwd + Adam",
            "grid": GRID, "modes": MODES, "width": WIDTH, "layers": LAYERS, "batch_per_gpu": BATCH,
            "global_batch": BATCH * n_gpus, "parallelism": f"dp{n_gpus}",
            "l2_policy": "inputs larger than L2: every activation tensor is 134 MB (> 126 MB L2), ~5 GB touched per step"}


def synthetic_fields(batch, grid, seed, device="cpu"):
    """Smooth Gaussian random fields (spectrum ~ (k^2 + 49)^-1.25), unit variance: NS-vorticity-like."""
    g = torch.Generator().manual_seed(seed)
    k = torch.fft.fftfreq(grid, 1.0 / grid)
    k2 = k[:, None] ** 2 + k[None, :] ** 2
    amp = (k2 + 49.0) ** (-1.25)
    noise = torch.randn(batch, grid, grid, 2, generator=g)
    f = torch.fft.ifft2(torch.view_as_complex(noise) * amp).real
    f = f / f.std(dim=(1, 2), keepdim=True)
    return f.unsqueeze(-1).float().to(device)


# ---------------------------------------------------------------------------------------------
# clocks sampler (NVML)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index=0, period=0.1):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self.index, self.period = index, period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        if self.nv is not None:                     # first calls of the sampled queries outside the timed region
            for fn in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
                try:
                    getattr(self.nv, fn)(self.h)
                    break
                except Exception:
                    pass
            try:
                self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
            except Exception:
                pass

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10, "applications_clocks": 0x2}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, sample_batch):
    """Times fwd + rel-L2 + bwd + Adam of FNO2dObserver on the CPU with every host thread.
    Uses the unmodified reference when B2NO_REFERENCE_ROOT names a checkout of it (kind 'reference'), else the oracle port."""
    from oracle import ref_loader, restated as rs
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    p = synthetic_fields(sample_batch, GRID, seed=1)
    tgt = synthetic_fields(sample_batch, GRID, seed=2).permute(0, 3, 1, 2).contiguous()
    if ref_loader.available():
        kind = "reference"
        model = ref_loader.RefFNO2dObserver(MODES, MODES, WIDTH)
        params = list(model.parameters())
        fwd = lambda: model(p)
    else:
        kind = "port"
        import pde_policylearning_b200 as P
        sd = {k: v.detach().clone().requires_grad_(True) for k, v in P.FNO2dObserver(MODES, MODES, WIDTH).state_dict().items()}
        params = list(sd.values())
        fwd = lambda: rs.fno2d_observer_forward(sd, p, MODES)
    opt = torch.optim.Adam(params, lr=1e-3, weight_decay=1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = rs.lp_rel(fwd(), tgt, size_average=False)
        loss.backward()
        opt.step()
        return loss

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": sample_batch / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
            "sample": (f"the full {BATCH}-sample step" if sample_batch == BATCH else f"batch {sample_batch} of the {BATCH}-sample step")
                      + f" (same model, grid and step), {steps} timed steps after {warmup} warm-up, {dt * 1e3:.1f} ms/step",
            "ms_per_step": dt * 1e3}


# ---------------------------------------------------------------------------------------------
# per-kernel probes (CUDA events on the launching stream) for the roofline object
# ---------------------------------------------------------------------------------------------
def _time_op(fn, iters=30, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in evs)
    return sum(ts) / len(ts) * 1e-3  # seconds, mean


def measured_tc_peaks(dev):
    """Dense tcgen05.mma issue rate measured on this GPU (csrc/tc_peak.cu: every SM issues back-to-back M=128, N=256 MMAs
    from resident shared-memory operands, cta_group::1), CUDA events around the launch, best of 5.  SURVEY.md 8d asked
    for a measured kind::tf32 figure in place of "bf16 / 2"."""
    import ctypes as C
    from pde_policylearning_b200 import _lib
    L = _lib.lib()
    out = {}
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for name, kind in (("tf32", 0), ("bf16", 1)):
        flops = C.c_double(0.0)
        best = None
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(L.b2no_tc_peak_probe(kind, 20000, C.byref(flops), st), "tc_peak_probe")
            e1.record()
            torch.cuda.synchronize()
            t = e0.elapsed_time(e1) * 1e-3
            best = t if best is None else min(best, t)
        out[name] = flops.value / best / 1e12
    return out


def kernel_probes(dev, hbm_peak_gbs, tf32_peak_tflops):
    """Times every hot kernel group of one training step at the workload's shape, each alone, with CUDA events on
    the launching stream, rotating over 3 buffer sets (working set > 126 MB L2).  Algorithmic bytes / flops per
    launch are SURVEY.md 8d's formulas (DESIGN.md section 4); the roofline fraction of a kernel is 8d's
    max(bytes / HBM, p * flops / TC) / t with p = 3 (every product is issued three times: 3xTF32)."""
    from pde_policylearning_b200 import ops
    B, C, N, H = BATCH, WIDTH, GRID, 256
    geom = ops.SpecGeom(nin=(N, N), half=(MODES // 2, MODES // 2), norm="forward")
    plan = ops.get_plan(geom, dev)
    nbuf = 3
    xs = [torch.randn(B, C, N, N, device=dev) for _ in range(nbuf)]
    outs = [torch.empty(B, C, N, N, device=dev) for _ in range(nbuf)]
    zs = [torch.randn(B, C, N, N, device=dev) for _ in range(nbuf)]
    spec = [torch.randn(B, C, *plan.kept, dtype=torch.complex64, device=dev) for _ in range(nbuf)]
    w = torch.randn(C, C, device=dev)
    bias = torch.randn(C, device=dev)
    w1, b1 = torch.randn(H, C, device=dev) * 0.2, torch.randn(H, device=dev)
    w2, b2 = torch.randn(H, device=dev) * 0.2, torch.randn(1, device=dev)
    g1 = [torch.randn(B, 1, N, N, device=dev) for _ in range(nbuf)]
    state = {"i": 0}

    def nxt():
        state["i"] = (state["i"] + 1) % nbuf
        return state["i"]

    def fwd_dft():
        ops.dft_forward(plan, 0, xs[nxt()])

    def inv_fused():
        i = nxt()
        ops.dft_inverse(plan, 0, spec[i], ops.make_epilogue(bias=bias, pw_w=w, pw_x=xs[i]), out=outs[i])

    def inv_fused_gelu():
        i = nxt()
        ops.dft_inverse(plan, 0, spec[i], ops.make_epilogue(bias=bias, pw_w=w, pw_x=xs[i], preact=zs[i], act="gelu"), out=outs[i])

    def inv_dact():
        i = nxt()
        ops.dft_inverse(plan, 1, spec[i], ops.make_epilogue(pw_w=w, pw_x=xs[i], pw_transposed=True, dact_z=zs[i], dact="gelu"), out=outs[i])

    def wgrad():
        i = nxt()
        ops.pw_wgrad(xs[i], outs[(i + 1) % nbuf], need_bias=False)

    def head_fwd():
        ops.mlp_head_fwd(xs[nxt()], w1, b1, w2, b2, "gelu")

    def head_bwd():
        i = nxt()
        ops.mlp_head_bwd_fused(xs[i], w1, b1, w2, g1[i], "gelu")

    bx = B * C * N * N * 4
    K = plan.modes
    px = B * N * N
    probes = [
        dict(kernel="dft_forward (k_fwd_tc)", fn=fwd_dft, bound="hbm", bytes=bx + B * C * K * 8, n=8),
        dict(kernel="dft_inverse + bias + 1x1 skip (k_inv_h + k_pw_tc<1>)", fn=inv_fused, bound="hbm", bytes=2 * bx + B * C * K * 8, n=4),
        dict(kernel="dft_inverse adjoint + W^T g, times GELU'(z) (k_inv_h + k_pw_tc<3>)", fn=inv_dact, bound="hbm", bytes=3 * bx + B * C * K * 8, n=2),
        dict(kernel="dft_inverse + bias + 1x1 skip + GELU, z saved (k_inv_h + k_pw_tc<2>)", fn=inv_fused_gelu, bound="hbm",
             bytes=3 * bx + B * C * K * 8, n=2),
        dict(kernel="1x1 weight gradient (k_wgrad_tc + reduce)", fn=wgrad, bound="hbm", bytes=2 * bx, n=5),
        dict(kernel="projection head forward (k_mlp_tc<fwd>)", fn=head_fwd, bound="tensor", bytes=bx + px * 4,
             flops=2.0 * px * (C * H + H), n=1),
        # algorithmic bytes: read x, read g, write gx -- the 256-wide hidden tensor and its gradient never touch HBM
        # (SURVEY 8d); flops: z1 recompute + gx + dW1 (three C x H products per pixel) + dw2
        dict(kernel="projection head backward, one kernel: gx + dW1 + db1 + dw2 (k_head_bwd)", fn=head_bwd, bound="tensor",
             bytes=2 * bx + px * 4, flops=2.0 * px * (3 * C * H + H), n=1),
    ]
    # flops of the SpectralConv stages (DFT-as-GEMM model of SURVEY 8d), so that the same formula applies to every row
    fl_w = 2.0 * B * C * N * N * 2 * (MODES // 2)               # last-dim real -> complex stage
    fl_h = 8.0 * B * C * (MODES // 2) * N * MODES               # second stage, complex
    for p, f in zip(probes[:4], (fl_w + fl_h, fl_w + fl_h + 2.0 * px * C * C, fl_w + fl_h + 2.0 * px * C * C,
                                 fl_w + fl_h + 2.0 * px * C * C)):
        p["flops"] = f
    probes[4]["flops"] = 2.0 * px * C * C
    for p in probes:
        t = _time_op(p.pop("fn"))
        p["seconds"] = t
        p["launches_per_step"] = p.pop("n")
        p["gbs"] = p["bytes"] / t / 1e9
        p["hbm_frac"] = p["gbs"] / hbm_peak_gbs
        # algorithmic flops (each product counted once); p = 3 issues per product in the fp32-accurate 3xTF32 mode
        p["tflops"] = p["flops"] / t / 1e12
        p["issue_factor_p"] = 3
        p["tensor_frac"] = 3.0 * p["tflops"] / tf32_peak_tflops
        # SURVEY 8d: the binding roof is the larger of the two ideal times
        p["bound"] = "tensor" if p["tensor_frac"] > p["hbm_frac"] else "hbm"
        p["frac"] = max(p["tensor_frac"], p["hbm_frac"])
    return probes



# ---------------------------------------------------------------------------------------------
# the other BASELINE configs: cfg3 (RNO training), cfg4 (PINO training), cfg5 (RNO control rollout)
# ---------------------------------------------------------------------------------------------
def _grf(shape_lead, n, seed, device):
    """Smooth Gaussian random planes (.., n, n), unit variance per plane (channel-flow wall-pressure-like)."""
    g = torch.Generator().manual_seed(seed)
    k = torch.fft.fftfreq(n, 1.0 / n)
    amp = (k[:, None] ** 2 + k[None, :] ** 2 + 49.0) ** (-1.25)
    f = torch.fft.ifft2(torch.view_as_complex(torch.randn(*shape_lead, n, n, 2, generator=g)) * amp).real
    return (f / f.std(dim=(-2, -1), keepdim=True)).float().to(device)


def bench_cfg3(dev, rank, world, timed, steps=3, warmup=2, B=None, T=None, graph=True):
    """cfg3: RNO observer (configs/matlab_rno.yaml: modes 12, width 34, layer_num 1, 32x32), trajectories of T = 100 frames,
    batch 256 per GPU; step = forward (199 recurrent cell steps + 100 regressor calls), rel-L2 loss, backward through time,
    (N > 1: NCCL gradient all-reduce), fused Adam.  `.eval()`: the regressor's dropout(0.3) is off, as in the parity tests."""
    import pde_policylearning_b200 as P
    B = int(os.environ.get("B2NO_CFG3_B", B or 256))
    T = int(os.environ.get("B2NO_CFG3_T", T or 100))
    torch.manual_seed(0)
    model = P.RNO2dObserver(12, 12, 34, 0, layer_num=1).to(dev).eval()
    x = _grf((B, T), 32, 300 + rank, dev).unsqueeze(-1)
    tgt = _grf((B,), 32, 400 + rank, dev).unsqueeze(-1)
    overlap = os.environ.get("B2NO_OVERLAP_AR", "0") not in ("", "0") and world > 1
    opt = P.FusedAdam(model.parameters(), lr=1e-3, weight_decay=1e-4, overlap_allreduce=overlap)
    lf = lambda o, t: P.rel_l2_loss(o.reshape(B, -1), t.reshape(B, -1), size_average=False)

    def eager():
        opt.zero_grad(set_to_none=True)
        loss = lf(model(x), tgt)
        loss.backward()
        opt.sync_grads()
        opt.step(grad_scale=1.0 / world)
        return loss.detach()

    gstep, mode = None, "eager"
    if graph:
        try:
            gstep = P.GraphedTrainStep(model, lf, opt, (x,), tgt, warmup=1)
            mode = f"one CUDA graph ({gstep.launches_per_step} library launches per step)"
        except Exception as e:  # noqa: BLE001
            print(f"warning: cfg3 graph capture failed ({type(e).__name__}: {e}); eager", file=sys.stderr)
            gstep = None
    fn = (lambda: gstep((x,), tgt)) if gstep is not None else eager
    for _ in range(warmup):
        fn()
    ms = timed(fn, steps) / steps
    peak_mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    if gstep is not None:
        gstep.close()
    convs = 8 * (2 * T - 1) + 2 * T
    # SURVEY 8d per-conv algorithmic bytes at B = 256: fwd 74.0 MB, bwd 96.7 MB (scaled linearly in B)
    alg_bytes = convs * (74.0e6 + 96.7e6) * B / 256.0
    return {"config": "cfg3", "workload": f"RNO2dObserver(12,12,34,layer_num=1) 32x32, T={T} frames, batch {B} per GPU, fp32, "
                                          "step = fwd + rel-L2 + BPTT + Adam, regressor dropout off (.eval())",
            "metric": "rno_fwd_bwd_trajectories_per_s", "value": round(B * world / (ms * 1e-3), 2), "unit": "trajectories/s",
            "ms_per_step": round(ms, 3), "ms_per_recurrent_step": round(ms / T, 4), "batch_per_gpu": B, "T": T, "n_gpus": world,
            "spectral_conv_calls_per_step": convs, "execution": mode, "peak_mem_gib": round(peak_mem, 1),
            "roofline": {"bound": "hbm", "algorithmic_bytes_per_step": alg_bytes, "unit": "GB/s",
                         "achieved": round(alg_bytes / (ms * 1e-3) / 1e9, 1),
                         "note": "whole step against HBM: spectral-conv calls x SURVEY 8d's per-conv fwd+bwd bytes / step time"}}


def bench_cfg4(dev, rank, world, timed, steps=5, warmup=3, B=None):
    """cfg4: PINObserver2d (pino-observer-pretrain-1s.yaml: 4 layers x 64 ch, modes 8, fc 128, pad 0.0625) on a 64x64x65
    space-time grid, batch 4 per GPU; step = forward, 5 data + 1 f + 1 ic loss (train_pino.py:87-107), backward,
    (N > 1: NCCL all-reduce of 269 MB of gradients), fused Adam."""
    import pde_policylearning_b200 as P
    B = int(os.environ.get("B2NO_CFG4_B", B or 4))
    S, T = 64, 65
    torch.manual_seed(0)
    model = P.PINObserver2d(modes1=[8] * 4, modes2=[8] * 4, modes3=[8] * 4, fc_dim=128, layers=[64] * 5, act="gelu",
                            pad_ratio=0.0625).to(dev)
    a0 = _grf((B,), S, 500 + rank, dev)
    gx = torch.linspace(0, 1, S + 1, device=dev)[:-1]
    gt = torch.linspace(0, 1, T, device=dev)
    a_in = torch.stack((gx.reshape(1, S, 1, 1).expand(B, S, S, T), gx.reshape(1, 1, S, 1).expand(B, S, S, T),
                        gt.reshape(1, 1, 1, T).expand(B, S, S, T), a0.unsqueeze(-1).expand(B, S, S, T)), dim=-1).contiguous()
    u = (a0.unsqueeze(-1) * torch.cos(gt * 3.0).reshape(1, 1, 1, T)).contiguous()
    re = (torch.randint(100, 501, (B,), generator=torch.Generator().manual_seed(600 + rank)).float()).to(dev)
    forcing = P.get_forcing(S, device=dev)
    overlap = os.environ.get("B2NO_OVERLAP_AR", "0") not in ("", "0") and world > 1
    opt = P.FusedAdam(model.parameters(), lr=1e-3, overlap_allreduce=overlap)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = P.pino_training_loss(model, a_in, re, u, forcing, xy_weight=5.0, f_weight=1.0, ic_weight=1.0, t_interval=0.5)
        loss.backward()
        opt.sync_grads()
        opt.step(grad_scale=1.0 / world)
        return loss.detach()

    for _ in range(warmup):
        step()
    ms = timed(step, steps) / steps
    px = S * S * 73
    alg_bytes = B * 4 * (679.5e6 + 750.8e6) / 4.0     # SURVEY 8d: per conv fwd 679.5 MB, bwd 750.8 MB at B = 4, four layers
    return {"config": "cfg4", "workload": f"PINObserver2d 4x64ch modes 8 on 64x64x65 (padded to 73), batch {B} per GPU, step = fwd + "
                                          "(5 data + f + ic) loss + bwd + Adam; the reference's second identical forward (train_pino.py:98, "
                                          "quirk Q6) is computed once",
            "metric": "pino_fwd_bwd_samples_per_s", "value": round(B * world / (ms * 1e-3), 2), "unit": "samples/s",
            "ms_per_step": round(ms, 3), "batch_per_gpu": B, "n_gpus": world, "execution": "eager",
            "grad_allreduce_bytes": int(sum((2 if p.is_complex() else 1) * p.numel() for p in model.parameters()) * 4),
            "roofline": {"bound": "hbm", "algorithmic_bytes_per_step": alg_bytes, "unit": "GB/s",
                         "achieved": round(alg_bytes / (ms * 1e-3) / 1e9, 1),
                         "note": "four SpectralConv3d layers fwd+bwd (SURVEY 8d bytes) / whole step time, pointwise head / tail and "
                                 "loss traffic not counted"}}


def bench_cfg5(dev, rank, world, timed, steps=20, warmup=5, B=None):
    """cfg5: batched control rollout -- the RNO observer called once per control step on B environments (run_control.py:150-151
    batched), no_grad, .eval(); the environment is a stub that emits GRF pressure planes.  128 environments per GPU
    (1024 over 8 GPUs); the single-GPU figure for all 1024 is reported next to it."""
    import pde_policylearning_b200 as P
    torch.manual_seed(0)
    model = P.RNO2dObserver(12, 12, 34, 0, layer_num=1).to(dev).eval()
    res = {}
    for tag, Bn in (("per_gpu_128", int(os.environ.get("B2NO_CFG5_B", B or 128))), ("single_gpu_1024", 1024)):
        x = _grf((Bn, 1), 32, 700 + rank, dev).unsqueeze(-1)
        with torch.no_grad():
            for _ in range(3):
                out = model(x)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            try:
                with torch.cuda.graph(g):
                    out = model(x)
                fn = g.replay
                mode = "CUDA graph"
            except Exception as e:  # noqa: BLE001
                print(f"warning: cfg5 graph capture failed ({type(e).__name__}: {e}); eager", file=sys.stderr)
                fn = lambda: model(x)
                mode = "eager"
            for _ in range(warmup):
                fn()
            ms = timed(fn, steps) / steps
        res[tag] = {"envs": Bn, "ms_per_control_step": round(ms, 4), "env_steps_per_s": round(Bn / (ms * 1e-3), 1), "execution": mode}
        del g
    r = res["per_gpu_128"]
    return {"config": "cfg5", "workload": "RNO2dObserver(12,12,34,layer_num=1) inference per control step on batched synthetic "
                                          "environments (32x32 pressure planes), no_grad, 128 environments per GPU",
            "metric": "rno_rollout_env_steps_per_s", "value": round(r["env_steps_per_s"] * world, 1), "unit": "env-steps/s",
            "ms_per_step": r["ms_per_control_step"], "n_gpus": world, "detail": res}


def other_configs(dev, rank, world, timed, args):
    out = []
    for name, fn in (("cfg3", bench_cfg3), ("cfg4", bench_cfg4), ("cfg5", bench_cfg5)):
        if args.only and args.only != name:
            continue
        import pde_policylearning_b200 as P
        t0 = time.perf_counter()
        try:
            P.set_precision("fp32")
            r = fn(dev, rank, world, timed)
            r["precision_mode"] = "fp32 (3xTF32 tensor-core products, parity <= 1e-5)"
            if not os.environ.get("B2NO_SKIP_TF32"):
                # the same step in the reduced-precision tensor-core mode (north star: <= 2e-2, stated per config)
                torch.cuda.empty_cache()
                P.set_precision("tf32")
                r2 = fn(dev, rank, world, timed)
                r["tf32_mode"] = {"value": r2["value"], "unit": r2["unit"], "ms_per_step": r2["ms_per_step"],
                                  "note": "single-pass TF32 MMAs (P.set_precision('tf32')); data stays fp32 in HBM; "
                                          "tolerance 2e-2, measured ~1e-4"}
        except Exception as e:  # noqa: BLE001
            import traceback
            traceback.print_exc(file=sys.stderr)
            r = {"config": name, "error": f"{type(e).__name__}: {e}"[:300]}
        finally:
            P.set_precision("fp32")
        r["wall_s"] = round(time.perf_counter() - t0, 1)
        out.append(r)
        torch.cuda.empty_cache()
    return out


def dump_outputs(out_dir, loss, model):
    """What the timed training step computed in its last step: the loss it returned, and the parameters (after the Adam
    update) and gradients it left in the model, as float32 .npy files (complex tensors as (..., 2) real views), ~5 MB in
    all.  The batch and the initial weights are seeded and the timed steps start from those weights, so two builds run with
    the same arguments compare file by file.  Some gradient reductions are not bitwise deterministic and training on one
    batch amplifies their rounding, so --steps 1 gives the tightest comparison."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss}
    for name, p in model.named_parameters():
        arrays[f"param.{name}"] = p
        if p.grad is not None:
            arrays[f"grad.{name}"] = p.grad
    for name, t in arrays.items():
        t = t.detach()
        t = torch.view_as_real(t) if t.is_complex() else t
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


# ---------------------------------------------------------------------------------------------
def run_b200(args):
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops, parallel
    import torch.distributed as dist

    rank, local_rank, world = parallel.init_from_env("nccl")
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    if args.only:
        res = other_configs(dev, rank, world, timed, args)
        if rank == 0:
            emit(json.dumps(res[0]))
        if world > 1:
            dist.barrier()
            os._exit(0)
        return

    torch.manual_seed(0)                                    # identical weights on every rank
    model = P.FNO2dObserver(MODES, MODES, WIDTH).to(dev)
    lp = P.LpLoss(size_average=False)
    loss_fn = lambda out, tgt: lp(out, tgt)
    overlap = os.environ.get("B2NO_OVERLAP_AR", "0") not in ("", "0") and world > 1
    opt = P.FusedAdam(model.parameters(), lr=1e-3, weight_decay=1e-4, overlap_allreduce=overlap,   # run_pde_observers.py:134
                      bucket_bytes=int(os.environ.get("B2NO_BUCKET_BYTES", str(1 << 20))))
    p_host = synthetic_fields(BATCH, GRID, seed=100 + rank).pin_memory()
    t_host = synthetic_fields(BATCH, GRID, seed=200 + rank).permute(0, 3, 1, 2).contiguous().pin_memory()
    p_dev, t_dev = p_host.to(dev), t_host.to(dev)

    # one training step = zero grads, forward, rel-L2 loss, backward, (N>1: NCCL sum all-reduce of the flat gradient
    # bucket), fused Adam -- captured once into a CUDA graph (P.GraphedTrainStep); --no-graph runs the same step eagerly
    graphed = None
    if not args.no_graph:
        try:
            graphed = P.GraphedTrainStep(model, loss_fn, opt, (p_dev,), t_dev, warmup=3)
        except Exception as e:  # noqa: BLE001
            print(f"warning: CUDA-graph capture failed ({type(e).__name__}: {e}); running the eager step", file=sys.stderr)
            graphed = None

    def eager_step(p, t):
        opt.zero_grad(set_to_none=True)
        loss = loss_fn(model(p, None), t)
        loss.backward()
        opt.sync_grads()
        opt.step(grad_scale=1.0 / world)
        return loss.detach()

    def step(p, t):
        return graphed((p,), t) if graphed is not None else eager_step(p, t)

    # resident inputs: the graph's static buffers already hold this rank's batch -> no copies in the timed region
    res_in = (graphed.static_in[0], graphed.static_tgt) if graphed is not None else (p_dev, t_dev)
    # The warm-up steps below train the model too; their updates are undone before the timed region, so the K timed steps
    # start from the seeded initial weights in every run (--dump-outputs with --steps 1 is one step on identical inputs)
    opt_state = (opt.flat_param, opt.exp_avg, opt.exp_avg_sq, opt.step_counter)
    init_state = [t.clone() for t in opt_state]
    # clock / power pre-warm (untimed, not part of W): a GPU that sat idle through the host-side set-up measured its first
    # 20 steps 9 % slow (2.61 vs 2.38 ms, profiles/r02_l) -- run the step ~0.3 s worth of times before the W warm-up steps
    # A FIXED number of steps: the step contains the gradient all-reduce at N > 1, so every rank must run the same count
    # (a time-based loop let the ranks drift apart and deadlocked / crawled at N = 8)
    for _ in range(120):
        step(*res_in)
    torch.cuda.synchronize()
    for _ in range(args.warmup):
        step(*res_in)
    for dst, src in zip(opt_state, init_state):
        dst.copy_(src)
    l0 = ops.launch_count()
    # The K-step region: barrier + synchronize on both sides, device-timed, max over ranks.  The cyclic GC is off for the
    # duration.  The loss of every step is kept (a list assignment on the host) so that --dump-outputs sees the last one.
    import gc
    gc.collect()
    gc.disable()
    last = [None]

    def timed_step():
        last[0] = step(*res_in)

    with ClockSampler(local_rank) as clk:
        ms = timed(timed_step, args.steps)
    gc.enable()
    launches = (ops.launch_count() - l0) // args.steps
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last[0], model)
    ms_per_step = ms / args.steps
    value = BATCH * world / (ms_per_step * 1e-3)

    if args.quick:
        if rank == 0:
            emit(json.dumps({"metric": METRIC, "value": round(value, 2), "ms_per_step": round(ms_per_step, 4), "n_gpus": world,
                             "clocks": clocks, "quick": True, "timed_region_ms": round(ms, 3)}))
        if world > 1:
            dist.barrier()
            if graphed is not None:
                graphed.close()
            os._exit(0)
        return

    # ---- e2e: pinned host inputs -> H2D -> public API step -> loss.item() (D2H) every step ----
    # Every step's batch is copied host->device inside the timed region; with the CUDA graph the copy of batch i+1 runs
    # on a copy stream while step i computes (P.HostBatchPipeline: the public input pipeline), so only the first copy
    # sits on the critical path; the 4-byte loss of every step is read back through pinned memory one step late.
    def e2e_run(steps):
        if graphed is not None:
            pipe = P.HostBatchPipeline(graphed)
            for loss in pipe.run_losses(((p_host,), t_host) for _ in range(steps)):
                assert loss == loss          # every step's loss arrives on the host (one step late)
        else:
            for _ in range(steps):
                eager_step(p_host.to(dev, non_blocking=True), t_host.to(dev, non_blocking=True)).item()

    e2e_run(2)
    ms_e2e = timed(lambda: e2e_run(args.steps), 1) / args.steps
    e2e = {"value": round(BATCH * world / (ms_e2e * 1e-3), 2), "unit": UNIT, "ms_per_step": round(ms_e2e, 4),
           "h2d_bytes_per_step": p_host.numel() * 4 + t_host.numel() * 4, "d2h_bytes_per_step": 4,
           "pipeline": "H2D of batch i+1 overlaps step i (copy stream, two staging sets); every step's loss is copied to "
                       "pinned host memory and read one step late"}

    out = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        bf16 = float(peaks.get("bf16_tflops", 1590.0))
        tcp = {}
        try:
            tcp = measured_tc_peaks(dev)
        except Exception as e:  # noqa: BLE001
            print(f"warning: tcgen05 peak probe failed ({e}); TF32 peak taken as bf16 / 2", file=sys.stderr)
        tf32 = float(tcp.get("tf32", bf16 / 2.0))
        peak_src = (("HBM: measured (MEASURED_PEAKS.json hbm_gbs); " if "hbm_gbs" in peaks else "HBM: fallback 6650 GB/s; ")
                    + (f"tensor: kind::tf32 dense tcgen05.mma rate measured in this run by csrc/tc_peak.cu = {tf32:.0f} TFLOP/s "
                       f"(kind::f16 bf16: {tcp.get('bf16', 0.0):.0f}; cuBLAS bf16 in MEASURED_PEAKS.json: {bf16:.0f})"
                       if tcp else "tensor: bf16_tflops / 2 (probe unavailable)"))
        probes = kernel_probes(dev, hbm, tf32)
        for p in probes:
            p["share_of_step"] = p["seconds"] * p["launches_per_step"] / (ms_per_step * 1e-3)
        top = max(probes, key=lambda p: p["share_of_step"])
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(top["kernel"])
        except Exception:
            pass
        if top["bound"] == "tensor":
            roofline = {"bound": "tensor", "kernel": top["kernel"], "achieved": round(3.0 * top["tflops"], 2), "peak": round(tf32, 1),
                        "unit": "TFLOP/s", "frac": round(top["frac"], 4), "traffic": traffic,
                        "note": "SURVEY 8d: frac = max(bytes / HBM, p * flops / TC) / t; achieved = p * algorithmic flops / launch "
                                "time with p = 3 (3xTF32 issues every product three times)",
                        "algorithmic_flops_per_launch": top["flops"], "issue_factor_p": 3}
        else:
            roofline = {"bound": "hbm", "kernel": top["kernel"], "achieved": round(top["gbs"], 1), "peak": hbm,
                        "unit": "GB/s", "frac": round(top["frac"], 4), "traffic": traffic}
        roofline.update({"peak_source": peak_src, "algorithmic_bytes_per_launch": top["bytes"],
                         "avg_launch_us": round(top["seconds"] * 1e6, 2),
                         "all": [{k: (round(v, 7 if k == "seconds" else 4) if isinstance(v, float) else v) for k, v in p.items()}
                                 for p in probes]})
        # the CPU leg runs at N = 1 only: at N > 1 the other ranks would spin in the next barrier on the same host cores
        cpu = cpu_reference_run(steps=20, warmup=2, sample_batch=16) if world == 1 else None   # ~10 s of host work
        cfg = config_dict(world)
        cfg["cuda_graph"] = graphed is not None
        cfg["prewarm_steps"] = 120          # untimed, before the W warm-up steps (fixed count: same on every rank)
        cfg["timed_region_ms"] = round(ms, 3)
        cfg["timing"] = f"one {args.steps}-step region bracketed by barrier + synchronize, CUDA events, max over ranks"
        cfg["optimizer"] = "fused flat Adam (lr 1e-3, weight_decay 1e-4), inside the timed step"
        cfg["grad_allreduce"] = ("none (1 GPU)" if world == 1 else
                                 ("per-bucket NCCL all-reduce launched from gradient hooks during backward (B2NO_OVERLAP_AR=1)"
                                  if overlap else "one NCCL all-reduce of the flat bucket after backward"))
        out = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": cfg, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
               "roofline": roofline}
        if cpu is not None:
            out["cpu_baseline"] = cpu
    # ---- the other BASELINE configs (cfg3 RNO training, cfg4 PINO training, cfg5 RNO control rollout), every rank ----
    others, tf32_line = None, None
    if not args.no_other:
        if graphed is not None:
            graphed.close()
            graphed = None
        del model, opt
        torch.cuda.empty_cache()
        # the headline step once more in the reduced-precision tensor-core mode (north star: stated per config)
        if not os.environ.get("B2NO_SKIP_TF32") and not args.no_graph:
            try:
                P.set_precision("tf32")
                torch.manual_seed(0)
                m2 = P.FNO2dObserver(MODES, MODES, WIDTH).to(dev)
                o2 = P.FusedAdam(m2.parameters(), lr=1e-3, weight_decay=1e-4)
                g2 = P.GraphedTrainStep(m2, loss_fn, o2, (p_dev,), t_dev, warmup=3)
                f2 = lambda: g2((g2.static_in[0],), g2.static_tgt)
                for _ in range(args.warmup):
                    f2()
                ms2 = timed(f2, args.steps) / args.steps
                tf32_line = {"value": round(BATCH * world / (ms2 * 1e-3), 2), "unit": UNIT, "ms_per_step": round(ms2, 4),
                             "note": "same step with single-pass TF32 MMAs (P.set_precision('tf32')); data stays fp32 in HBM; "
                                     "tolerance 2e-2, measured 6e-5 on this model's output"}
                g2.close()
                del m2, o2, g2
            except Exception as e:  # noqa: BLE001
                print(f"warning: tf32-mode measurement failed ({type(e).__name__}: {e})", file=sys.stderr)
            finally:
                P.set_precision("fp32")
                torch.cuda.empty_cache()
        others = other_configs(dev, rank, world, timed, args)
    if out is not None:
        if tf32_line is not None:
            out["tf32_mode"] = tf32_line
        if others is not None:
            out["other_configs"] = others
        emit(json.dumps(out))
    if world > 1:
        # tear down: the captured graph holds NCCL work, and destroying the communicator under a live graph blocks
        # (seen on 2 GPUs) -- release the graph first, and never let the teardown outlive the result
        dist.barrier()
        if graphed is not None:
            graphed.close()
            graphed = None
        torch.cuda.synchronize()
        t = threading.Thread(target=dist.destroy_process_group, daemon=True)
        t.start()
        t.join(20.0)
        if t.is_alive():
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the reference arm runs the SAME configuration (batch 64 per step) with every host thread: ~1-4 s per step, so K
    # steps + W warm-up steps end within a couple of minutes
    steps = max(1, min(args.steps, 50))
    warm = max(1, min(args.warmup, 5))
    r = cpu_reference_run(steps=steps, warmup=warm, sample_batch=BATCH)
    out = {"impl": "reference", "metric": METRIC, "value": round(r["value"], 3), "unit": UNIT, "n_gpus": args.gpus,
           "steps": steps, "warmup": warm, "ms_per_step": round(r["ms_per_step"], 2), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config_dict(args.gpus),
           "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
           "e2e": {"value": round(r["value"], 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(json.dumps(out))


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, warnings) was sent to stderr."""
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, (line + "\n").encode())
    else:
        print(line, flush=True)


def main():
    global _REAL_STDOUT
    # keep stdout clean for the JSON line: libraries (NCCL prints its version banner on stdout) write to fd 1
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if os.environ.get("B2NO_HANG_DUMP_S"):
        # debugging aid: dump every thread's Python stack (and exit) if the run is still going after N seconds
        import faulthandler
        faulthandler.dump_traceback_later(float(os.environ["B2NO_HANG_DUMP_S"]), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--quick", action="store_true", help="device-timed value only (no e2e, probes or CPU baseline): A/B runs")
    ap.add_argument("--no-graph", action="store_true", help="run the training step eagerly instead of as one CUDA graph")
    ap.add_argument("--no-other", action="store_true", help="skip the cfg3 / cfg4 / cfg5 measurements (other_configs)")
    ap.add_argument("--only", default=None, choices=["cfg3", "cfg4", "cfg5"], help="measure one of the other configs alone")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, parameters and gradients of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.only):
        ap.error("--dump-outputs applies to the b200 training step (not --impl reference or --only)")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the b200 arm has no CPU fallback (use --impl reference)")
        run_b200(args)


if __name__ == "__main__":
    main()
