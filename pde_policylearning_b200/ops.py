"""Thin tensor-level wrappers over the C ABI (no autograd here).  PyTorch owns every buffer; the C side
only sees device pointers, sizes and the current CUDA stream."""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ACT, NORM, Epilogue, Geom, Weights, check


# kernels replayed from captured CUDA graphs (the C-side counter only sees direct launches)
_REPLAYED = [0]


def launch_count() -> int:
    """Number of libb2no kernels launched so far, graph replays included (bench.py reports the per-step count as
    `gpu_launches`)."""
    return int(_lib.lib().b2no_kernel_launches()) + _REPLAYED[0]


def set_tensor_core_mode(on: bool) -> bool:
    """Toggle the tcgen05 kernels (both settings are CUDA paths; used by tests and A/B measurements)."""
    return bool(_lib.lib().b2no_set_tensor_core_mode(1 if on else 0))


def set_precision(mode: str) -> str:
    """'fp32' (default): every tensor-core product is issued three times on tf32 splits (3xTF32), outputs match the
    reference's fp32 torch.fft / einsum path to <= 1e-5.  'tf32': single-pass TF32 tensor-core mode (one MMA per product),
    the reduced-precision mode of the north star (tolerance 2e-2; measured ~1e-3).  Data stays fp32 in HBM either way."""
    modes = {"fp32": 0, "3xtf32": 0, "tf32": 1, "fast": 1}
    if mode not in modes:
        raise ValueError(f"precision mode {mode!r}: expected 'fp32' or 'tf32'")
    return "tf32" if _lib.lib().b2no_set_precision(modes[mode]) == 1 else "fp32"


def tensor_core_launches() -> int:
    return int(_lib.lib().b2no_tensor_core_launches())


def _require_cuda(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                "pde_policylearning_b200: the spectral-conv hot path runs only on CUDA (sm_100a); "
                f"got a tensor on {t.device}.  There is no CPU fallback.")
        if t.device.index != torch.cuda.current_device():
            # launches go to the CURRENT device's current stream (one process per GPU: parallel.init_from_env sets it)
            raise RuntimeError(f"pde_policylearning_b200: tensor on {t.device} but the current CUDA device is "
                               f"cuda:{torch.cuda.current_device()}; call torch.cuda.set_device first")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---------------------------------------------------------------------------------------------
# geometry / plans
# ---------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class SpecGeom:
    """Same fields as include/b2no.h::b2no_geom (and oracle/closed_form.py::SpecGeom)."""
    nin: Tuple[int, ...]
    half: Tuple[int, ...]
    norm: str = "backward"
    nfft: Optional[Tuple[int, ...]] = None
    nout: Optional[Tuple[int, ...]] = None
    # layout of the kept-mode spectra: 0 = (batch, channel, *kept), 1 = mode-major (*kept, batch, channel) -- see b2no_geom
    layout: int = 0

    def resolved(self) -> "SpecGeom":
        nfft = tuple(self.nin) if self.nfft is None else tuple(self.nfft)
        nout = nfft if self.nout is None else tuple(self.nout)
        return SpecGeom(tuple(self.nin), tuple(self.half), self.norm, nfft, nout, int(self.layout))

    def with_layout(self, layout: int) -> "SpecGeom":
        return SpecGeom(self.nin, self.half, self.norm, self.nfft, self.nout, int(layout))

    @property
    def ndim(self):
        return len(self.nin)

    def scales(self):
        g = self.resolved()
        n, npr = math.prod(g.nfft), math.prod(g.nout)
        if g.norm == "forward":
            return 1.0 / n, 1.0
        if g.norm == "backward":
            return 1.0, 1.0 / npr
        if g.norm == "ortho":
            return 1.0 / math.sqrt(n), 1.0 / math.sqrt(npr)
        raise ValueError(f"unknown fft norm {g.norm!r}")


class Plan:
    def __init__(self, geom: SpecGeom, device: torch.device):
        g = geom.resolved()
        if not 1 <= g.ndim <= _lib.MAX_DIM:
            raise NotImplementedError(f"spectral conv supports 1-3 spatial dims, got {g.ndim}")
        if g.norm not in NORM:
            raise ValueError(f"unknown fft norm {g.norm!r}")
        for j in range(g.ndim - 1):
            if g.half[j] > g.nfft[j]:
                raise ValueError("kept modes exceed the grid size")
        cg = Geom()
        cg.ndim = g.ndim
        for j in range(g.ndim):
            cg.nin[j], cg.nfft[j], cg.nout[j], cg.half[j] = g.nin[j], g.nfft[j], g.nout[j], g.half[j]
        cg.norm = NORM[g.norm]
        cg.spec_layout = int(g.layout)
        handle = C.c_void_p()
        with torch.cuda.device(device):
            check(_lib.lib().b2no_plan_create(C.byref(cg), C.byref(handle)), "plan_create")
        self.handle = handle
        self.geom = g
        self.device = device
        kept = (C.c_int32 * _lib.MAX_DIM)()
        check(_lib.lib().b2no_plan_kept(handle, C.byref(kept)), "plan_kept")
        self.kept = tuple(int(kept[j]) for j in range(g.ndim))
        self.modes = math.prod(self.kept)
        self.s_f, self.s_i = g.scales()
        self.layout = int(g.layout)

    def spec_shape(self, batch: int, channels: int):
        return (self.kept + (batch, channels)) if self.layout else ((batch, channels) + self.kept)

    def spec_bc(self, spec: torch.Tensor):
        """(batch, channels) of a spectrum tensor of this plan's layout."""
        if self.layout:
            if tuple(spec.shape[:-2]) != self.kept:
                raise ValueError(f"expected kept modes {self.kept} (mode-major), got {tuple(spec.shape)}")
            return int(spec.shape[-2]), int(spec.shape[-1])
        if tuple(spec.shape[2:]) != self.kept:
            raise ValueError(f"expected kept modes {self.kept}, got {tuple(spec.shape[2:])}")
        return int(spec.shape[0]), int(spec.shape[1])

    def layout_supported(self, batch: int, channels: int) -> bool:
        return bool(_lib.lib().b2no_plan_layout_supported(self.handle, batch, channels))

    def workspace(self, batch: int, channels: int) -> Optional[torch.Tensor]:
        n = int(_lib.lib().b2no_plan_workspace_floats(self.handle, batch, channels))
        if n < 0:
            check(n, "workspace")
        if n == 0:
            return None
        return torch.empty(n, dtype=torch.float32, device=self.device)

    def __del__(self):
        try:
            if self.handle:
                _lib.lib().b2no_plan_destroy(self.handle)
        except Exception:
            pass


_plans = {}


def get_plan(geom: SpecGeom, device: torch.device) -> Plan:
    key = (geom.resolved(), device.index if device.index is not None else torch.cuda.current_device())
    p = _plans.get(key)
    if p is None:
        p = Plan(geom, torch.device("cuda", key[1]))
        _plans[key] = p
    return p


# ---------------------------------------------------------------------------------------------
# weights
# ---------------------------------------------------------------------------------------------
def weights_struct(corners: Sequence[torch.Tensor], ndim: int) -> Weights:
    """corners: canonical order; each complex64 (Ci,Co,*h) or float32 real pairs (Ci,Co,*h,2)."""
    w = Weights()
    t0 = corners[0]
    for i, t in enumerate(corners):
        _require_cuda(t)
        if t.is_complex():
            if t.dtype != torch.complex64:
                raise TypeError("spectral weights must be complex64")
            strides = t.stride()
        else:
            if t.dtype != torch.float32 or t.shape[-1] != 2 or t.stride(-1) != 1:
                raise TypeError("real-pair spectral weights must be float32 (..., 2) with unit last stride")
            if any(s % 2 for s in t.stride()[:-1]):
                raise TypeError("real-pair weight strides must be even")
            strides = tuple(s // 2 for s in t.stride()[:-1])
        if i == 0:
            s0 = strides
        elif tuple(strides) != tuple(s0) or t.shape != t0.shape:
            raise ValueError("all corner weights must share shape and strides")
        w.corner[i] = t.data_ptr()
    w.stride_i, w.stride_o = s0[0], s0[1]
    for j in range(ndim):
        w.stride_k[j] = s0[2 + j]
    return w


# ---------------------------------------------------------------------------------------------
# raw ops
# ---------------------------------------------------------------------------------------------
def dft_forward(plan: Plan, which: int, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x (B, C, *grid) fp32 contiguous -> spectrum (B, C, *kept) complex64."""
    _require_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous()
    B, Cc = x.shape[:2]
    grid = plan.geom.nin if which == 0 else plan.geom.nout
    if tuple(x.shape[2:]) != tuple(grid):
        raise ValueError(f"expected grid {tuple(grid)}, got {tuple(x.shape[2:])}")
    if out is None:
        spec = torch.empty(plan.spec_shape(B, Cc), dtype=torch.complex64, device=x.device)
    else:
        spec = out
        assert spec.dtype == torch.complex64 and spec.is_contiguous() and tuple(spec.shape) == plan.spec_shape(B, Cc)
    work = plan.workspace(B, Cc)
    check(_lib.lib().b2no_dft_forward(plan.handle, which, _ptr(x), _ptr(spec), _ptr(work), B * Cc, _stream()),
          "dft_forward")
    return spec


def make_epilogue(bias=None, pw_w=None, pw_x=None, pw_transposed=False, pw2_w=None, pw2_x=None,
                  pw2_transposed=False, add=None, mul=None, preact=None, act=None, dact_z=None, dact=None,
                  gate_z=None, gate_h=None) -> Epilogue:
    """mul / gate_z may be channel slices ``t[:, a:b]`` of a wider contiguous (batch, channels, *grid) tensor: their batch
    stride is passed to the kernel (b2no_epilogue.mul_bstride / gate_bstride)."""
    e = Epilogue()
    keep = []
    for name, t in (("bias", bias), ("pw_w", pw_w), ("pw_x", pw_x), ("pw2_w", pw2_w), ("pw2_x", pw2_x),
                    ("add", add), ("mul", mul), ("preact", preact), ("dact_z", dact_z), ("gate_z", gate_z),
                    ("gate_h", gate_h)):
        if t is not None:
            _require_cuda(t)
            assert t.dtype == torch.float32, name
            if name in ("mul", "gate_z") and not t.is_contiguous():
                # a channel slice: dense inside a sample, batch stride of the parent tensor
                assert t.dim() >= 2 and t[0].is_contiguous(), name
                setattr(e, name + "_bstride" if name == "mul" else "gate_bstride", t.stride(0))
            else:
                assert t.is_contiguous(), name
            setattr(e, name, t.data_ptr())
            keep.append(t)
    if (gate_z is None) != (gate_h is None):
        raise ValueError("gate_z and gate_h go together")
    if pw_w is not None:
        e.pw_ci = pw_x.shape[1]
        e.pw_transposed = 1 if pw_transposed else 0
    if pw2_w is not None:
        e.pw2_ci = pw2_x.shape[1]
        e.pw2_transposed = 1 if pw2_transposed else 0
    e.act = ACT[act]
    e.dact = ACT[dact] if dact_z is not None else 0
    e._keep = keep
    return e


def dft_inverse(plan: Plan, which: int, spec: torch.Tensor, epi: Optional[Epilogue] = None,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """spectrum (B, C, *kept) complex64 -> y (B, C, *grid) fp32, with the fused epilogue."""
    _require_cuda(spec)
    assert spec.dtype == torch.complex64 and spec.is_contiguous()
    B, Cc = plan.spec_bc(spec)
    grid = plan.geom.nout if which == 0 else plan.geom.nin
    y = out if out is not None else torch.empty((B, Cc) + tuple(grid), dtype=torch.float32, device=spec.device)
    work = plan.workspace(B, Cc)
    check(_lib.lib().b2no_dft_inverse(plan.handle, which, _ptr(spec), _ptr(y), _ptr(work), B, Cc,
                                      math.prod(grid), C.byref(epi) if epi is not None else None, _stream()),
          "dft_inverse")
    return y


def pointwise(batch: int, channels: int, grid: Tuple[int, ...], device, epi: Epilogue) -> torch.Tensor:
    """y = act(bias + pw + pw2 + add) * mul  with no spectral term."""
    y = torch.empty((batch, channels) + tuple(grid), dtype=torch.float32, device=device)
    check(_lib.lib().b2no_dft_inverse(None, 0, None, _ptr(y), None, batch, channels, math.prod(grid),
                                      C.byref(epi), _stream()), "pointwise")
    return y


def mix(plan: Plan, mode: int, spec: torch.Tensor, corners: Sequence[torch.Tensor], ci: int, co: int,
        out: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    _require_cuda(spec)
    assert spec.dtype == torch.complex64 and spec.is_contiguous()
    B, cspec = plan.spec_bc(spec)
    cin, cout = (ci, co) if mode == 0 else (co, ci)
    assert cspec == cin, (spec.shape, cin)
    if out is None:
        out = torch.empty(plan.spec_shape(B, cout), dtype=torch.complex64, device=spec.device)
        accumulate = False
    w = weights_struct(corners, plan.geom.ndim)
    check(_lib.lib().b2no_mix(plan.handle, mode, _ptr(spec), C.byref(w), _ptr(out), B, ci, co,
                              1 if accumulate else 0, _stream()), "mix")
    return out


def mix_dw(plan: Plan, xh: torch.Tensor, gyh: torch.Tensor, like: Sequence[torch.Tensor], needs_zero: bool,
           out: Optional[Sequence[torch.Tensor]] = None, accumulate: bool = False):
    """Returns the list of corner gradients shaped/typed like `like`; with `out` (contiguous tensors of that shape) the
    gradients are written -- or, with accumulate, added -- in place (BPTT over the recurrent steps of the RNO)."""
    B, ci = plan.spec_bc(xh)
    co = plan.spec_bc(gyh)[1]
    if out is None:
        alloc = torch.zeros_like if needs_zero else torch.empty_like
        grads = [alloc(t, memory_format=torch.contiguous_format) for t in like]
        accumulate = False
    else:
        grads = list(out)
    w = weights_struct(grads, plan.geom.ndim)
    check(_lib.lib().b2no_mix_dw(plan.handle, _ptr(xh), _ptr(gyh), C.byref(w), B, ci, co, 1 if accumulate else 0,
                                 _stream()), "mix_dw")
    return grads


def spec_norm_fwd(plan: Plan, spec: torch.Tensor, bias: Optional[torch.Tensor], gamma: Optional[torch.Tensor],
                  beta: Optional[torch.Tensor], groups: int, eps: float):
    """GroupNorm(groups) of the spectral conv output s = IDFT(spec) + bias, applied to the spectrum (b2no_spec_norm_fwd):
    returns (the normalised spectrum, for dft_inverse without a bias; the statistics the backward reads)."""
    _require_cuda(spec, bias, gamma, beta)
    assert spec.dtype == torch.complex64 and spec.is_contiguous()
    B, Cc = plan.spec_bc(spec)
    for t in (bias, gamma, beta):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.numel() == Cc)
    out = torch.empty_like(spec)
    stats = torch.empty(2 * B * (Cc + groups), dtype=torch.float32, device=spec.device)
    check(_lib.lib().b2no_spec_norm_fwd(plan.handle, _ptr(spec), _ptr(bias), _ptr(gamma), _ptr(beta), float(eps), _ptr(out),
                                        _ptr(stats), B, Cc, int(groups), _stream()), "spec_norm_fwd")
    return out, stats


def spec_norm_bwd(plan: Plan, spec: torch.Tensor, gspec: torch.Tensor, stats: torch.Tensor, gamma: Optional[torch.Tensor],
                  groups: int, need_bias: bool, need_affine: bool, db_out: Optional[torch.Tensor] = None):
    """Backward of spec_norm_fwd (b2no_spec_norm_bwd): gspec = dL/d(normalised spectrum) -> (dL/dspec, dbias | None,
    dgamma | None, dbeta | None).  db_out: contiguous (channels,) destination for dbias."""
    _require_cuda(spec, gspec)
    assert gspec.dtype == torch.complex64 and gspec.is_contiguous() and gspec.shape == spec.shape
    B, Cc = plan.spec_bc(spec)
    dev = spec.device
    L = _lib.lib()
    gout = torch.empty_like(spec)
    db = None
    if need_bias:
        db = db_out if db_out is not None else torch.empty((Cc,), dtype=torch.float32, device=dev)
        assert db.is_contiguous() and db.numel() == Cc and db.dtype == torch.float32
    dg = torch.empty((Cc,), dtype=torch.float32, device=dev) if need_affine else None
    dbt = torch.empty((Cc,), dtype=torch.float32, device=dev) if need_affine else None
    scratch = torch.empty(int(L.b2no_spec_norm_bwd_scratch_floats(B, Cc)), dtype=torch.float32, device=dev)
    check(L.b2no_spec_norm_bwd(plan.handle, _ptr(spec), _ptr(gspec), _ptr(stats), _ptr(gamma), _ptr(gout), _ptr(db), _ptr(dg),
                               _ptr(dbt), _ptr(scratch), B, Cc, int(groups), _stream()), "spec_norm_bwd")
    return gout, db, dg, dbt


def act_bwd(gy: torch.Tensor, z: torch.Tensor, act) -> torch.Tensor:
    gz = torch.empty_like(gy)
    check(_lib.lib().b2no_act_bwd(_ptr(gy), _ptr(z), _ptr(gz), gy.numel(), ACT[act], _stream()), "act_bwd")
    return gz


def pw_wgrad(g: torch.Tensor, x: torch.Tensor, need_bias: bool, db_out: Optional[torch.Tensor] = None):
    """g (B, Co, *grid), x (B, Ci, *grid) -> dW (Co, Ci), db (Co) | None.  db_out: contiguous (Co,) destination for db."""
    B, co = g.shape[:2]
    ci = x.shape[1]
    P = math.prod(g.shape[2:])
    L = _lib.lib()
    n = int(L.b2no_pw_wgrad_scratch_floats(ci, co))
    partial = torch.empty(n, dtype=torch.float32, device=g.device)
    dw = torch.empty((co, ci), dtype=torch.float32, device=g.device)
    db = None
    if need_bias:
        db = db_out if db_out is not None else torch.empty((co,), dtype=torch.float32, device=g.device)
        assert db.is_contiguous() and db.numel() == co and db.dtype == torch.float32
    check(L.b2no_pw_wgrad(_ptr(g), _ptr(x), _ptr(dw), _ptr(db), _ptr(partial), B, ci, co, P, _stream()), "pw_wgrad")
    return dw, db


def dft_inverse_wgrad(plan: Plan, which: int, spec: torch.Tensor, epi: Epilogue, x: torch.Tensor, need_bias: bool,
                      db_out: Optional[torch.Tensor] = None):
    """dft_inverse(plan, which, spec, epi) and pw_wgrad(g, x) in one pass over the pixel tiles, g = the epilogue's pw_x
    (b2no_dft_inverse_wgrad).  Returns (y, dW (Co, Ci), db | None), or None -- with nothing computed -- when the fused pass
    does not support the shape; the caller then makes the two calls."""
    _require_cuda(spec, x)
    assert spec.dtype == torch.complex64 and spec.is_contiguous()
    assert x.dtype == torch.float32 and x.is_contiguous()
    B, Cc = plan.spec_bc(spec)
    grid = plan.geom.nout if which == 0 else plan.geom.nin
    if tuple(x.shape) != (B, x.shape[1]) + tuple(grid):
        raise ValueError(f"x {tuple(x.shape)} does not match batch {B} and grid {tuple(grid)}")
    co, ci = int(epi.pw_ci), int(x.shape[1])
    L = _lib.lib()
    y = torch.empty((B, Cc) + tuple(grid), dtype=torch.float32, device=spec.device)
    work = plan.workspace(B, Cc)
    partial = torch.empty(int(L.b2no_pw_wgrad_scratch_floats(ci, co)), dtype=torch.float32, device=spec.device)
    dw = torch.empty((co, ci), dtype=torch.float32, device=spec.device)
    db = None
    if need_bias:
        db = db_out if db_out is not None else torch.empty((co,), dtype=torch.float32, device=spec.device)
        assert db.is_contiguous() and db.numel() == co and db.dtype == torch.float32
    rc = L.b2no_dft_inverse_wgrad(plan.handle, which, _ptr(spec), _ptr(y), _ptr(work), B, Cc, math.prod(grid), C.byref(epi),
                                  _ptr(x), ci, _ptr(dw), _ptr(db), _ptr(partial), _stream())
    if rc == -2:
        return None
    check(rc, "dft_inverse_wgrad")
    return y, dw, db


def mlp_head_fwd(x, w1, b1, w2, b2, act="gelu") -> torch.Tensor:
    B, ci = x.shape[:2]
    grid = tuple(x.shape[2:])
    hidden = w1.shape[0]
    per_sample = b1 is not None and b1.dim() == 2
    out = torch.empty((B, 1) + grid, dtype=torch.float32, device=x.device)
    check(_lib.lib().b2no_mlp_head_fwd(_ptr(x), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), _ptr(out), B, ci, hidden,
                                       math.prod(grid), 1 if per_sample else 0, ACT[act], _stream()), "mlp_head_fwd")
    return out


def mlp_head_bwd_supported(ci: int, hidden: int, pixels: int) -> bool:
    return bool(_lib.lib().b2no_mlp_head_bwd_supported(ci, hidden, pixels))


def mlp_head_bwd(x, w1, b1, w2, g, act="gelu", want_gz=True, dact_z=None, dact=None):
    """Fused backward (input-gradient half) of the Ci -> hidden -> act -> 1 head.  Returns (gx, gz | None, dw2) or
    None when the shape has no tensor-core kernel."""
    B, ci = x.shape[:2]
    grid = tuple(x.shape[2:])
    hidden = w1.shape[0]
    P = math.prod(grid)
    L = _lib.lib()
    per_sample = b1 is not None and b1.dim() == 2
    gx = torch.empty_like(x)
    gz = torch.empty((B, hidden) + grid, dtype=torch.float32, device=x.device) if want_gz else None
    dw2 = torch.empty((hidden,), dtype=torch.float32, device=x.device)
    partial = torch.empty(int(L.b2no_mlp_head_bwd_scratch_floats(hidden)), dtype=torch.float32, device=x.device)
    rc = L.b2no_mlp_head_bwd(_ptr(x), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(g), _ptr(gx), _ptr(gz), _ptr(dw2), _ptr(partial),
                             B, ci, hidden, P, 1 if per_sample else 0, ACT[act], _ptr(dact_z),
                             ACT[dact] if dact_z is not None else 0, _stream())
    if rc == -2:
        return None
    check(rc, "mlp_head_bwd")
    return gx, gz, dw2


def mlp_head_bwd_fused_supported(ci: int, hidden: int, pixels: int) -> bool:
    return bool(_lib.lib().b2no_mlp_head_bwd_fused_supported(ci, hidden, pixels))


def mlp_head_bwd_fused(x, w1, b1, w2, g, act="gelu", dact_z=None, dact=None):
    """Whole backward of the Ci -> hidden -> act -> 1 head in one kernel (csrc/tc_head_bwd.cu): returns
    (gx, dW1 (hidden, ci), db1 (hidden), dw2 (hidden), db2 (1)); the hidden-channel gradient is never written to memory."""
    B, ci = x.shape[:2]
    hidden = w1.shape[0]
    P = math.prod(x.shape[2:])
    L = _lib.lib()
    assert b1 is None or b1.dim() == 1
    gx = torch.empty_like(x)
    grads = torch.empty((hidden * ci + 2 * hidden + 1,), dtype=torch.float32, device=x.device)
    partial = torch.empty(int(L.b2no_mlp_head_bwd_fused_scratch_floats(ci, hidden)), dtype=torch.float32, device=x.device)
    check(L.b2no_mlp_head_bwd_fused(_ptr(x), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(g), _ptr(gx), _ptr(grads), _ptr(partial),
                                    B, ci, hidden, P, ACT[act], _ptr(dact_z), ACT[dact] if dact_z is not None else 0,
                                    _stream()), "mlp_head_bwd_fused")
    n = hidden * ci
    return gx, grads[:n].view(hidden, ci), grads[n:n + hidden], grads[n + hidden:n + 2 * hidden], grads[n + 2 * hidden:]


def mlp_head_multi_supported(x: torch.Tensor, hidden: int, out_channels: int) -> bool:
    """True when the fused head with out_channels = 2..4 runs for x, forward and backward (b2no_mlp_head_bwd_multi_supported;
    its shapes are a subset of the forward's): a CUDA tensor, 16-byte aligned for the tensor-map load."""
    if not x.is_cuda or x.data_ptr() % 16 != 0:
        return False
    return bool(_lib.lib().b2no_mlp_head_bwd_multi_supported(x.shape[1], hidden, out_channels, math.prod(x.shape[2:])))


def mlp_head_fwd_multi(x, w1, b1, w2, b2, act="gelu") -> Optional[torch.Tensor]:
    """Ci -> hidden -> act -> O head, O = w2.shape[0] in 2..4, without the hidden tensor (b2no_mlp_head_fwd_multi).
    Returns (B, O, *grid), or None -- with nothing computed -- when the shape has no kernel."""
    B, ci = x.shape[:2]
    grid = tuple(x.shape[2:])
    hidden, O = w1.shape[0], w2.shape[0]
    per_sample = b1 is not None and b1.dim() == 2
    out = torch.empty((B, O) + grid, dtype=torch.float32, device=x.device)
    rc = _lib.lib().b2no_mlp_head_fwd_multi(_ptr(x), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), _ptr(out), B, ci, hidden, O,
                                            math.prod(grid), 1 if per_sample else 0, ACT[act], _stream())
    if rc == -2:
        return None
    check(rc, "mlp_head_fwd_multi")
    return out


def mlp_head_bwd_multi(x, w1, b1, w2, g, act="gelu", want_gz=True, dact_z=None, dact=None):
    """Input-gradient half of the backward of the Ci -> hidden -> act -> O head (b2no_mlp_head_bwd_multi), g (B, O, *grid).
    Returns (gx, gz | None, dw2 (O, hidden)) or None when the shape has no tensor-core kernel."""
    B, ci = x.shape[:2]
    grid = tuple(x.shape[2:])
    hidden, O = w1.shape[0], w2.shape[0]
    L = _lib.lib()
    per_sample = b1 is not None and b1.dim() == 2
    gx = torch.empty_like(x)
    gz = torch.empty((B, hidden) + grid, dtype=torch.float32, device=x.device) if want_gz else None
    dw2 = torch.empty((O, hidden), dtype=torch.float32, device=x.device)
    partial = torch.empty(int(L.b2no_mlp_head_bwd_multi_scratch_floats(hidden, O)), dtype=torch.float32, device=x.device)
    rc = L.b2no_mlp_head_bwd_multi(_ptr(x), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(g), _ptr(gx), _ptr(gz), _ptr(dw2), _ptr(partial),
                                   B, ci, hidden, O, math.prod(grid), 1 if per_sample else 0, ACT[act], _ptr(dact_z),
                                   ACT[dact] if dact_z is not None else 0, _stream())
    if rc == -2:
        return None
    check(rc, "mlp_head_bwd_multi")
    return gx, gz, dw2


def channel_mlp_supported(x: torch.Tensor, channels: int, hidden: int) -> bool:
    """True when the channel-MLP kernels (b2no_channel_mlp_fwd / _bwd) run for x: a CUDA tensor and a supported shape."""
    return x.is_cuda and bool(_lib.lib().b2no_channel_mlp_supported(channels, hidden, math.prod(x.shape[2:])))


def channel_mlp_fwd(u, x, w1, b1, w2, b2, g, act=None, want_pre=False):
    """s = gelu(W2 gelu(W1 u + b1) + b2) + g x, y = act(s) (b2no_channel_mlp_fwd): returns (y, pre | None), pre = s written when
    want_pre and act is set.  Every tensor contiguous float32; w1 (H, C), w2 (C, H), g (C)."""
    B, Cc = u.shape[:2]
    hidden = w1.shape[0]
    y = torch.empty_like(u)
    pre = torch.empty_like(u) if (want_pre and ACT[act]) else None
    check(_lib.lib().b2no_channel_mlp_fwd(_ptr(u), _ptr(x), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), _ptr(g), _ptr(y), _ptr(pre),
                                          B, Cc, hidden, math.prod(u.shape[2:]), ACT[act], _stream()), "channel_mlp_fwd")
    return y, pre


def channel_mlp_bwd(u, x, pre, gy, w1, b1, w2, b2, g, act=None):
    """Backward of channel_mlp_fwd (b2no_channel_mlp_bwd): returns (du, dx (the skip's share), h, d1, d2, dg)."""
    B, Cc = u.shape[:2]
    grid = tuple(u.shape[2:])
    hidden = w1.shape[0]
    L = _lib.lib()
    du, dx, d2 = torch.empty_like(u), torch.empty_like(u), torch.empty_like(u)
    h = torch.empty((B, hidden) + grid, dtype=torch.float32, device=u.device)
    d1 = torch.empty_like(h)
    dg = torch.empty((Cc,), dtype=torch.float32, device=u.device)
    scratch = torch.empty(int(L.b2no_channel_mlp_scratch_floats(Cc)), dtype=torch.float32, device=u.device)
    check(L.b2no_channel_mlp_bwd(_ptr(u), _ptr(x), _ptr(pre), _ptr(gy), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), _ptr(g), _ptr(du),
                                 _ptr(dx), _ptr(h), _ptr(d1), _ptr(d2), _ptr(dg), _ptr(scratch), B, Cc, hidden, math.prod(grid),
                                 ACT[act], _stream()), "channel_mlp_bwd")
    return du, dx, h, d1, d2, dg


def rno_gate_fwd(z, z2, hh, h):
    out = torch.empty_like(h)
    check(_lib.lib().b2no_rno_gate_fwd(_ptr(z), _ptr(z2), _ptr(hh), _ptr(h), _ptr(out), h.numel(), _stream()), "gate")
    return out


def rno_gate_bwd(g, z, z2, hh, h):
    outs = [torch.empty_like(h) for _ in range(4)]
    check(_lib.lib().b2no_rno_gate_bwd(_ptr(g), _ptr(z), _ptr(z2), _ptr(hh), _ptr(h), *[_ptr(o) for o in outs],
                                       h.numel(), _stream()), "gate_bwd")
    return outs


def rno_cell_bwd(g, h, zz2, ah, g_zz2, g_ah):
    """Pre-activation gradients of the fused RNO cell update (see include/b2no.h); g_zz2 / g_ah are written in place,
    returns the direct dh term g (1 - z)."""
    B, Cc = h.shape[:2]
    P = math.prod(h.shape[2:])
    g_h = torch.empty_like(h)
    for t in (g, h, zz2, ah, g_zz2, g_ah):
        assert t.is_contiguous() and t.dtype == torch.float32
    check(_lib.lib().b2no_rno_cell_bwd(_ptr(g), _ptr(h), _ptr(zz2), _ptr(ah), _ptr(g_zz2), _ptr(g_ah), _ptr(g_h), B, Cc, P,
                                       _stream()), "rno_cell_bwd")
    return g_h


def rno_reset_bwd(g_rh, h, ar, g_ar, g_h):
    """g_ar = g_rh h r (1 - r) (written in place), g_h += g_rh r, with r = sigmoid(ar)."""
    for t in (g_rh, h, ar, g_ar, g_h):
        assert t.is_contiguous() and t.dtype == torch.float32
    check(_lib.lib().b2no_rno_reset_bwd(_ptr(g_rh), _ptr(h), _ptr(ar), _ptr(g_ar), _ptr(g_h), h.numel(), _stream()),
          "rno_reset_bwd")


def rel_l2_sums(x, y):
    B = x.shape[0]
    n = x.numel() // B
    sums = torch.empty((B, 2), dtype=torch.float32, device=x.device)
    check(_lib.lib().b2no_rel_l2_sums(_ptr(x), _ptr(y), _ptr(sums), B, n, _stream()), "rel_l2_sums")
    return sums


def rel_l2_bwd(x, y, coef):
    B = x.shape[0]
    dx = torch.empty_like(x)
    check(_lib.lib().b2no_rel_l2_bwd(_ptr(x), _ptr(y), _ptr(coef), _ptr(dx), B, x.numel() // B, _stream()), "rel_l2_bwd")
    return dx


def rel_l2_finish(sums, size_average: bool):
    """sums (B, 2) -> (loss scalar tensor, coef (B,)): the tail of LpLoss.rel on the device, one launch."""
    B = sums.shape[0]
    loss = torch.empty((), dtype=torch.float32, device=sums.device)
    coef = torch.empty((B,), dtype=torch.float32, device=sums.device)
    check(_lib.lib().b2no_rel_l2_finish(_ptr(sums), _ptr(loss), _ptr(coef), B, 1 if size_average else 0, _stream()),
          "rel_l2_finish")
    return loss, coef


def rel_l2_bwd_g(x, y, coef, g):
    """dx = g * coef[b] * (x - y), g a 0-dim device tensor (the upstream gradient)."""
    B = x.shape[0]
    dx = torch.empty_like(x)
    check(_lib.lib().b2no_rel_l2_bwd_g(_ptr(x), _ptr(y), _ptr(coef), _ptr(g), _ptr(dx), B, x.numel() // B, _stream()),
          "rel_l2_bwd_g")
    return dx


def gather_segments(flat, ptr_table, offsets, counts, nseg: int):
    check(_lib.lib().b2no_gather_segments(_ptr(flat), _ptr(ptr_table), _ptr(offsets), _ptr(counts), nseg, _stream()),
          "gather_segments")



def pino_residual_supported(n: int) -> bool:
    return 8 <= n <= 64 and n % 4 == 0


def pino_residual_fwd(w, u0, forcing2d, nu, t_interval: float):
    """Fused PINO residual + IC loss (csrc/pino_loss.cu).  w (B, N, N, T), u0 (B, N, N), forcing2d (N, N), nu (B,).
    Returns (loss2 = [loss_ic, loss_f], coef (B, 2), du_p (B, T, N, N), fields (4, B, T, N, N))."""
    _require_cuda(w, u0, forcing2d, nu)
    B, N, _, T = w.shape
    for t in (w, u0, forcing2d, nu):
        assert t.dtype == torch.float32 and t.is_contiguous()
    dev = w.device
    du_p = torch.empty((B, T, N, N), dtype=torch.float32, device=dev)
    fields = torch.empty((4, B, T, N, N), dtype=torch.float32, device=dev)
    partial = torch.empty((B, T, 4), dtype=torch.float32, device=dev)
    loss2 = torch.empty((2,), dtype=torch.float32, device=dev)
    coef = torch.empty((B, 2), dtype=torch.float32, device=dev)
    check(_lib.lib().b2no_pino_residual_fwd(_ptr(w), _ptr(u0), _ptr(forcing2d), _ptr(nu), float(t_interval), _ptr(du_p),
                                            _ptr(fields), _ptr(partial), _ptr(loss2), _ptr(coef), B, N, T, _stream()),
          "pino_residual_fwd")
    return loss2, coef, du_p, fields


def pino_residual_bwd(w, u0, forcing2d, nu, t_interval: float, du_p, fields, coef, gup):
    """dw (B, N, N, T) = gup[0] d loss_ic / dw + gup[1] d loss_f / dw."""
    B, N, _, T = w.shape
    assert gup.dtype == torch.float32 and gup.is_contiguous() and gup.numel() == 2
    dw = torch.empty_like(w)
    check(_lib.lib().b2no_pino_residual_bwd(_ptr(w), _ptr(u0), _ptr(forcing2d), _ptr(nu), float(t_interval), _ptr(du_p),
                                            _ptr(fields), _ptr(coef), _ptr(gup), _ptr(dw), B, N, T, _stream()),
          "pino_residual_bwd")
    return dw
