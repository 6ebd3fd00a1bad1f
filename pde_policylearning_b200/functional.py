"""Autograd layer over the C-ABI ops: forward and hand-derived backward of the fused blocks.

The math is SURVEY.md 8a.0 (verified against the reference by oracle/closed_form.py):

    Xh  = s_f DFT_trunc(x)                   Yh = sum_i Xh W            y = act(s_i IDFT_trunc(Yh) + bias + Wp x)
    gz  = gy act'(z)                         gYh = adj_inverse(gz)      dW = sum_b conj(Xh) gYh
    gXh = sum_o gYh conj(W)                  dx  = adj_forward(gXh) + Wp^T gz       dWp = sum gz x^T
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence

import torch

from . import ops
from .ops import SpecGeom, get_plan


def _contig(t: torch.Tensor) -> torch.Tensor:
    return t if t.is_contiguous() else t.contiguous()


def _fused_wgrad_ok(g: torch.Tensor) -> bool:
    """The dx pass may also compute the 1x1 weight gradient (ops.dft_inverse_wgrad, which itself declines shapes it does
    not support): CUDA tensors only."""
    return g.is_cuda


def _geom_has_overlap(geom: SpecGeom) -> bool:
    g = geom.resolved()
    return any(2 * g.half[j] > g.nfft[j] for j in range(g.ndim - 1))


class SpectralBlockFn(torch.autograd.Function):
    """y = act( spectral_conv(x; corners) + bias + pw_w @ x ) -- FNOBlocks layer (fno_block.py:131-150),
    FourierLayer2d (rno.py:224-228), PINO layer (pinobserver.py:222-226) and, with pw_w=None, the bare
    spectral convolutions (spectral_convolution.py:303-347, rno.py:60-77, basics.py:114-143)."""

    @staticmethod
    def forward(ctx, x, bias, pw_w, geom: SpecGeom, act, *corners):
        ops._require_cuda(x)
        x = _contig(x.float())
        plan = get_plan(geom, x.device)
        B, ci = x.shape[:2]
        co = corners[0].shape[1]
        if corners[0].shape[0] != ci:
            raise ValueError(f"input has {ci} channels, weights expect {corners[0].shape[0]}")
        det = [c.detach() for c in corners]
        xh = ops.dft_forward(plan, 0, x)
        yh = ops.mix(plan, 0, xh, det, ci, co)
        need_z = act not in (None, "none") and any(ctx.needs_input_grad)
        grid = plan.geom.nout
        z = torch.empty((B, co) + tuple(grid), dtype=torch.float32, device=x.device) if need_z else None
        pw2d = None
        if pw_w is not None:
            if tuple(plan.geom.nout) != tuple(plan.geom.nin):
                raise NotImplementedError("fused 1x1 skip needs matching input/output grids")
            pw2d = _contig(pw_w.detach().reshape(pw_w.shape[0], -1).float())
        epi = ops.make_epilogue(bias=None if bias is None else _contig(bias.detach().reshape(-1).float()),
                                pw_w=pw2d, pw_x=x if pw2d is not None else None, preact=z, act=act)
        y = ops.dft_inverse(plan, 0, yh, epi)
        ctx.geom, ctx.act = geom, act
        ctx.has_bias, ctx.has_pw = bias is not None, pw_w is not None
        ctx.pw_shape = None if pw_w is None else tuple(pw_w.shape)
        ctx.bias_shape = None if bias is None else tuple(bias.shape)
        ctx.save_for_backward(x, xh, z, pw2d, *det)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, xh, z, pw2d, *det = ctx.saved_tensors
        geom, act = ctx.geom, ctx.act
        plan = get_plan(geom, x.device)
        B, ci = x.shape[:2]
        co = det[0].shape[1]
        gy = _contig(gy.float())
        gz = ops.act_bwd(gy, z, act) if z is not None else gy
        need_x, need_b, need_pw = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        need_w = any(ctx.needs_input_grad[5:])
        gyh = ops.dft_forward(plan, 1, gz)
        dbias = dpw = dx = None
        dcorners: List[Optional[torch.Tensor]] = [None] * len(det)
        if need_w:
            dcorners = ops.mix_dw(plan, xh, gyh, det, needs_zero=_geom_has_overlap(geom))
        fused = None
        if need_x:
            gxh = ops.mix(plan, 1, gyh, det, ci, co)
            epi = ops.make_epilogue(pw_w=pw2d, pw_x=gz if pw2d is not None else None, pw_transposed=True)
            if need_pw and _fused_wgrad_ok(gz):
                fused = ops.dft_inverse_wgrad(plan, 1, gxh, epi, x, need_bias=need_b)
            dx = fused[0] if fused is not None else ops.dft_inverse(plan, 1, gxh, epi)
        if need_pw:
            dpw, db2 = fused[1:] if fused is not None else ops.pw_wgrad(gz, x, need_bias=need_b)
            dpw = dpw.reshape(ctx.pw_shape)
            if need_b:
                dbias = db2.reshape(ctx.bias_shape)
        elif need_b:
            # dbias[o] = sum_{b,n} gz = DC mode of the (scaled) truncated DFT: gYh[b,o,0..0] = s_i * sum_n gz
            dc = gyh.reshape(B, co, -1)[:, :, 0].real.sum(dim=0) / plan.s_i
            dbias = dc.reshape(ctx.bias_shape)
        return (dx, dbias, dpw, None, None) + tuple(dcorners)


def spectral_block(x, corners: Sequence[torch.Tensor], geom: SpecGeom, bias=None, pw_weight=None, act=None):
    return SpectralBlockFn.apply(x, bias, pw_weight, geom, act, *corners)


class FNOStackFn(torch.autograd.Function):
    """n_layers x [ y = act_l( spectral_conv_l(x) + bias_l + skip_l x ) ] as ONE autograd node (FNO.forward's loop over
    FNOBlocks, tfno.py:203-204 + fno_block.py:131-150).  Same kernels as SpectralBlockFn, but the backward chains the
    layers: the dx pass of layer l multiplies by act'(z_{l-1}) in its epilogue and so emits gz_{l-1} directly -- no
    separate activation-backward pass over the activations.

    bias_all = the (n_layers, Co, 1, ...) bias parameter of the conv stack (spectral_convolution.py:271-272), taken whole
    so that its gradient is written once by the weight-gradient kernels instead of being assembled from per-layer
    slices; params = for each layer: pw_w (Co, Ci, 1...) | n_corners corner tensors."""

    @staticmethod
    def forward(ctx, x, geom: SpecGeom, acts, n_corners, bias_all, *params):
        ops._require_cuda(x)
        x = _contig(x.float())
        plan = get_plan(geom, x.device)
        per = 1 + n_corners
        L = len(params) // per
        need_grad = any(ctx.needs_input_grad)
        saved, meta = [], []
        cur = x
        b2d = _contig(bias_all.detach().reshape(L, -1).float())
        for l in range(L):
            pw_w = params[l * per]
            det = [c.detach() for c in params[l * per + 1:(l + 1) * per]]
            B, ci = cur.shape[:2]
            co = det[0].shape[1]
            xh = ops.dft_forward(plan, 0, cur)
            yh = ops.mix(plan, 0, xh, det, ci, co)
            act = acts[l]
            need_z = act not in (None, "none") and need_grad
            z = torch.empty((B, co) + tuple(plan.geom.nout), dtype=torch.float32, device=x.device) if need_z else None
            pw2d = _contig(pw_w.detach().reshape(pw_w.shape[0], -1).float())
            epi = ops.make_epilogue(bias=b2d[l], pw_w=pw2d, pw_x=cur, preact=z, act=act)
            y = ops.dft_inverse(plan, 0, yh, epi)
            saved += [cur, xh, z if z is not None else cur.new_empty(0), pw2d] + det
            meta.append((tuple(pw_w.shape), ci, co, need_z))
            cur = y
        ctx.geom, ctx.acts, ctx.n_corners, ctx.meta = geom, acts, n_corners, meta
        ctx.bias_shape = tuple(bias_all.shape)
        ctx.save_for_backward(*saved)
        return cur

    @staticmethod
    def backward(ctx, gy):
        geom, acts, nc, meta = ctx.geom, ctx.acts, ctx.n_corners, ctx.meta
        saved = ctx.saved_tensors
        per_s = 4 + nc
        L = len(meta)
        plan = get_plan(geom, gy.device)
        per = 1 + nc
        grads = [None] * (L * per)
        need_bias = ctx.needs_input_grad[4]
        dbias = gy.new_empty((L, meta[0][2])) if need_bias else None
        g = _contig(gy.float())
        # top layer: gradient w.r.t. its pre-activation
        if meta[L - 1][3]:
            g = ops.act_bwd(g, saved[(L - 1) * per_s + 2], acts[L - 1])
        for l in range(L - 1, -1, -1):
            x, xh, _, pw2d = saved[l * per_s: l * per_s + 4]
            det = list(saved[l * per_s + 4: (l + 1) * per_s])
            pw_shape, ci, co, _ = meta[l]
            need = ctx.needs_input_grad[5 + l * per: 5 + (l + 1) * per]
            gyh = ops.dft_forward(plan, 1, g)
            if any(need[1:]):
                dcs = ops.mix_dw(plan, xh, gyh, det, needs_zero=_geom_has_overlap(geom))
                for j in range(nc):
                    grads[l * per + 1 + j] = dcs[j]
            need_wgrad = need_bias or need[0]
            db_out = dbias[l] if need_bias else None
            fused = None
            if l > 0 or ctx.needs_input_grad[0]:
                gxh = ops.mix(plan, 1, gyh, det, ci, co)
                zprev = saved[(l - 1) * per_s + 2] if (l > 0 and meta[l - 1][3]) else None
                epi = ops.make_epilogue(pw_w=pw2d, pw_x=g, pw_transposed=True, dact_z=zprev,
                                        dact=acts[l - 1] if zprev is not None else None)
                # the dx pass reads g tile by tile anyway: it also computes dWp and dbias[l] when it can
                if need_wgrad and _fused_wgrad_ok(g):
                    fused = ops.dft_inverse_wgrad(plan, 1, gxh, epi, x, need_bias=need_bias, db_out=db_out)
                if fused is None:
                    if need_wgrad:
                        dpw, _ = ops.pw_wgrad(g, x, need_bias=need_bias, db_out=db_out)
                        grads[l * per] = dpw.reshape(pw_shape)
                    g = ops.dft_inverse(plan, 1, gxh, epi)
                else:
                    g = fused[0]
                    grads[l * per] = fused[1].reshape(pw_shape)
            elif need_wgrad:
                dpw, _ = ops.pw_wgrad(g, x, need_bias=need_bias, db_out=db_out)
                grads[l * per] = dpw.reshape(pw_shape)
        return (g if ctx.needs_input_grad[0] else None, None, None, None,
                dbias.reshape(ctx.bias_shape) if need_bias else None) + tuple(grads)


def fno_stack(x, geom: SpecGeom, bias_all, layers, acts):
    """bias_all: (n_layers, Co, 1, ...) bias of the conv stack; layers: list of (pw_weight, [corners]); acts: activation
    name (or None) per layer."""
    flat = []
    for pw_w, corners in layers:
        flat += [pw_w] + list(corners)
    return FNOStackFn.apply(x, geom, tuple(acts), len(layers[0][1]), bias_all, *flat)


class PointwiseConvFn(torch.autograd.Function):
    """y = act(W x + b), channels-first 1x1 convolution (tfno.py:11-38 Lifting / Projection convs,
    skip_connections.py:31)."""

    @staticmethod
    def forward(ctx, x, weight, bias, act):
        ops._require_cuda(x)
        x = _contig(x.float())
        B, ci = x.shape[:2]
        grid = tuple(x.shape[2:])
        w2d = _contig(weight.detach().reshape(weight.shape[0], -1).float())
        co = w2d.shape[0]
        if w2d.shape[1] != ci:
            raise ValueError(f"input has {ci} channels, weight expects {w2d.shape[1]}")
        need_z = act not in (None, "none") and any(ctx.needs_input_grad)
        z = torch.empty((B, co) + grid, dtype=torch.float32, device=x.device) if need_z else None
        epi = ops.make_epilogue(bias=None if bias is None else _contig(bias.detach().float()), pw_w=w2d, pw_x=x,
                                preact=z, act=act)
        y = ops.pointwise(B, co, grid, x.device, epi)
        ctx.act = act
        ctx.w_shape = tuple(weight.shape)
        ctx.save_for_backward(x, z, w2d)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, z, w2d = ctx.saved_tensors
        gy = _contig(gy.float())
        gz = ops.act_bwd(gy, z, ctx.act) if z is not None else gy
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            epi = ops.make_epilogue(pw_w=w2d, pw_x=gz, pw_transposed=True)
            dx = ops.pointwise(x.shape[0], x.shape[1], tuple(x.shape[2:]), x.device, epi)
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dw, db = ops.pw_wgrad(gz, x, need_bias=ctx.needs_input_grad[2])
            dw = dw.reshape(ctx.w_shape)
        return dx, dw, db, None


def pointwise_conv(x, weight, bias=None, act=None):
    return PointwiseConvFn.apply(x, weight, bias, act)


class PointwiseConv2Fn(torch.autograd.Function):
    """y = act(W x + W2 x2 + b): two channels-first operands on the same grid (used where a per-sample
    scalar such as the Reynolds number enters as an extra 1-channel map, pinobserver.py:51-58)."""

    @staticmethod
    def forward(ctx, x, weight, bias, act, x2, weight2):
        ops._require_cuda(x, x2)
        x, x2 = _contig(x.float()), _contig(x2.float())
        B, ci = x.shape[:2]
        grid = tuple(x.shape[2:])
        if tuple(x2.shape[2:]) != grid or x2.shape[0] != B:
            raise ValueError("both operands must share batch and grid")
        w2d = _contig(weight.detach().reshape(weight.shape[0], -1).float())
        w2d2 = _contig(weight2.detach().reshape(weight2.shape[0], -1).float())
        co = w2d.shape[0]
        need_z = act not in (None, "none") and any(ctx.needs_input_grad)
        z = torch.empty((B, co) + grid, dtype=torch.float32, device=x.device) if need_z else None
        epi = ops.make_epilogue(bias=None if bias is None else _contig(bias.detach().float()), pw_w=w2d, pw_x=x,
                                pw2_w=w2d2, pw2_x=x2, preact=z, act=act)
        y = ops.pointwise(B, co, grid, x.device, epi)
        ctx.act = act
        ctx.w_shape, ctx.w2_shape = tuple(weight.shape), tuple(weight2.shape)
        ctx.save_for_backward(x, x2, z, w2d, w2d2)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, x2, z, w2d, w2d2 = ctx.saved_tensors
        gy = _contig(gy.float())
        gz = ops.act_bwd(gy, z, ctx.act) if z is not None else gy
        dx = dw = db = dx2 = dw2 = None
        if ctx.needs_input_grad[0]:
            dx = ops.pointwise(x.shape[0], x.shape[1], tuple(x.shape[2:]), x.device,
                               ops.make_epilogue(pw_w=w2d, pw_x=gz, pw_transposed=True))
        if ctx.needs_input_grad[4]:
            dx2 = ops.pointwise(x2.shape[0], x2.shape[1], tuple(x2.shape[2:]), x2.device,
                                ops.make_epilogue(pw_w=w2d2, pw_x=gz, pw_transposed=True))
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dw, db = ops.pw_wgrad(gz, x, need_bias=ctx.needs_input_grad[2])
            dw = dw.reshape(ctx.w_shape)
        if ctx.needs_input_grad[5]:
            dw2, _ = ops.pw_wgrad(gz, x2, need_bias=False)
            dw2 = dw2.reshape(ctx.w2_shape)
        return dx, dw, db, None, dx2, dw2


def pointwise_conv2(x, weight, bias, act, x2, weight2):
    return PointwiseConv2Fn.apply(x, weight, bias, act, x2, weight2)


class MlpHeadFn(torch.autograd.Function):
    """out = b2 + w2 . act(W1 x + b1), out_channels == 1 (tfno.py:34-38, pinobserver.py:230-232, rno.py:170-174).
    The hidden tensor is never stored: the backward recomputes it on the tensor cores (csrc/tc_mlp.cu), emits
    gx and dw2 directly and writes gz = g w2 act'(z1) once for the weight-gradient kernel."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, act):
        ops._require_cuda(x)
        x = _contig(x.float())
        w1m = _contig(w1.detach().reshape(w1.shape[0], -1).float())
        w2v = _contig(w2.detach().reshape(-1).float())
        b1c = None if b1 is None else _contig(b1.detach().float())
        out = ops.mlp_head_fwd(x, w1m, b1c, w2v, None if b2 is None else _contig(b2.detach().float()), act)
        ctx.act = act
        ctx.shapes = (tuple(w1.shape), None if b1 is None else tuple(b1.shape), tuple(w2.shape),
                      None if b2 is None else tuple(b2.shape))
        ctx.save_for_backward(x, w1m, b1c, w2v)
        return out

    @staticmethod
    def backward(ctx, g):
        x, w1m, b1c, w2v = ctx.saved_tensors
        g = _contig(g.float())
        need_x, need_w1, need_b1, need_w2, need_b2 = ctx.needs_input_grad[:5]
        per_sample_b1 = b1c is not None and b1c.dim() == 2
        if (not per_sample_b1 and g.data_ptr() % 16 == 0
                and ops.mlp_head_bwd_fused_supported(x.shape[1], w1m.shape[0], math.prod(x.shape[2:]))):
            # one kernel: gx, dW1, db1, dw2 (csrc/tc_head_bwd.cu)
            gx, dw1, db1, dw2, db2 = ops.mlp_head_bwd_fused(x, w1m, b1c, w2v, g, ctx.act)
            db2 = db2.reshape(ctx.shapes[3]) if need_b2 else None
            return (gx if need_x else None, dw1.reshape(ctx.shapes[0]) if need_w1 else None,
                    db1.reshape(ctx.shapes[1]) if (need_b1 and b1c is not None) else None,
                    dw2.reshape(ctx.shapes[2]) if need_w2 else None, db2, None)
        res = ops.mlp_head_bwd(x, w1m, b1c, w2v, g, ctx.act, want_gz=need_w1 or need_b1)
        if res is None:
            raise RuntimeError("mlp_head backward: shape lost its tensor-core kernel between forward and backward")
        gx, gz, dw2 = res
        dw1 = db1 = None
        if need_w1 or need_b1:
            per_sample = b1c is not None and b1c.dim() == 2
            dw1, db1 = ops.pw_wgrad(gz, x, need_bias=need_b1 and not per_sample)
            dw1 = dw1.reshape(ctx.shapes[0])
            if need_b1 and per_sample:
                db1 = gz.sum(dim=tuple(range(2, gz.dim())))
            if db1 is not None:
                db1 = db1.reshape(ctx.shapes[1])
        db2 = g.sum().reshape(ctx.shapes[3]) if need_b2 else None
        return (gx if need_x else None, dw1 if need_w1 else None, db1 if need_b1 else None,
                dw2.reshape(ctx.shapes[2]) if need_w2 else None, db2, None)


class MlpHeadMultiFn(torch.autograd.Function):
    """out[:, o] = b2[o] + w2[o] . act(W1 x + b1) for 2..4 outputs: PINObserverFullField's tail (plane_num * out_dim channels,
    pinobserver.py:230-232) and Projection with out_channels > 1 (tfno.py:34-38).  Like MlpHeadFn, the hidden tensor is never
    stored: the backward recomputes it on the tensor cores (csrc/tc_mlp.cu), emits gx and dW2 directly and writes
    gz = act'(z1) sum_o g[o] w2[o] once for the weight-gradient kernel."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, act):
        ops._require_cuda(x)
        x = _contig(x.float())
        w1m = _contig(w1.detach().reshape(w1.shape[0], -1).float())
        w2m = _contig(w2.detach().reshape(w2.shape[0], -1).float())
        b1c = None if b1 is None else _contig(b1.detach().float())
        out = ops.mlp_head_fwd_multi(x, w1m, b1c, w2m, None if b2 is None else _contig(b2.detach().float()), act)
        if out is None:
            raise RuntimeError("mlp_head: the multi-output head kernel declined a shape mlp_head_fused_available accepted")
        ctx.act = act
        ctx.shapes = (tuple(w1.shape), None if b1 is None else tuple(b1.shape), tuple(w2.shape),
                      None if b2 is None else tuple(b2.shape))
        ctx.save_for_backward(x, w1m, b1c, w2m)
        return out

    @staticmethod
    def backward(ctx, g):
        x, w1m, b1c, w2m = ctx.saved_tensors
        g = _contig(g.float())
        need_x, need_w1, need_b1, need_w2, need_b2 = ctx.needs_input_grad[:5]
        res = ops.mlp_head_bwd_multi(x, w1m, b1c, w2m, g, ctx.act, want_gz=need_w1 or need_b1)
        if res is None:
            raise RuntimeError("mlp_head backward: shape lost its tensor-core kernel between forward and backward")
        gx, gz, dw2 = res
        dw1 = db1 = None
        if need_w1 or need_b1:
            per_sample = b1c is not None and b1c.dim() == 2
            dw1, db1 = ops.pw_wgrad(gz, x, need_bias=need_b1 and not per_sample)
            dw1 = dw1.reshape(ctx.shapes[0])
            if need_b1 and per_sample:
                db1 = gz.sum(dim=tuple(range(2, gz.dim())))
            if db1 is not None:
                db1 = db1.reshape(ctx.shapes[1])
        db2 = g.sum(dim=[0] + list(range(2, g.dim()))).reshape(ctx.shapes[3]) if need_b2 else None
        return (gx if need_x else None, dw1 if need_w1 else None, db1 if need_b1 else None,
                dw2.reshape(ctx.shapes[2]) if need_w2 else None, db2, None)


def mlp_head_fused_available(x, w1, w2, b1, needs_grad: bool) -> bool:
    """True when mlp_head() runs the fused tensor-core head for these operands (the hidden tensor is never materialised).
    One output: the kernels of MlpHeadFn; 2..4 outputs: those of MlpHeadMultiFn, in training and inference alike."""
    n_out = w2.reshape(-1, w1.shape[0]).shape[0]
    if 2 <= n_out <= 4 and (b1 is None or b1.dim() <= 2):
        return ops.mlp_head_multi_supported(x, w1.shape[0], n_out)
    if not x.is_cuda or n_out != 1 or (b1 is not None and b1.dim() > 2):
        return False
    if needs_grad:
        return bool(ops.mlp_head_bwd_supported(x.shape[1], w1.shape[0], math.prod(x.shape[2:]))) and x.data_ptr() % 16 == 0
    return x.shape[1] in (8, 16, 32, 64)


def mlp_head(x, w1, b1, w2, b2, act="gelu"):
    """Projection head Ci -> hidden -> act -> O (tfno.py:34-38).  For O = 1..4 the fused kernels never materialise the
    hidden tensor in the forward; other O and shapes without a fused kernel compose two pointwise convs (hidden saved for
    backward)."""
    ops._require_cuda(x, w1, b1, w2, b2)
    needs_grad = torch.is_grad_enabled() and any(
        t is not None and t.requires_grad for t in (x, w1, b1, w2, b2))
    if mlp_head_fused_available(x, w1, w2, b1, needs_grad):
        if w2.reshape(-1, w1.shape[0]).shape[0] > 1:
            if needs_grad:
                return MlpHeadMultiFn.apply(x, w1, b1, w2, b2, act)
            out = ops.mlp_head_fwd_multi(_contig(x.float()), _contig(w1.reshape(w1.shape[0], -1).float()),
                                         None if b1 is None else _contig(b1.float()),
                                         _contig(w2.reshape(w2.shape[0], -1).float()),
                                         None if b2 is None else _contig(b2.float()), act)
            if out is None:
                raise RuntimeError("mlp_head: the multi-output head kernel declined a shape mlp_head_fused_available accepted")
            return out
        if needs_grad:
            return MlpHeadFn.apply(x, w1, b1, w2, b2, act)
        return ops.mlp_head_fwd(_contig(x.float()), _contig(w1.reshape(w1.shape[0], -1).float()),
                                None if b1 is None else _contig(b1.float()), _contig(w2.reshape(-1).float()),
                                None if b2 is None else _contig(b2.float()), act)
    if b1 is not None and b1.dim() == 2:
        # the composed path's epilogue reads bias[o] only: a (batch, hidden) bias would silently use sample 0's row
        raise ValueError("mlp_head: a per-sample bias needs the fused head kernel (mlp_head_fused_available); pass the "
                         "per-sample term as a 1-channel map through pointwise_conv2 instead")
    h = pointwise_conv(x, w1, b1, act)
    return pointwise_conv(h, w2, b2, None)


class RelL2Fn(torch.autograd.Function):
    """LpLoss.rel with p=2 (libs/utilities3.py:323-334): sum_b or mean_b of ||x_b - y_b|| / ||y_b||.  Three launches in
    all: per-sample sums, the scalar tail (sqrt, ratio, sum) on the device, and dx = g coef_b (x - y)."""

    @staticmethod
    def forward(ctx, x, y, size_average):
        ops._require_cuda(x, y)
        B = x.shape[0]
        xf, yf = _contig(x.float()).reshape(B, -1), _contig(y.float()).reshape(B, -1)
        sums = ops.rel_l2_sums(xf, yf)
        loss, coef = ops.rel_l2_finish(sums, bool(size_average))
        ctx.save_for_backward(xf, yf, coef, sums)
        ctx.x_shape, ctx.y_shape = tuple(x.shape), tuple(y.shape)
        return loss

    @staticmethod
    def backward(ctx, g):
        xf, yf, coef, sums = ctx.saved_tensors
        dx = ops.rel_l2_bwd_g(xf, yf, coef, _contig(g.float()))
        dy = None
        if ctx.needs_input_grad[1]:
            # LpLoss.rel is differentiable in the target too (libs/utilities3.py:323-334):
            #   d/dy ||x-y|| / ||y|| = -(x-y) / (||x-y|| ||y||) - ||x-y|| y / ||y||^3 = -dx/g - coef (||x-y||^2 / ||y||^2) y
            ratio = (g.float() * coef * sums[:, 0] / sums[:, 1]).reshape(-1, 1)
            dy = (-dx - ratio * yf).reshape(ctx.y_shape)
        return dx.reshape(ctx.x_shape), dy, None


def rel_l2_loss(x, y, size_average=True):
    return RelL2Fn.apply(x, y, size_average)


class RnoGateFn(torch.autograd.Function):
    """h_next = (1 - z) * h + z2 * hhat  (rno.py:259)."""

    @staticmethod
    def forward(ctx, z, z2, hhat, h):
        z, z2, hhat, h = (_contig(t.float()) for t in (z, z2, hhat, h))
        ctx.save_for_backward(z, z2, hhat, h)
        return ops.rno_gate_fwd(z, z2, hhat, h)

    @staticmethod
    def backward(ctx, g):
        z, z2, hhat, h = ctx.saved_tensors
        return tuple(ops.rno_gate_bwd(_contig(g.float()), z, z2, hhat, h))


def rno_gate(z, z2, hhat, h):
    return RnoGateFn.apply(z, z2, hhat, h)


# =============================================================================================
# RNO layer: the GRU-style recurrent cell of rno.py:254-290 as ONE autograd node over all time steps
# =============================================================================================
_RNO_XCHUNK = 8192      # planes-batches per x-side launch (bounds the A' workspace and gridDim.y)


class RnoLayerFn(torch.autograd.Function):
    """h_t = cell(x_t, h_{t-1}) for t = 0..T'-1 (RNO_layer.forward, rno.py:275-290; RNO_cell.forward, rno.py:254-260).

    The reference evaluates eight FourierLayer2d per step, each with its own rfft2 / irfft2.  Every f_k is LINEAR, so the
    cell is regrouped (same sums, SURVEY.md 8f rank 1):

      x side, no recurrence -> hoisted over ALL T' frames and batched:   Xh = F(x);  Gx_g = F^-1(Xh W_g) + P_g x + bias_g
                                                                         for the gate groups g = [z | z2], r, hhat
      h side, per step:   Hh = F(h)
                          [z | z2] = sigmoid(F^-1(Hh [W2 | W8]) + [Wc2; Wc8] h + Gx_zz2[t])          one inverse, 2C channels
                          r h      = sigmoid(F^-1(Hh W4) + Wc4 h + Gx_r[t]) * h                       `mul` epilogue
                          h'       = (1 - z) h + z2 selu(F^-1(F(r h) W6) + Wc6 (r h) + Gx_h[t])      gate epilogue

    i.e. 2 forward + 3 inverse transforms per recurrent step instead of 8 + 8, all sigmoid / SELU / gate arithmetic inside
    the inverse-transform epilogues.  The backward walks the steps in reverse (BPTT) with the adjoint kernels, accumulating
    the weight gradients of all steps in place, and does the x side once, batched.

    x_tm: (T', B, C, H, W) time-major; h0: (B, C, H, W); params: for k = 1..8 (fourier_weight.0, fourier_weight.1,
    norm_conv1d.weight, norm_conv1d.bias), then b1..b4 (rno.py:249-252)."""

    @staticmethod
    def forward(ctx, x_tm, h0, geom: SpecGeom, return_sequences: bool, *params):
        ops._require_cuda(x_tm, h0)
        x_tm, h0 = _contig(x_tm.float()), _contig(h0.float())
        Tn, B, Cc, H, W = x_tm.shape
        plan, geom = _rno_plan(geom, x_tm.device, B, Cc)
        pk = _rno_pack(params, Cc)
        xf = x_tm.reshape(Tn * B, Cc, H, W)
        # ---- x side, batched over whole frames ----
        Gzz2 = torch.empty((Tn * B, 2 * Cc, H, W), dtype=torch.float32, device=xf.device)
        Gr = torch.empty((Tn * B, Cc, H, W), dtype=torch.float32, device=xf.device)
        Gh = torch.empty_like(Gr)
        chunk = max(1, _RNO_XCHUNK // B) * B
        Xh = []                                  # one spectrum per chunk (a mode-major spectrum cannot be sliced by batch)
        for s in range(0, Tn * B, chunk):
            e = min(Tn * B, s + chunk)
            xs = xf[s:e]
            xh = ops.dft_forward(plan, 0, xs)
            Xh.append(xh)
            for Wc, Pm, bias, co, G in ((pk["Wx_zz2"], pk["Px_zz2"], pk["bias_zz2"], 2 * Cc, Gzz2),
                                        (pk["Wx_r"], pk["Px_r"], pk["bias_r"], Cc, Gr),
                                        (pk["Wx_h"], pk["Px_h"], pk["bias_h"], Cc, Gh)):
                S = ops.mix(plan, 0, xh, Wc, Cc, co)
                ops.dft_inverse(plan, 0, S, ops.make_epilogue(bias=bias, pw_w=Pm, pw_x=xs), out=G[s:e])
        Gzz2, Gr, Gh = (G.reshape(Tn, B, -1, H, W) for G in (Gzz2, Gr, Gh))
        # ---- recurrence ----
        need_grad = any(ctx.needs_input_grad)
        hs = []
        saved = []
        h = h0
        for t in range(Tn):
            Hh = ops.dft_forward(plan, 0, h)
            S = ops.mix(plan, 0, Hh, pk["Wh_zz2"], Cc, 2 * Cc)
            zz2 = ops.dft_inverse(plan, 0, S, ops.make_epilogue(pw_w=pk["Ph_zz2"], pw_x=h, add=Gzz2[t], act="sigmoid"))
            S = ops.mix(plan, 0, Hh, pk["Wh_r"], Cc, Cc)
            ar = torch.empty_like(h) if need_grad else None
            rh = ops.dft_inverse(plan, 0, S, ops.make_epilogue(pw_w=pk["Ph_r"], pw_x=h, add=Gr[t], act="sigmoid", mul=h,
                                                                preact=ar))
            RHh = ops.dft_forward(plan, 0, rh)
            S = ops.mix(plan, 0, RHh, pk["W6"], Cc, Cc)
            ah = torch.empty_like(h) if need_grad else None
            hn = ops.dft_inverse(plan, 0, S, ops.make_epilogue(pw_w=pk["P6"], pw_x=rh, add=Gh[t], act="selu", preact=ah,
                                                                mul=zz2[:, Cc:], gate_z=zz2[:, :Cc], gate_h=h))
            if return_sequences:
                hs.append(hn)
            if need_grad:
                saved += [h, Hh, zz2, ar, rh, RHh, ah]
            h = hn
        ctx.geom, ctx.dims, ctx.return_sequences = geom, (Tn, B, Cc, H, W), return_sequences
        ctx.param_shapes = [tuple(p.shape) for p in params]
        ctx.n_chunks, ctx.chunk = len(Xh), chunk
        if need_grad:
            ctx.save_for_backward(xf, *Xh, *[p.detach() for p in params], *saved)
        return torch.stack(hs, dim=0) if return_sequences else h

    @staticmethod
    def backward(ctx, gout):
        Tn, B, Cc, H, W = ctx.dims
        geom = ctx.geom
        sv = ctx.saved_tensors
        nch = ctx.n_chunks
        xf, Xh = sv[0], sv[1:1 + nch]
        params = sv[1 + nch:37 + nch]
        steps = sv[37 + nch:]
        plan = get_plan(geom, xf.device)
        pk = _rno_pack(params, Cc)
        dev = xf.device
        gout = _contig(gout.float())
        gGzz2 = torch.empty((Tn, B, 2 * Cc, H, W), dtype=torch.float32, device=dev)
        gGr = torch.empty((Tn, B, Cc, H, W), dtype=torch.float32, device=dev)
        gGh = torch.empty_like(gGr)
        overlap = _geom_has_overlap(geom)
        zl = torch.zeros_like if overlap else torch.empty_like
        dWh_zz2 = [zl(w) for w in pk["Wh_zz2"]]
        dWh_r = [zl(w) for w in pk["Wh_r"]]
        dW6 = [zl(w) for w in pk["W6"]]
        dPh_zz2 = dPh_r = dP6 = None

        def acc_(a, d):
            return d if a is None else a.add_(d)

        g = gout[Tn - 1] if ctx.return_sequences else gout
        first = True
        for t in range(Tn - 1, -1, -1):
            h, Hh, zz2, ar, rh, RHh, ah = steps[7 * t: 7 * t + 7]
            if ctx.return_sequences and t < Tn - 1:
                g = g + gout[t]
            g_hdir = ops.rno_cell_bwd(_contig(g), h, zz2, ah, gGzz2[t], gGh[t])
            g_ah = gGh[t]
            # candidate-state branch: a_h = F^-1(F(rh) W6) + Wc6 rh + Gx_h
            gY = ops.dft_forward(plan, 1, g_ah)
            ops.mix_dw(plan, RHh, gY, pk["W6"], False, out=dW6, accumulate=not first)
            gRH = ops.mix(plan, 1, gY, pk["W6"], Cc, Cc)
            g_rh = ops.dft_inverse(plan, 1, gRH, ops.make_epilogue(pw_w=pk["P6"], pw_x=g_ah, pw_transposed=True))
            dP6 = acc_(dP6, ops.pw_wgrad(g_ah, rh, need_bias=False)[0])
            ops.rno_reset_bwd(g_rh, h, ar, gGr[t], g_hdir)
            g_azz2, g_ar = gGzz2[t], gGr[t]
            # gates: [a_z | a_z2] and a_r, all functions of h
            gYz = ops.dft_forward(plan, 1, g_azz2)
            gYr = ops.dft_forward(plan, 1, g_ar)
            ops.mix_dw(plan, Hh, gYz, pk["Wh_zz2"], False, out=dWh_zz2, accumulate=not first)
            ops.mix_dw(plan, Hh, gYr, pk["Wh_r"], False, out=dWh_r, accumulate=not first)
            gH = ops.mix(plan, 1, gYz, pk["Wh_zz2"], Cc, 2 * Cc)
            ops.mix(plan, 1, gYr, pk["Wh_r"], Cc, Cc, out=gH, accumulate=True)
            t1 = ops.pointwise(B, Cc, (H, W), dev, ops.make_epilogue(pw_w=pk["Ph_zz2"], pw_x=g_azz2, pw_transposed=True,
                                                                     add=g_hdir))
            g = ops.dft_inverse(plan, 1, gH, ops.make_epilogue(pw_w=pk["Ph_r"], pw_x=g_ar, pw_transposed=True, add=t1))
            dPh_zz2 = acc_(dPh_zz2, ops.pw_wgrad(g_azz2, h, need_bias=False)[0])
            dPh_r = acc_(dPh_r, ops.pw_wgrad(g_ar, h, need_bias=False)[0])
            first = False
        g_h0 = g if ctx.needs_input_grad[1] else None
        # ---- x side, batched ----
        need_x = ctx.needs_input_grad[0]
        gx = torch.empty_like(xf) if need_x else None
        dWx = {k: [zl(w) for w in pk[k]] for k in ("Wx_zz2", "Wx_r", "Wx_h")}
        dPx, dbx = {}, {}
        groups = (("Wx_zz2", "Px_zz2", gGzz2.reshape(Tn * B, 2 * Cc, H, W), 2 * Cc),
                  ("Wx_r", "Px_r", gGr.reshape(Tn * B, Cc, H, W), Cc),
                  ("Wx_h", "Px_h", gGh.reshape(Tn * B, Cc, H, W), Cc))
        firstc = True
        for j, s in enumerate(range(0, Tn * B, ctx.chunk)):
            e = min(Tn * B, s + ctx.chunk)
            xs, xh = xf[s:e], Xh[j]
            gX = None
            for wk, pkey, G, co in groups:
                gs = G[s:e]
                gY = ops.dft_forward(plan, 1, gs)
                ops.mix_dw(plan, xh, gY, pk[wk], False, out=dWx[wk], accumulate=not firstc)
                dw, db = ops.pw_wgrad(gs, xs, need_bias=True)
                dPx[pkey] = acc_(dPx.get(pkey), dw)
                dbx[pkey] = acc_(dbx.get(pkey), db)
                if need_x:
                    if gX is None:
                        gX = ops.mix(plan, 1, gY, pk[wk], Cc, co)
                    else:
                        ops.mix(plan, 1, gY, pk[wk], Cc, co, out=gX, accumulate=True)
            if need_x:
                n = e - s
                t1 = ops.pointwise(n, Cc, (H, W), dev, ops.make_epilogue(pw_w=pk["Px_zz2"], pw_x=groups[0][2][s:e],
                                                                         pw_transposed=True))
                t2 = ops.pointwise(n, Cc, (H, W), dev, ops.make_epilogue(pw_w=pk["Px_h"], pw_x=groups[2][2][s:e],
                                                                         pw_transposed=True, add=t1))
                ops.dft_inverse(plan, 1, gX, ops.make_epilogue(pw_w=pk["Px_r"], pw_x=groups[1][2][s:e], pw_transposed=True,
                                                               add=t2), out=gx[s:e])
            firstc = False
        # ---- unpack into the reference's parameters ----
        C = Cc
        sp = {1: (dWx["Wx_zz2"], 0), 7: (dWx["Wx_zz2"], 1), 3: (dWx["Wx_r"], None), 5: (dWx["Wx_h"], None),
              2: (dWh_zz2, 0), 8: (dWh_zz2, 1), 4: (dWh_r, None), 6: (dW6, None)}
        pw = {1: (dPx["Px_zz2"], 0), 7: (dPx["Px_zz2"], 1), 3: (dPx["Px_r"], None), 5: (dPx["Px_h"], None),
              2: (dPh_zz2, 0), 8: (dPh_zz2, 1), 4: (dPh_r, None), 6: (dP6, None)}
        db_zz2, db_r, db_h = dbx["Px_zz2"], dbx["Px_r"], dbx["Px_h"]
        cbg = {1: db_zz2[:C], 2: db_zz2[:C], 7: db_zz2[C:], 8: db_zz2[C:], 3: db_r, 4: db_r, 5: db_h, 6: db_h}
        grads = []
        for k in range(1, 9):
            gl, half = sp[k]
            for j in (0, 1):
                w = gl[j] if half is None else gl[j][:, half * C:(half + 1) * C]
                grads.append(w.reshape(ctx.param_shapes[4 * (k - 1) + j]))
            m, half = pw[k]
            m = m if half is None else m[half * C:(half + 1) * C]
            grads.append(m.reshape(ctx.param_shapes[4 * (k - 1) + 2]))
            grads.append(cbg[k].reshape(ctx.param_shapes[4 * (k - 1) + 3]))
        for v in (db_zz2[:C], db_r, db_h, db_zz2[C:]):            # b1, b2, b3, b4 (rno.py:255-258)
            grads.append(v.sum().reshape(()))
        gx_out = gx.reshape(Tn, B, Cc, H, W) if need_x else None
        return (gx_out, g_h0, None, None) + tuple(grads)


def _rno_plan(geom: SpecGeom, device, batch: int, channels: int):
    """The plan of the RNO layer: mode-major spectra (the per-mode [batch x channel] slabs of the tensor-core mixing are
    then contiguous) when every call of the layer is eligible for it, else the default layout."""
    g1 = geom.with_layout(1)
    try:
        p1 = get_plan(g1, device)
        if p1.layout_supported(batch, channels):
            return p1, g1
    except (RuntimeError, NotImplementedError):
        pass
    g0 = geom.with_layout(0)
    return get_plan(g0, device), g0


def _rno_pack(params, C):
    """Gate-grouped operands of the regrouped cell (concatenated along the OUTPUT channel): the reference's parameters are
    only read, the packs are rebuilt from them at every call (a few MB)."""
    P_ = [p.detach() for p in params]
    fw = lambda k, j: P_[4 * (k - 1) + j]
    cw = lambda k: P_[4 * (k - 1) + 2].reshape(C, C).float()
    cb = lambda k: P_[4 * (k - 1) + 3].float()
    b1, b2, b3, b4 = (P_[32 + i].float() for i in range(4))
    cat = torch.cat
    return {
        "Wx_zz2": [cat((fw(1, j), fw(7, j)), dim=1).contiguous() for j in (0, 1)],
        "Wx_r": [_contig(fw(3, j)) for j in (0, 1)], "Wx_h": [_contig(fw(5, j)) for j in (0, 1)],
        "Wh_zz2": [cat((fw(2, j), fw(8, j)), dim=1).contiguous() for j in (0, 1)],
        "Wh_r": [_contig(fw(4, j)) for j in (0, 1)], "W6": [_contig(fw(6, j)) for j in (0, 1)],
        "Px_zz2": cat((cw(1), cw(7)), dim=0).contiguous(), "Px_r": _contig(cw(3)), "Px_h": _contig(cw(5)),
        "Ph_zz2": cat((cw(2), cw(8)), dim=0).contiguous(), "Ph_r": _contig(cw(4)), "P6": _contig(cw(6)),
        "bias_zz2": cat((cb(1) + cb(2) + b1, cb(7) + cb(8) + b4)).contiguous(),
        "bias_r": (cb(3) + cb(4) + b2).contiguous(), "bias_h": (cb(5) + cb(6) + b3).contiguous(),
    }


def rno_layer_supported(x, C, H, W) -> bool:
    return x.is_cuda and H == W and (C * H * W) % 4 == 0


def rno_layer(x_tm, h0, geom: SpecGeom, return_sequences, params):
    return RnoLayerFn.apply(x_tm, h0, geom, bool(return_sequences), *params)
