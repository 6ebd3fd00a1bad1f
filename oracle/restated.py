"""TEST INFRASTRUCTURE ONLY -- CPU restatement ("port") of the reference's model-level algorithm.

Functional PyTorch (torch.fft + einsum, autograd) re-expressions of the reference modules on the
hot path, driven by a ``state_dict`` with the reference's own key names.  They follow the reference's
*algorithm* (full rfftn, slice corners, einsum, scatter into zeros, irfftn), i.e. what the reference's CPU
path does -- this is what ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs time on the GPU
machine's host cores (``kind: "port"`` where no checkout of the reference is named) and what the model-level
parity tests compare against at sizes too large for committed fixtures.

Pinned against the reference itself in tests/test_oracle_vs_reference.py (runs where B2NO_REFERENCE_ROOT
names a checkout of it) and against tests/golden/*.pt (generated from the reference by tests/golden/make_golden.py).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference legs may import this.
"""
from __future__ import annotations

import itertools
import math
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F


# ---------------------------------------------------------------------------------------------
# a1  neuralop/models/spectral_convolution.py:303-347
# ---------------------------------------------------------------------------------------------
def neuralop_spectral_conv(x, corners: Sequence[torch.Tensor], bias, n_modes, fft_norm="forward",
                           out_grid=None):
    """corners in itertools.product order (spectral_convolution.py:330-337); bias (Co,) or None."""
    order = len(n_modes)
    half = [m // 2 for m in n_modes]
    B, C, *grid = x.shape
    Co = corners[0].shape[1]
    cdt = torch.complex128 if x.dtype == torch.float64 else torch.complex64
    fft_size = list(grid)
    fft_size[-1] = fft_size[-1] // 2 + 1
    xf = torch.fft.rfftn(x, norm=fft_norm, dim=list(range(-order, 0)))
    out = torch.zeros([B, Co, *fft_size], dtype=cdt, device=x.device)
    mode_indexing = [((None, m), (-m, None)) for m in half[:-1]] + [((None, half[-1]),)]
    for i, bounds in enumerate(itertools.product(*mode_indexing)):
        idx = (slice(None), slice(None)) + tuple(slice(*b) for b in bounds)
        out[idx] = torch.einsum("bi...,io...->bo...", xf[idx], corners[i].to(cdt))
    s = tuple(grid) if out_grid is None else tuple(out_grid)
    y = torch.fft.irfftn(out, s=s, norm=fft_norm)
    if bias is not None:
        y = y + bias.reshape((1, -1) + (1,) * order)
    return y


def _as_complex(t: torch.Tensor) -> torch.Tensor:
    """tltorch ComplexDense may register a real view (...,2) (SURVEY 8a.4); accept both."""
    if t.is_complex():
        return t
    return torch.view_as_complex(t.contiguous())


# ---------------------------------------------------------------------------------------------
# a3  neuralop/models/fno_block.py:123-170, tfno.py:11-38,195-211
# ---------------------------------------------------------------------------------------------
def fno_forward(sd: Dict[str, torch.Tensor], x, n_modes, n_layers=4, fft_norm="forward"):
    """FNO (any n_dim) with the defaults FNO2d/FNO3d force: linear skips, no mlp/norm,
    GELU only when index < n_layers - index (fno_block.py:149, quirk Q1)."""
    nd = len(n_modes)
    dt = x.dtype
    g = lambda k: sd[k].to(dt) if not sd[k].is_complex() else sd[k]

    def conv1x1(t, w, b=None):
        w2 = w.reshape(w.shape[0], w.shape[1])
        y = torch.einsum("oi,bi...->bo...", w2, t)
        if b is not None:
            y = y + b.reshape((1, -1) + (1,) * nd)
        return y

    x = conv1x1(x, g("lifting.fc.weight"), g("lifting.fc.bias"))
    nw = 2 ** (nd - 1)
    wkeys = sorted([k for k in sd if k.startswith("fno_blocks.convs.weight.")],
                   key=lambda k: int(k.split(".")[3]))
    bias = g("fno_blocks.convs.bias")
    for l in range(n_layers):
        skip = conv1x1(x, g(f"fno_blocks.fno_skips.{l}.weight"))
        cdt = torch.complex128 if dt == torch.float64 else torch.complex64
        corners = [_as_complex(sd[wkeys[nw * l + i]]).to(cdt) for i in range(nw)]
        y = neuralop_spectral_conv(x, corners, bias[l].reshape(-1), n_modes, fft_norm)
        x = y + skip
        if l < n_layers - l:
            x = F.gelu(x)
    x = conv1x1(x, g("projection.fc1.weight"), g("projection.fc1.bias"))
    x = F.gelu(x)
    x = conv1x1(x, g("projection.fc2.weight"), g("projection.fc2.bias"))
    return x


def fno2d_observer_forward(sd, p_plane, modes, n_layers=4):
    """libs/models/fno_models.py:41-57: concat (p, gridx, gridy) with inclusive linspace, NCHW."""
    b, sx, sy = p_plane.shape[:3]
    dt = p_plane.dtype
    gx = torch.tensor(np.linspace(0, 1, sx), dtype=torch.float).reshape(1, sx, 1, 1).repeat([b, 1, sy, 1])
    gy = torch.tensor(np.linspace(0, 1, sy), dtype=torch.float).reshape(1, 1, sy, 1).repeat([b, sx, 1, 1])
    x = torch.cat((p_plane, gx.to(dt), gy.to(dt)), dim=-1).permute(0, 3, 1, 2)
    sub = {k[len("fno2d."):]: v for k, v in sd.items() if k.startswith("fno2d.")}
    return fno_forward(sub, x, (modes, modes), n_layers)


def lp_rel(x, y, size_average=True):
    """libs/utilities3.py:323-334 / libs/pino_utils/losses.py:182-194 (p=2)."""
    n = x.shape[0]
    d = torch.norm(x.reshape(n, -1) - y.reshape(n, -1), 2, 1)
    yn = torch.norm(y.reshape(n, -1), 2, 1)
    r = d / yn
    return r.mean() if size_average else r.sum()


# ---------------------------------------------------------------------------------------------
# a4/a5  neuralop/models/rno.py
# ---------------------------------------------------------------------------------------------
def rno_spectral_conv(x, w0, w1, m1, m2):
    """rno.py:60-77. w*: real pairs (Ci,Co,m1,m2,2)."""
    n = x.shape[-1]
    cdt = torch.complex128 if x.dtype == torch.float64 else torch.complex64
    xf = torch.fft.rfft2(x, s=(n, n), norm="ortho")
    Co = w0.shape[1]
    out = torch.zeros(x.shape[0], Co, n, n // 2 + 1, dtype=cdt, device=x.device)
    c0 = torch.view_as_complex(w0.to(x.dtype).contiguous())
    c1 = torch.view_as_complex(w1.to(x.dtype).contiguous())
    out[:, :, :m1, :m2] = torch.einsum("bixy,ioxy->boxy", xf[:, :, :m1, :m2], c0)
    out[:, :, -m1:, :m2] = torch.einsum("bixy,ioxy->boxy", xf[:, :, -m1:, :m2], c1)
    return torch.fft.irfft2(out, s=(n, n), norm="ortho")


def _fourier_layer(sd, pre, x, m1, m2):
    """rno.py:224-228  spec_conv(x) + Conv1d(k=1)(x)."""
    dt = x.dtype
    y = rno_spectral_conv(x, sd[pre + "spec_conv.fourier_weight.0"], sd[pre + "spec_conv.fourier_weight.1"], m1, m2)
    w = sd[pre + "norm_conv1d.weight"].to(dt)[:, :, 0]
    b = sd[pre + "norm_conv1d.bias"].to(dt)
    return y + torch.einsum("oi,bixy->boxy", w, x) + b.reshape(1, -1, 1, 1)


def rno_cell(sd, pre, x, h, m1, m2):
    """rno.py:254-260."""
    dt = x.dtype
    f = lambda k, t: _fourier_layer(sd, f"{pre}f{k}.", t, m1, m2)
    b = lambda k: sd[f"{pre}b{k}"].to(dt)
    z = torch.sigmoid(f(1, x) + f(2, h) + b(1))
    z2 = torch.sigmoid(f(7, x) + f(8, h) + b(4))
    r = torch.sigmoid(f(3, x) + f(4, h) + b(2))
    hh = F.selu(f(5, x) + f(6, r * h) + b(3))
    return (1.0 - z) * h + z2 * hh


def rno2d_forward(sd, x, modes1, modes2, width, recurrent_index=0, layer_num=1, dropout_eval=True):
    """rno.py:320-379 without padding; dropout treated as eval (Q4)."""
    dt = x.dtype
    B, T = x.shape[:2]

    def one_step(xs, states):
        t = xs @ sd["input_projection_layer.weight"].to(dt).t() + sd["input_projection_layer.bias"].to(dt)
        t = t.permute(0, 1, 4, 2, 3)
        finals = []
        for i in range(layer_num):
            h = states[i]
            if h is None:
                h = torch.zeros(t.shape[0], width, t.shape[3], t.shape[4], dtype=dt, device=t.device) + sd[f"layers.{i}.bias_h"].to(dt)
            outs = []
            for s in range(t.shape[1]):
                h = rno_cell(sd, f"layers.{i}.cell.", t[:, s], h, modes1, modes2)
                outs.append(h)
            if i < layer_num - 1:
                t = t + torch.stack(outs, dim=1)
                finals.append(t[:, -1])
            else:
                finals.append(h)
        h = finals[-1].permute(0, 2, 3, 1)
        # SpectralRegressor rno.py:180-212 (2x SpectralConvWithFC + MLP), modes = modes2 (Q4)
        for j in range(2):
            pre = f"regressor.spectral_conv.{j}."
            res = h @ sd[pre + "linear.weight"].to(dt).t() + sd[pre + "linear.bias"].to(dt)
            c = rno_spectral_conv(h.permute(0, 3, 1, 2), sd[pre + "spec_conv.fourier_weight.0"],
                                  sd[pre + "spec_conv.fourier_weight.1"], modes2, modes2).permute(0, 2, 3, 1)
            h = F.relu(c + res)
        h = F.relu(h @ sd["regressor.regressor.0.weight"].to(dt).t() + sd["regressor.regressor.0.bias"].to(dt))
        pred = h @ sd["regressor.regressor.2.weight"].to(dt).t() + sd["regressor.regressor.2.bias"].to(dt)
        return pred, finals

    states = [None] * layer_num
    outs = []
    for _ in range(T):
        pred, states = one_step(x, states)
        outs.append(pred)
        x = pred.reshape(pred.shape[0], 1, pred.shape[1], pred.shape[2], pred.shape[3])
    return torch.stack(outs, dim=1)[:, recurrent_index]


# ---------------------------------------------------------------------------------------------
# a6/a7  libs/models/pino_models/{basics,pinobserver}.py
# ---------------------------------------------------------------------------------------------
def pino_spectral_conv3d(x, w1, w2, w3, w4, m1, m2, m3):
    """basics.py:114-143 incl. the z_dim zero-extension."""
    cdt = torch.complex128 if x.dtype == torch.float64 else torch.complex64
    B = x.shape[0]
    Co = w1.shape[1]
    xf = torch.fft.rfftn(x, dim=[2, 3, 4])
    zd = min(xf.shape[4], m3)
    out = torch.zeros(B, Co, xf.shape[2], xf.shape[3], m3, dtype=cdt, device=x.device)

    def corner(sl1, sl2, w):
        c = torch.zeros(B, x.shape[1], m1, m2, m3, dtype=cdt, device=x.device)
        c[..., :zd] = xf[:, :, sl1, sl2, :zd]
        return torch.einsum("bixyz,ioxyz->boxyz", c, w.to(cdt))

    lo1, hi1, lo2, hi2 = slice(None, m1), slice(-m1, None), slice(None, m2), slice(-m2, None)
    out[:, :, lo1, lo2] = corner(lo1, lo2, w1)
    out[:, :, hi1, lo2] = corner(hi1, lo2, w2)
    out[:, :, lo1, hi2] = corner(lo1, hi2, w3)
    out[:, :, hi1, hi2] = corner(hi1, hi2, w4)
    return torch.fft.irfftn(out, s=(x.size(2), x.size(3), x.size(4)), dim=[2, 3, 4])


def pino_spectral_conv2d(x, w1, w2, m1, m2):
    """basics.py:79-96: rfftn (norm 'backward'), weights1 on rows [0, m1), weights2 on rows [-m1, N), columns [0, m2),
    modes un-halved; the high corner is assigned last (overwrites on overlap)."""
    cdt = torch.complex128 if x.dtype == torch.float64 else torch.complex64
    B, Co = x.shape[0], w1.shape[1]
    xf = torch.fft.rfftn(x, dim=[2, 3])
    out = torch.zeros(B, Co, x.size(-2), x.size(-1) // 2 + 1, dtype=cdt, device=x.device)
    out[:, :, :m1, :m2] = torch.einsum("bixy,ioxy->boxy", xf[:, :, :m1, :m2], w1.to(cdt))
    out[:, :, -m1:, :m2] = torch.einsum("bixy,ioxy->boxy", xf[:, :, -m1:, :m2], w2.to(cdt))
    return torch.fft.irfftn(out, s=(x.size(-2), x.size(-1)), dim=[2, 3])


def pino_fno2d_forward(sd, x, modes1, modes2, layers, pad_ratio=(0.0, 0.0), act=F.gelu):
    """libs/models/pino_models/fourier2d.py:54-87: fc0, [SpectralConv2d + Conv1d(k=1)] stack with the activation after
    every layer but the last, optional zero padding of both grid dims (:61-65,:71,:80), three-layer tail fc1-act-fc2-act-fc3."""
    dt = x.dtype
    if isinstance(pad_ratio, float):
        pad_ratio = [pad_ratio, pad_ratio]
    s1, s2 = x.shape[1], x.shape[2]
    padded = max(pad_ratio) > 0
    np1 = [round(r * s1) for r in pad_ratio] if padded else [0, 0]
    np2 = [round(r * s2) for r in pad_ratio] if padded else [0, 0]
    L = len(layers) - 1
    t = x @ sd["fc0.weight"].to(dt).t() + sd["fc0.bias"].to(dt)
    t = t.permute(0, 3, 1, 2)
    if max(np1) > 0 or max(np2) > 0:
        t = F.pad(t, (np2[0], np2[1], np1[0], np1[1]), "constant", 0.0)
    for i in range(L):
        x1 = pino_spectral_conv2d(t, sd[f"sp_convs.{i}.weights1"], sd[f"sp_convs.{i}.weights2"], modes1[i], modes2[i])
        w = sd[f"ws.{i}.weight"].to(dt)[:, :, 0]
        x2 = torch.einsum("oi,bixy->boxy", w, t) + sd[f"ws.{i}.bias"].to(dt).reshape(1, -1, 1, 1)
        t = x1 + x2
        if i != L - 1:
            t = act(t)
    if max(np1) > 0 or max(np2) > 0:
        t = t[..., np1[0]:t.shape[-2] - np1[1], np2[0]:t.shape[-1] - np2[1]]
    t = t.permute(0, 2, 3, 1)
    t = act(t @ sd["fc1.weight"].to(dt).t() + sd["fc1.bias"].to(dt))
    t = act(t @ sd["fc2.weight"].to(dt).t() + sd["fc2.bias"].to(dt))
    return t @ sd["fc3.weight"].to(dt).t() + sd["fc3.bias"].to(dt)


def _mult_net(sd, pre, t, re):
    """pinobserver.py:41-59: input1 @ B^T + re @ A^T + bias (affine)."""
    dt = t.dtype
    if re.dim() < 2:
        re = re.unsqueeze(-1)
    code = re.to(dt) @ sd[pre + "A"].to(dt).t()
    return t @ sd[pre + "B"].to(dt).t() + code[:, None, None, None, :] + sd[pre + "bias"].to(dt)


def pinobserver2d_forward(sd, x, re, modes1, modes2, modes3, layers, pad_ratio=0.0625, act=F.gelu, head="", re_scale=1.0):
    """pinobserver.py:192-233.  head / re_scale: the same trunk as used by PINObserverFullField (:341-368: parameters of
    the Fourier stack and the tail live under `observer_head.`, re / max_re with max_re = 1000 :313,350) and PolicyModel2D
    (:436-463: under `pred_net.`, same re scaling); fc0 and the two MultiplicativeNets stay at the top level."""
    dt = x.dtype
    re = re.float() / re_scale if re_scale != 1.0 else re
    if isinstance(pad_ratio, float):
        pad_ratio = [pad_ratio, pad_ratio]
    size_z = x.shape[-2]
    num_pad = [round(size_z * r) for r in pad_ratio] if max(pad_ratio) > 0 else [0, 0]
    B = x.shape[0]
    L = len(layers) - 1
    t = x @ sd["fc0.weight"].to(dt).t() + sd["fc0.bias"].to(dt)
    t = _mult_net(sd, "multiplicative_net1.", t, re.float())
    t = t.permute(0, 4, 1, 2, 3)
    if max(num_pad) > 0:
        t = F.pad(t, (num_pad[0], num_pad[1]), "constant", 0)
    for i in range(L):
        ws = [sd[f"{head}sp_convs.{i}.weights{j}"] for j in (1, 2, 3, 4)]
        x1 = pino_spectral_conv3d(t, *ws, modes1[i], modes2[i], modes3[i])
        w = sd[f"{head}ws.{i}.weight"].to(dt)[:, :, 0]
        x2 = torch.einsum("oi,bixyz->boxyz", w, t) + sd[f"{head}ws.{i}.bias"].to(dt).reshape(1, -1, 1, 1, 1)
        t = x1 + x2
        if i != L - 1:
            t = act(t)
    if max(num_pad) > 0:
        t = t[..., num_pad[0]:-num_pad[1]]
    t = t.permute(0, 2, 3, 4, 1)
    t = _mult_net(sd, "multiplicative_net2.", t, re.float())
    t = act(t @ sd[f"{head}fc1.weight"].to(dt).t() + sd[f"{head}fc1.bias"].to(dt))
    return t @ sd[f"{head}fc2.weight"].to(dt).t() + sd[f"{head}fc2.bias"].to(dt)


def pinobserver_fullfield_forward(sd, x, re, modes1, modes2, modes3, layers, pad_ratio=0.0625, act=F.gelu):
    """PINObserverFullField.forward, pinobserver.py:341-368: one shared trunk whose tail emits out_dim * plane_num channels,
    returned planes-first (b, p, x, y, t)."""
    out = pinobserver2d_forward(sd, x, re, modes1, modes2, modes3, layers, pad_ratio, act, head="observer_head.", re_scale=1000.0)
    return out.permute(0, 4, 1, 2, 3)


def policy_model2d_forward(sd, x, re, modes1, modes2, modes3, layers, pad_ratio=0.0625, act=F.gelu):
    """PolicyModel2D.forward, pinobserver.py:436-463 (the constructor zero-initialises every parameter, :432-433)."""
    return pinobserver2d_forward(sd, x, re, modes1, modes2, modes3, layers, pad_ratio, act, head="pred_net.", re_scale=1000.0)


# ---------------------------------------------------------------------------------------------
# a8  libs/envs/diff_control_env.py:5-60, libs/pino_utils/losses.py:288-291
# ---------------------------------------------------------------------------------------------
def fdm_ns_vorticity(w, v, t_interval=1.0):
    B, nx, ny, nt = w.shape
    dt_ = w.dtype
    wh = torch.fft.fft2(w, dim=[1, 2])
    kmax = nx // 2
    N = nx
    k1 = torch.cat((torch.arange(0, kmax), torch.arange(-kmax, 0)), 0).to(dt_).to(w.device)
    kx = k1.reshape(N, 1).repeat(1, N).reshape(1, N, N, 1)
    ky = k1.reshape(1, N).repeat(N, 1).reshape(1, N, N, 1)
    lap = kx ** 2 + ky ** 2
    lap[0, 0, 0, 0] = 1.0
    fh = wh / lap
    c = lambda t: torch.fft.irfft2(t[:, :, : kmax + 1], dim=[1, 2])
    ux, uy = c(1j * ky * fh), c(-1j * kx * fh)
    wx, wy, wlap = c(1j * kx * wh), c(1j * ky * wh), c(-lap * wh)
    dt = t_interval / (nt - 1)
    wt = (w[:, :, :, 2:] - w[:, :, :, :-2]) / (2 * dt)
    return wt + (ux * wx + uy * wy - v.reshape(-1, 1, 1, 1) * wlap)[..., 1:-1]


def get_forcing(S, dtype=torch.float32):
    x2 = torch.tensor(np.linspace(0, 2 * np.pi, S, endpoint=False), dtype=torch.float).reshape(1, S).repeat(S, 1)
    return (-4 * torch.cos(4 * x2)).reshape(1, S, S, 1).to(dtype)


def channelflow_pino_loss(out, u0, forcing, v, t_interval=1.0):
    B, nx, ny, nt = out.shape[:4]
    out = out.reshape(B, nx, ny, nt)
    loss_ic = lp_rel(out[:, :, :, 0], u0)
    Du = fdm_ns_vorticity(out, v, t_interval)
    f = forcing.repeat(B, 1, 1, nt - 2)
    return loss_ic, lp_rel(Du, f)
