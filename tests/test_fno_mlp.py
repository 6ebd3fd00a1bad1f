"""Channel-MLP FNO blocks (FNOBlocks(use_mlp=True), b2no_channel_mlp_fwd / b2no_channel_mlp_bwd, functional.ChannelMlpFn and
its composed fallback, convert_).

CPU: FNO1d / FNO2d / FNO3d with channel-MLP blocks (FNOBlocks(use_mlp=True) as fno_blocks) through emulated ops against a
float64 restatement of fno_block.py:123-170 (output and every gradient), on the kernel route and on the composed route;
state_dict keys and parameter order; the unsupported combinations; convert_ re-using the MLP and gating modules.  GPU: the ops against float64 autograd, declined shapes, the
launch counter, FNO2d at the cfg2 shape and a captured training step."""
import contextlib
import os
import sys

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ops_emulator as emu  # noqa: E402
from oracle import ref_loader  # noqa: E402
from oracle import restated as rs  # noqa: E402

RD, CD = torch.float64, torch.complex128


def rel(a, b):
    cv = lambda t: t.detach().cpu().to(CD if t.is_complex() else RD)
    a, b = cv(a), cv(b)
    den = torch.linalg.vector_norm(b).item()
    return torch.linalg.vector_norm(a - b).item() / (den if den > 0 else 1.0)


def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


# ------------------------------------------------------------------------------------------------------------------------
# float64 statement of the channel MLP (include/b2no.h) and of the FNO with use_mlp
# ------------------------------------------------------------------------------------------------------------------------
def channel_mlp_ref(u, x, w1, b1, w2, b2, g, act):
    """act(gelu(W2 gelu(W1 u + b1) + b2) + g x) and its pre-activation; w1 (H, C), w2 (C, H), g (C)."""
    nd = u.dim() - 2
    col = lambda t: t.reshape((1, -1) + (1,) * nd)
    h = F.gelu(torch.einsum("jc,bc...->bj...", w1, u) + col(b1))
    s = F.gelu(torch.einsum("cj,bj...->bc...", w2, h) + col(b2)) + col(g) * x
    return (s if act is None else emu._act(s, act)), s, h


def fno_mlp_forward(sd, x, n_modes, n_layers=4, fft_norm="forward"):
    """oracle/restated.py::fno_forward with the channel MLP of fno_block.py:123-170 (use_mlp, mlp_skip='soft-gating'):
    u = gelu(SpectralConv_l(x) + bias_l + skip_l x);  y = gelu(fc1 gelu(fc0 u)) + g_l x;  gelu(y) for l < n_layers - 1."""
    nd = len(n_modes)
    dt = x.dtype
    cdt = CD if dt == RD else torch.complex64
    g = lambda k: sd[k].to(dt) if not sd[k].is_complex() else sd[k]

    def conv1x1(t, w, b=None):
        y = torch.einsum("oi,bi...->bo...", w.reshape(w.shape[0], w.shape[1]), t)
        return y if b is None else y + b.reshape((1, -1) + (1,) * nd)

    x = conv1x1(x, g("lifting.fc.weight"), g("lifting.fc.bias"))
    nw = 2 ** (nd - 1)
    wkeys = sorted([k for k in sd if k.startswith("fno_blocks.convs.weight.")], key=lambda k: int(k.split(".")[3]))
    bias = g("fno_blocks.convs.bias")
    for l in range(n_layers):
        skip = conv1x1(x, g(f"fno_blocks.fno_skips.{l}.weight"))
        corners = [rs._as_complex(sd[wkeys[nw * l + i]]).to(cdt) for i in range(nw)]
        u = F.gelu(rs.neuralop_spectral_conv(x, corners, bias[l].reshape(-1), n_modes, fft_norm) + skip)
        m = f"fno_blocks.mlp.{l}.fcs."
        v = F.gelu(conv1x1(F.gelu(conv1x1(u, g(m + "0.weight"), g(m + "0.bias"))), g(m + "1.weight"), g(m + "1.bias")))
        x = v + g(f"fno_blocks.mlp_skips.{l}.weight") * x
        if l < n_layers - 1:
            x = F.gelu(x)
    x = F.gelu(conv1x1(x, g("projection.fc1.weight"), g("projection.fc1.bias")))
    return conv1x1(x, g("projection.fc2.weight"), g("projection.fc2.bias"))


def _randomise_mlp(m, seed):
    """Non-trivial gating weights (the constructor's are ones)."""
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if ".mlp_skips." in n:
                p.copy_((torch.randn(p.shape, generator=gen) * 0.5 + 1.0).to(p.device))


def _restated_grads(m, x, n_modes, dev="cpu", weight=None):
    leaves = {k: v.detach().to(dev).to(CD if v.is_complex() else RD).requires_grad_(True) for k, v in m.state_dict().items()}
    ref = fno_mlp_forward(leaves, x.detach().to(dev).double(), n_modes, n_layers=m.n_layers)
    loss = ref.square().sum() if weight is None else (ref * weight.to(dev).double()).sum()
    gs = torch.autograd.grad(loss, list(leaves.values()))
    return ref, dict(zip(leaves.keys(), gs))


# ------------------------------------------------------------------------------------------------------------------------
# the emulated ops
# ------------------------------------------------------------------------------------------------------------------------
def _emu_fwd(u, x, w1, b1, w2, b2, g, act=None, want_pre=False):
    d = lambda t: t.detach().to(RD)
    y, s, _ = channel_mlp_ref(d(u), d(x), d(w1), d(b1), d(w2), d(b2), d(g), act)
    return y.float(), (s.float() if (want_pre and act not in (None, "none")) else None)


def _emu_bwd(u, x, pre, gy, w1, b1, w2, b2, g, act=None):
    """Definition of b2no_channel_mlp_bwd: (du, dx, h, d1, d2, dg)."""
    nd = u.dim() - 2
    col = lambda t: t.reshape((1, -1) + (1,) * nd)
    ud, xd, gd = (t.detach().to(RD).requires_grad_(True) for t in (u, x, g))
    w1d, b1d, w2d, b2d = (t.detach().to(RD) for t in (w1, b1, w2, b2))
    with torch.enable_grad():
        y, _, _ = channel_mlp_ref(ud, xd, w1d, b1d, w2d, b2d, gd, act)
        du, dx, dg = torch.autograd.grad(y, [ud, xd, gd], gy.to(RD))
    a1 = torch.einsum("jc,bc...->bj...", w1d, ud.detach()) + col(b1d)
    h = F.gelu(a1)
    a2 = torch.einsum("cj,bj...->bc...", w2d, h) + col(b2d)
    dy = gy.to(RD) * (emu._act_grad(pre.to(RD), act) if pre is not None else 1.0)
    d2 = dy * emu._act_grad(a2, "gelu")
    d1 = torch.einsum("cj,bc...->bj...", w2d, d2) * emu._act_grad(a1, "gelu")
    return tuple(t.float() for t in (du, dx, h, d1, d2, dg))


@contextlib.contextmanager
def _emulated(kernel=True):
    """ops_emulator.installed() plus the channel-MLP ops; kernel=False declines every shape (the composed route)."""
    import pde_policylearning_b200.ops as ops
    names = ("channel_mlp_supported", "channel_mlp_fwd", "channel_mlp_bwd")
    saved = {n: getattr(ops, n) for n in names}
    with emu.installed():
        try:
            ops.channel_mlp_supported = lambda x, c, h: kernel
            ops.channel_mlp_fwd, ops.channel_mlp_bwd = _emu_fwd, _emu_bwd
            yield
        finally:
            for n, f in saved.items():
                setattr(ops, n, f)


# ------------------------------------------------------------------------------------------------------------------------
# CPU: host logic
# ------------------------------------------------------------------------------------------------------------------------
def with_mlp(m, **kw):
    """m (an FNO / FNO1d / FNO2d / FNO3d mirror) with channel-MLP blocks: FNOBlocks(use_mlp=True) of the same configuration as
    its fno_blocks (the mirrored model classes themselves reject use_mlp)."""
    import pde_policylearning_b200 as P
    b = m.fno_blocks
    m.fno_blocks = P.FNOBlocks(b.in_channels, b.out_channels, b.n_modes, n_layers=b.n_layers, use_mlp=True,
                               non_linearity=b.non_linearity, fft_norm=b.fft_norm, **kw)
    return m


def _model(dims, **kw):
    import pde_policylearning_b200 as P
    if dims == 1:
        return (8,), torch.randn(2, 3, 16), with_mlp(P.FNO1d(8, 8, in_channels=3, out_channels=1, lifting_channels=8,
                                                             projection_channels=8), **kw)
    if dims == 2:
        return (6, 6), torch.randn(2, 3, 12, 10), with_mlp(P.FNO2d(6, 6, 8, in_channels=3, out_channels=1,
                                                                   lifting_channels=16, projection_channels=16), **kw)
    return (4, 4, 4), torch.randn(2, 3, 6, 8, 7), with_mlp(P.FNO3d(4, 4, 4, 6, in_channels=3, out_channels=1,
                                                                   lifting_channels=8, projection_channels=8), **kw)


@pytest.mark.parametrize("kernel", [True, False], ids=["kernel", "composed"])
@pytest.mark.parametrize("dims", [1, 2, 3])
def test_fno_with_mlp_emulated(dims, kernel):
    """FNO1d / FNO2d / FNO3d with use_mlp through emulated ops against the float64 restatement: output and every parameter
    and input gradient, on the ChannelMlpFn route and on the composed fallback."""
    torch.manual_seed(3 + dims)
    n_modes, x, m = _model(dims, mlp_expansion=0.75 if dims == 2 else 0.5)
    _randomise_mlp(m, dims)
    x.requires_grad_(True)
    params = [p for _, p in m.named_parameters()]
    with _emulated(kernel):
        out = m(x)
        gs = torch.autograd.grad(out.square().sum(), params + [x])
    leaves = {k: v.detach().to(CD if v.is_complex() else RD).requires_grad_(True) for k, v in m.state_dict().items()}
    xd = x.detach().double().requires_grad_(True)
    ref = fno_mlp_forward(leaves, xd, n_modes)
    rg = torch.autograd.grad(ref.square().sum(), list(leaves.values()) + [xd])
    rgd = dict(zip(list(leaves.keys()) + ["x"], rg))
    assert rel(out, ref) < 1e-6
    names = [n for n, _ in m.named_parameters()] + ["x"]
    assert any(".mlp." in n for n in names) and any(".mlp_skips." in n for n in names)
    for n, g in zip(names, gs):
        assert rel(g, rgd[n]) < 1e-5, (n, rel(g, rgd[n]))


def test_state_dict_and_parameter_order():
    import pde_policylearning_b200 as P
    m = with_mlp(P.FNO2d(6, 6, 8), mlp_expansion=0.5)
    sd = m.state_dict()
    extra = {f"fno_blocks.mlp.{l}.fcs.{i}.{k}" for l in range(4) for i in (0, 1) for k in ("weight", "bias")} | \
        {f"fno_blocks.mlp_skips.{l}.weight" for l in range(4)}
    assert set(sd) == set(P.FNO2d(6, 6, 8).state_dict()) | extra
    assert tuple(sd["fno_blocks.mlp.1.fcs.0.weight"].shape) == (4, 8, 1, 1)
    assert tuple(sd["fno_blocks.mlp.1.fcs.1.weight"].shape) == (8, 4, 1, 1)
    assert tuple(sd["fno_blocks.mlp_skips.2.weight"].shape) == (1, 8, 1, 1)
    assert bool((sd["fno_blocks.mlp_skips.2.weight"] == 1).all())
    # registration order: convs, fno_skips, mlp, mlp_skips (fno_block.py:58-84) -- it sets the FusedAdam offsets
    names = [n for n, _ in m.fno_blocks.named_parameters()]
    first = lambda s: min(i for i, n in enumerate(names) if n.startswith(s))
    last = lambda s: max(i for i, n in enumerate(names) if n.startswith(s))
    assert last("convs.") < first("fno_skips.") and last("fno_skips.") < first("mlp.") and last("mlp.") < first("mlp_skips.")
    assert names[first("mlp."):first("mlp.") + 4] == ["mlp.0.fcs.0.weight", "mlp.0.fcs.0.bias", "mlp.0.fcs.1.weight",
                                                      "mlp.0.fcs.1.bias"]
    with pytest.raises(NotImplementedError):      # the mirrored model classes do not build MLP blocks themselves
        P.FNO2d(6, 6, 8, use_mlp=True)
    b = P.FNOBlocks(8, 8, (4,), n_layers=2, use_mlp=True, mlp_expansion=1.0)
    assert b.mlp[0].n_layers == 2 and b.mlp[0].dropout is None and b.mlp[0].non_linearity is F.gelu
    assert b.mlp_skips[1].bias is None and tuple(b.mlp[0].fcs[0].weight.shape) == (8, 8, 1)


@pytest.mark.parametrize("kw", [dict(norm="group_norm"), dict(norm="instance_norm"), dict(mlp_dropout=0.1),
                                dict(mlp_skip="linear"), dict(mlp_skip="identity"), dict(preactivation=True)],
                         ids=["group_norm", "instance_norm", "dropout", "linear", "identity", "preactivation"])
def test_unsupported_combinations_raise(kw):
    import pde_policylearning_b200 as P
    with pytest.raises(NotImplementedError):
        P.FNOBlocks(8, 8, (6, 6), n_layers=4, use_mlp=True, **kw)


def _as_reference_blocks(blocks):
    """A stand-in of the reference's FNOBlocks: the reference's class name, outside this package."""
    blocks.__class__ = type("FNOBlocks", (type(blocks),), {"__module__": "reference_stand_in", "preactivation": False})
    return blocks


@pytest.mark.parametrize("kind", ["plain", "relu", "dropout", "three_layers", "gating_bias", "norm"])
def test_convert_reuses_mlp_modules(kind):
    """convert_ swaps a reference FNOBlocks with supported MLPs for the native block, re-using the same MLP and gating modules
    (state_dict keys and Parameters unchanged); other MLPs leave the block in torch."""
    import pde_policylearning_b200 as P
    nn = torch.nn
    m = with_mlp(P.FNO2d(4, 4, 8, n_layers=2))
    blocks = m.fno_blocks
    if kind == "relu":
        blocks.mlp[1].non_linearity = F.relu
    elif kind == "dropout":
        blocks.mlp[0].dropout = nn.ModuleList([nn.Dropout(0.1) for _ in range(2)])
    elif kind == "three_layers":
        blocks.mlp[0] = P.MLP(8, hidden_channels=4, n_layers=3)
    elif kind == "gating_bias":
        blocks.mlp_skips[0] = P.SoftGating(8, 8, bias=True)
    elif kind == "norm":
        blocks.norm = nn.ModuleList([nn.GroupNorm(1, 8) for _ in range(2)])
    mlp, skips = blocks.mlp, blocks.mlp_skips
    _as_reference_blocks(blocks)
    keys, before = list(m.state_dict().keys()), dict(m.named_parameters())
    c = P.convert_(m)
    assert list(c.state_dict().keys()) == keys
    assert all(p is before[k] for k, p in c.named_parameters())
    native = type(c.fno_blocks).__module__.startswith("pde_policylearning_b200")
    assert native == (kind == "plain")
    if native:
        assert c.fno_blocks.mlp is mlp and c.fno_blocks.mlp_skips is skips
        x = torch.randn(2, 3, 8, 8)
        sd = {k: v.detach().to(CD if v.is_complex() else RD) for k, v in c.state_dict().items()}
        with _emulated(), torch.no_grad():
            assert rel(c(x), fno_mlp_forward(sd, x.double(), (4, 4), n_layers=2)) < 1e-6


@pytest.mark.skipif(not ref_loader.available(), reason="B2NO_REFERENCE_ROOT does not name a checkout of the reference")
def test_reference_fno2d_with_mlp():
    """The unmodified reference FNO2d(use_mlp=True) against the restatement (its MLP keeps the F.gelu default, mlp.py:49), and
    convert_ re-using its MLP and gating modules; with the emulated ops the converted model reproduces the reference."""
    import pde_policylearning_b200 as P
    ref = ref_loader.load()
    torch.manual_seed(11)
    r = ref.FNO2d(6, 6, 8, in_channels=3, out_channels=1, lifting_channels=16, projection_channels=16, use_mlp=True)
    _randomise_mlp(r, 5)
    x = torch.randn(2, 3, 12, 12)
    with torch.no_grad():
        y_ref = r(x)
    sd = {k: v.detach().to(CD if v.is_complex() else RD) for k, v in r.state_dict().items()}
    assert rel(y_ref, fno_mlp_forward(sd, x.double(), (6, 6))) < 1e-5
    mlp = r.fno_blocks.mlp
    c = P.convert_(r)
    assert type(c.fno_blocks).__module__.startswith("pde_policylearning_b200") and c.fno_blocks.mlp is mlp
    with _emulated(), torch.no_grad():
        assert rel(c(x), y_ref) < 1e-5


# ------------------------------------------------------------------------------------------------------------------------
# GPU: the ops
# ------------------------------------------------------------------------------------------------------------------------
def _op_grads(u, x, w1, b1, w2, b2, g, act, gy):
    leaves = [t.detach().double().requires_grad_(True) for t in (u, x, w1, b1, w2, b2, g)]
    y, s, _ = channel_mlp_ref(*leaves, act)
    return y, s, torch.autograd.grad(y, leaves, gy.double())


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32", 2e-2)])
@pytest.mark.parametrize("act", ["gelu", None], ids=["act", "last"])
@pytest.mark.parametrize("shape", [(1, (128,)), (3, (32, 48)), (64, (64, 64))], ids=["B1-P128", "B3-P1536", "B64-P4096"])
@pytest.mark.parametrize("C,H", [(8, 4), (8, 8), (32, 16), (32, 32), (34, 17), (34, 34), (64, 32), (64, 64)])
def test_channel_mlp_op(C, H, shape, act, precision, tol):
    """ChannelMlpFn (both kernels, the weight gradients from pw_wgrad) against float64 autograd: y and the gradients of u, x,
    W1, b1, W2, b2 and g."""
    import pde_policylearning_b200.functional as Fn
    from pde_policylearning_b200 import ops
    dev = _dev()
    B, grid = shape
    gen = torch.Generator().manual_seed(C * 100 + H + B)
    r = lambda *s, sc=1.0: (torch.randn(*s, generator=gen) * sc).to(dev)
    u, x = r(B, C, *grid), r(B, C, *grid)
    w1, b1 = r(H, C, *(1,) * len(grid), sc=C ** -0.5), r(H, sc=0.3)
    w2, b2 = r(C, H, *(1,) * len(grid), sc=H ** -0.5), r(C, sc=0.3)
    g = r(1, C, *(1,) * len(grid), sc=0.5) + 1.0
    gy = r(B, C, *grid)
    assert ops.channel_mlp_supported(u, C, H)
    y_ref, _, rg = _op_grads(u, x, w1.reshape(H, C), b1, w2.reshape(C, H), b2, g.reshape(-1), act, gy)
    leaves = [t.clone().requires_grad_(True) for t in (u, x, w1, b1, w2, b2, g)]
    n0 = ops.tensor_core_launches()
    try:
        ops.set_precision(precision)
        y = Fn.channel_mlp(*leaves, act)
        gs = torch.autograd.grad(y, leaves, gy)
        torch.cuda.synchronize()
    finally:
        ops.set_precision("fp32")
    assert ops.tensor_core_launches() - n0 == 4          # forward, backward and the two weight-gradient kernels
    assert rel(y, y_ref) < tol, rel(y, y_ref)
    for name, a, b in zip(("u", "x", "w1", "b1", "w2", "b2", "g"), gs, rg):
        # dW1 / dW2 are fp32 sums over B * P pixels of per-pixel products (b2no_pw_wgrad): at 262144 pixels their rounding
        # alone reaches 1.0-1.1e-5 against float64
        t = 2 * tol if (name in ("w1", "w2") and precision == "fp32") else tol
        assert rel(a.reshape(b.shape), b) < t, (name, rel(a.reshape(b.shape), b))


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,grid", [(8, 4, (10, 10)), (16, 80, (16, 16)), (72, 36, (16, 8))],
                         ids=["pixels%128", "H>64", "C>64"])
def test_channel_mlp_declined_shapes_compose(C, H, grid):
    """Shapes without the kernels take the composed fallback (native pointwise convs); results against float64 autograd."""
    import pde_policylearning_b200.functional as Fn
    from pde_policylearning_b200 import ops
    dev = _dev()
    gen = torch.Generator().manual_seed(C + H)
    r = lambda *s, sc=1.0: (torch.randn(*s, generator=gen) * sc).to(dev)
    u, x, gy = r(2, C, *grid), r(2, C, *grid), r(2, C, *grid)
    w1, b1, w2, b2 = r(H, C, 1, 1, sc=C ** -0.5), r(H, sc=0.3), r(C, H, 1, 1, sc=H ** -0.5), r(C, sc=0.3)
    g = r(1, C, 1, 1, sc=0.5) + 1.0
    assert not ops.channel_mlp_supported(u, C, H)
    assert ops.channel_mlp_supported(u, 8, 8) == (grid[0] * grid[1] % 128 == 0)
    y_ref, _, rg = _op_grads(u, x, w1.reshape(H, C), b1, w2.reshape(C, H), b2, g.reshape(-1), "gelu", gy)
    leaves = [t.clone().requires_grad_(True) for t in (u, x, w1, b1, w2, b2, g)]
    y = Fn.channel_mlp(*leaves, "gelu")
    gs = torch.autograd.grad(y, leaves, gy)
    assert rel(y, y_ref) < 1e-5
    for name, a, b in zip(("u", "x", "w1", "b1", "w2", "b2", "g"), gs, rg):
        assert rel(a.reshape(b.shape), b) < 1e-5, (name, rel(a.reshape(b.shape), b))


# ------------------------------------------------------------------------------------------------------------------------
# GPU: models
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fno2d_cfg2_with_mlp():
    """FNO2d(12, 12, 32) with channel-MLP blocks at the cfg2 shape (batch 64, 128 x 128) against the float64 restatement (run on the
    GPU): output and every gradient, within 5e-5 or within 4x what the restatement itself reaches in float32 (the last layer's
    spectral-weight gradient is a sum with cancellation over 64 x 16384 pixels)."""
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops
    dev = _dev()
    torch.manual_seed(21)
    m = with_mlp(P.FNO2d(12, 12, 32, in_channels=3, out_channels=1))
    _randomise_mlp(m, 9)
    m = m.to(dev)
    x = torch.randn(64, 3, 128, 128, device=dev)
    w = torch.randn(64, 1, 128, 128, device=dev)
    params = [p for _, p in m.named_parameters()]
    n0 = ops.tensor_core_launches()
    out = m(x)
    gs = torch.autograd.grad((out * w).sum(), params)
    assert ops.tensor_core_launches() > n0
    ref, rg = _restated_grads(m, x, (12, 12), dev=dev, weight=w)
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    ref32 = fno_mlp_forward(leaves, x, (12, 12))
    rg32 = dict(zip(leaves.keys(), torch.autograd.grad((ref32 * w).sum(), list(leaves.values()))))
    assert rel(out, ref) < 5e-5
    for (n, _), g in zip(m.named_parameters(), gs):
        bound = max(5e-5, 4.0 * rel(rg32[n], rg[n]))
        print(n, f"{rel(g, rg[n]):.2e}", f"fp32 restatement {rel(rg32[n], rg[n]):.2e}")
        assert rel(g, rg[n]) < bound, (n, rel(g, rg[n]), rel(rg32[n], rg[n]))


@pytest.mark.gpu
def test_graphed_train_step_with_mlp_matches_eager():
    """GraphedTrainStep of an FNO2d with use_mlp follows the same trajectory as the eager step."""
    import pde_policylearning_b200 as P
    dev = _dev()

    def build():
        torch.manual_seed(31)
        m = with_mlp(P.FNO2d(6, 6, 16, in_channels=3, out_channels=1))
        _randomise_mlp(m, 4)
        m = m.to(dev)
        return m, P.FusedAdam(m.parameters(), lr=1e-3, weight_decay=1e-4)

    torch.manual_seed(32)
    xs = [torch.randn(4, 3, 32, 32, device=dev) for _ in range(3)]
    ts = [torch.randn(4, 1, 32, 32, device=dev) for _ in range(3)]
    loss_fn = lambda o, t: P.rel_l2_loss(o, t, size_average=False)
    m1, o1 = build()
    eager = []
    for x, t in zip(xs, ts):
        o1.zero_grad()
        loss = loss_fn(m1(x), t)
        loss.backward()
        o1.step()
        eager.append(loss.item())
    m2, o2 = build()
    step = P.GraphedTrainStep(m2, loss_fn, o2, (xs[0],), ts[0])
    graphed = [step((x,), t).item() for x, t in zip(xs, ts)]
    for a, b in zip(eager, graphed):
        assert abs(a - b) < 1e-5 * abs(a), (eager, graphed)
    assert rel(o2.flat_param, o1.flat_param) < 1e-5
