"""GPU parity: the CUDA path, called through the reference-facing modules (which go through the C ABI in
libb2no.so), against (1) the committed golden vectors made by the unmodified reference, (2) the float64
closed-form oracle on seeded inputs, (3) size-independent properties at BASELINE sizes.
Tolerance: north_star -- relative L2 <= 1e-5 in fp32."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def rel(a, b):
    from oracle.closed_form import rel_l2
    return rel_l2(a, b)


# --------------------------------------------------------------------------------------------
# raw C-ABI stages vs the closed-form oracle (locates a failure to a kernel)
# --------------------------------------------------------------------------------------------
STAGE_CASES = [
    # nin, half, norm, nfft, nout, Ci, Co, B
    ((12,), (5,), "forward", None, None, 3, 4, 2),
    ((16, 12), (4, 3), "forward", None, None, 3, 5, 2),
    ((128, 128), (6, 6), "forward", None, None, 4, 4, 2),
    ((64, 64), (8, 8), "backward", None, None, 3, 3, 3),
    ((32, 32), (12, 12), "ortho", (32, 32), (32, 32), 34, 34, 2),
    ((9, 11), (3, 3), "ortho", None, None, 2, 3, 2),
    ((8, 12), (6, 3), "forward", None, None, 2, 2, 2),          # overlap 2h > N
    ((15, 12), (4, 3), "ortho", (12, 12), (12, 12), 3, 2, 2),   # rno crop
    ((9, 12), (4, 3), "ortho", (12, 12), (12, 12), 3, 2, 2),    # rno zero-pad
    ((16, 12), (4, 3), "forward", None, (8, 6), 3, 4, 2),       # output scaling 0.5
    ((16, 12), (4, 3), "backward", None, (32, 24), 3, 4, 2),    # output scaling 2
    ((8, 8, 9), (3, 2, 4), "backward", None, None, 3, 4, 2),
    ((8, 8, 9), (3, 2, 6), "backward", None, None, 3, 4, 2),    # modes3 > Z/2+1
    ((16, 16, 73), (8, 8, 8), "backward", None, None, 4, 4, 1),
    ((20, 200), (4, 20), "forward", None, None, 2, 2, 2),       # long rows, many modes (chunked)
]


@pytest.mark.parametrize("case", STAGE_CASES, ids=lambda c: "x".join(map(str, c[0])) + f"-h{'x'.join(map(str, c[1]))}-{c[2]}")
def test_stages_vs_closed_form(case):
    from oracle import closed_form as cf
    from pde_policylearning_b200 import ops
    nin, half, norm, nfft, nout, ci, co, B = case
    dev = _dev()
    torch.manual_seed(7)
    g64 = cf.SpecGeom(nin=nin, half=half, norm=norm, nfft=nfft, nout=nout)
    geom = ops.SpecGeom(nin=nin, half=half, norm=norm, nfft=nfft, nout=nout)
    plan = ops.get_plan(geom, dev)
    assert plan.kept == g64.kept()
    sf, si = g64.scales()
    d = len(nin)
    x = torch.randn(B, ci, *nin)
    hshape = tuple(half)
    corners = [torch.randn(ci, co, *hshape, dtype=torch.cfloat) for _ in range(2 ** (d - 1))]
    # forward transform
    xh = ops.dft_forward(plan, 0, x.to(dev).contiguous())
    xh64 = cf.dft_trunc(g64, x, sf)
    assert rel(xh, xh64) < TOL, "dft_forward(which=0)"
    # mixing
    cd = [c.to(dev) for c in corners]
    yh = ops.mix(plan, 0, xh, cd, ci, co)
    W = cf.gather_weight(g64, corners)
    yh64 = torch.einsum("bi...,io...->bo...", xh64, W)
    assert rel(yh, yh64) < TOL, "mix(mode=0)"
    # inverse transform (no epilogue)
    y = ops.dft_inverse(plan, 0, yh, None)
    y64 = cf.idft_trunc(g64, yh64, si)
    assert rel(y, y64) < TOL, "dft_inverse(which=0)"
    # adjoints
    gy = torch.randn(B, co, *g64.nout)
    gyh = ops.dft_forward(plan, 1, gy.to(dev).contiguous())
    gyh64 = cf.dft_trunc(g64, gy, si, use_inv_conj=True)
    assert rel(gyh, gyh64) < TOL, "dft_forward(which=1)"
    gxh = ops.mix(plan, 1, gyh, cd, ci, co)
    gxh64 = torch.einsum("bo...,io...->bi...", gyh64, W.conj())
    assert rel(gxh, gxh64) < TOL, "mix(mode=1)"
    dx = ops.dft_inverse(plan, 1, gxh, None)
    dx64 = cf.idft_trunc(g64, gxh64, sf, use_fwd_conj=True)
    assert rel(dx, dx64) < TOL, "dft_inverse(which=1)"
    overlap = any(2 * half[j] > g64.nfft[j] for j in range(d - 1))
    dws = ops.mix_dw(plan, xh, gyh, cd, needs_zero=overlap)
    dW64 = cf.scatter_weight_grad(g64, torch.einsum("bi...,bo...->io...", xh64.conj(), gyh64),
                                  [tuple(c.shape) for c in corners])
    for a, b in zip(dws, dW64):
        if b.abs().max() > 0:
            assert rel(a, b) < TOL, "mix_dw"
        else:
            assert a.abs().max().item() == 0.0


def test_epilogue_and_pointwise():
    """fused epilogue: bias + 1x1 skip + second operand + add + act + mul + preact."""
    from pde_policylearning_b200 import ops
    dev = _dev()
    torch.manual_seed(3)
    for grid, ci, ci2, co, act in (((16, 12), 5, 3, 7, "gelu"), ((130,), 32, 1, 256, "relu"),
                                   ((6, 5, 9), 34, 2, 1, "selu"), ((128, 128), 32, 4, 32, "sigmoid"),
                                   ((64, 64), 3, 2, 32, "tanh")):
        B = 2
        x = torch.randn(B, ci, *grid, device=dev)
        x2 = torch.randn(B, ci2, *grid, device=dev)
        w = torch.randn(co, ci, device=dev)
        w2 = torch.randn(co, ci2, device=dev)
        b = torch.randn(co, device=dev)
        add = torch.randn(B, co, *grid, device=dev)
        mul = torch.randn(B, co, *grid, device=dev)
        z = torch.empty(B, co, *grid, device=dev)
        y = ops.pointwise(B, co, grid, dev, ops.make_epilogue(bias=b, pw_w=w, pw_x=x, pw2_w=w2, pw2_x=x2, add=add,
                                                              mul=mul, preact=z, act=act))
        z64 = (torch.einsum("oi,bi...->bo...", w.double(), x.double()) + torch.einsum("oi,bi...->bo...", w2.double(), x2.double())
               + b.double().reshape((1, -1) + (1,) * len(grid)) + add.double())
        f = {"gelu": torch.nn.functional.gelu, "relu": torch.relu, "selu": torch.selu, "sigmoid": torch.sigmoid,
             "tanh": torch.tanh}[act]
        assert rel(z, z64) < TOL
        assert rel(y, f(z64) * mul.double()) < TOL
        # transposed weight (dx pass)
        g = torch.randn(B, co, *grid, device=dev)
        dx = ops.pointwise(B, ci, grid, dev, ops.make_epilogue(pw_w=w, pw_x=g, pw_transposed=True))
        assert rel(dx, torch.einsum("oi,bo...->bi...", w.double(), g.double())) < TOL
        # weight gradient
        dw, db = ops.pw_wgrad(g, x, need_bias=True)
        assert rel(dw, torch.einsum("bo...,bi...->oi", g.double(), x.double())) < TOL
        assert rel(db, g.double().sum(dim=[0] + list(range(2, g.dim())))) < TOL
        # activation backward
        gz = ops.act_bwd(g, z, act)
        zz = z.double().requires_grad_(True)
        (f(zz) * g.double()).sum().backward()
        assert rel(gz, zz.grad) < TOL


def test_mlp_head_rel_l2_gate():
    from pde_policylearning_b200 import ops
    import pde_policylearning_b200 as P
    dev = _dev()
    torch.manual_seed(4)
    for ci, hid, grid in ((32, 256, (40, 33)), (64, 128, (5, 6, 7)), (8, 16, (300,))):
        B = 3
        x = torch.randn(B, ci, *grid, device=dev)
        w1, b1 = torch.randn(hid, ci, device=dev) * 0.2, torch.randn(hid, device=dev)
        w2, b2 = torch.randn(hid, device=dev) * 0.2, torch.randn(1, device=dev)
        out = ops.mlp_head_fwd(x, w1, b1, w2, b2, "gelu")
        h = torch.nn.functional.gelu(torch.einsum("ji,bi...->bj...", w1.double(), x.double()) + b1.double().reshape((1, -1) + (1,) * len(grid)))
        ref = torch.einsum("j,bj...->b...", w2.double(), h).unsqueeze(1) + b2.double()
        assert rel(out, ref) < TOL
        b1ps = torch.randn(B, hid, device=dev)
        out = ops.mlp_head_fwd(x, w1, b1ps, w2, b2, "gelu")
        h = torch.nn.functional.gelu(torch.einsum("ji,bi...->bj...", w1.double(), x.double()) + b1ps.double().reshape((B, hid) + (1,) * len(grid)))
        assert rel(out, torch.einsum("j,bj...->b...", w2.double(), h).unsqueeze(1) + b2.double()) < TOL
    # rel-L2 loss + grad
    x = torch.randn(5, 1, 37, 41, device=dev, requires_grad=True)
    y = torch.randn(5, 1, 37, 41, device=dev)
    for avg in (True, False):
        loss = P.rel_l2_loss(x, y, avg)
        xd = x.detach().double().requires_grad_(True)
        r = torch.norm((xd - y.double()).reshape(5, -1), 2, 1) / torch.norm(y.double().reshape(5, -1), 2, 1)
        lref = r.mean() if avg else r.sum()
        assert abs(loss.item() - lref.item()) < 1e-5 * abs(lref.item())
        (g,) = torch.autograd.grad(loss, x)
        (gref,) = torch.autograd.grad(lref, xd)
        assert rel(g, gref) < TOL
    # gate
    z, z2, hh, h = (torch.randn(2, 6, 9, 9, device=dev, requires_grad=True) for _ in range(4))
    out = P.rno_gate(z, z2, hh, h)
    ref = (1 - z) * h + z2 * hh
    assert rel(out, ref) < 1e-6
    go = torch.randn_like(out)
    for a, b in zip(torch.autograd.grad(out, [z, z2, hh, h], go), torch.autograd.grad(ref, [z, z2, hh, h], go)):
        assert rel(a, b) < 1e-6


# --------------------------------------------------------------------------------------------
# modules vs golden vectors from the unmodified reference
# --------------------------------------------------------------------------------------------
A1 = ["2d_forward", "2d_backward", "2d_ortho", "1d_forward", "3d_forward", "2d_overlap", "2d_oddgrid",
      "2d_scale_half", "2d_scale_2", "2d_cfg1_small"]


def _run_conv(mod, c, dev):
    mod = mod.to(dev)
    x = c["x"].to(dev).requires_grad_(True)
    y = mod(x)
    names = [n for n, _ in mod.named_parameters()]
    gs = torch.autograd.grad(y, [x] + [p for _, p in mod.named_parameters()], c["gy"].to(dev))
    assert rel(y, c["y"]) < TOL, "y"
    assert rel(gs[0], c["dx"]) < TOL, "dx"
    for n, g in zip(names, gs[1:]):
        ref = c["grads"][n]
        if ref.abs().max() == 0:
            assert g.abs().max().item() == 0
        else:
            assert rel(g, ref) < TOL, n


@pytest.mark.parametrize("name", A1)
def test_golden_neuralop_conv(golden, name):
    import pde_policylearning_b200 as P
    c = golden("a1_neuralop_conv")[name]
    ci, co = c["params"]["weight.0.tensor"].shape[:2]
    m = P.SpectralConv(ci, co, c["n_modes"], n_layers=1, factorization=None, implementation="factorized",
                       fft_norm=c["fft_norm"], **c["kw"])
    m.load_state_dict(c["params"])
    _run_conv(m, c, _dev())


def test_golden_layer_index(golden):
    import pde_policylearning_b200 as P
    c = golden("a1_neuralop_conv")["2d_layer_index2"]
    m = P.SpectralConv(4, 4, (6, 6), n_layers=3, factorization=None, implementation="factorized", fft_norm="forward")
    m.load_state_dict(c["params"])
    m = m.to(_dev())
    assert rel(m(c["x"].to(_dev()), 2), c["y"]) < TOL
    assert rel(m[2](c["x"].to(_dev())), c["y"]) < TOL


@pytest.mark.parametrize("name", ["square", "cfg3_small", "tall", "short"])
def test_golden_rno_conv(golden, name):
    import pde_policylearning_b200 as P
    c = golden("a4_rno_conv")[name]
    ci, co, m1, m2, _ = c["params"]["fourier_weight.0"].shape
    m = P.RnoSpectralConv2d(ci, co, m1, m2)
    m.load_state_dict(c["params"])
    _run_conv(m, c, _dev())


@pytest.mark.parametrize("name", ["basic", "zpad", "cfg4_small"])
def test_golden_pino_conv(golden, name):
    import pde_policylearning_b200 as P
    c = golden("a6_pino_conv")[name]
    ci, co, m1, m2, m3 = c["params"]["weights1"].shape
    m = P.PinoSpectralConv3d(ci, co, m1, m2, m3)
    m.load_state_dict(c["params"])
    _run_conv(m, c, _dev())


def _run_model(mod, c, dev, loss_fn=None, tol=TOL, gtol=5e-5):
    mod.load_state_dict(c["state_dict"])
    mod = mod.to(dev)
    out = mod(*[t.to(dev) for t in c["inputs"]])
    assert rel(out, c["out"]) < tol, "output"
    loss = out.square().mean() if loss_fn is None else loss_fn(out)
    assert abs(loss.item() - c["loss"].item()) <= 2e-5 * abs(c["loss"].item()), "loss"
    names = [n for n, _ in mod.named_parameters()]
    gs = torch.autograd.grad(loss, [p for _, p in mod.named_parameters()], allow_unused=True)
    worst, where = 0.0, ""
    for n, g in zip(names, gs):
        assert g is not None, f"{n} got no gradient"   # test_tfno.py:61-65: every parameter is reached
        e = rel(g, c["grads"][n])
        if e > worst:
            worst, where = e, n
        assert e < gtol, (n, e)
    # the margin against the tolerance is part of the record (pytest -s)
    print(f"[{type(mod).__name__}] output {rel(out, c['out']):.2e} (tol {tol:.0e}), worst parameter gradient {worst:.2e} at {where} "
          f"(tol {gtol:.0e})")
    return worst


def test_golden_fno2d(golden):
    import pde_policylearning_b200 as P
    c = golden("a3_fno2d")
    dev = _dev()
    m = P.FNO2d(8, 8, 16, in_channels=3, out_channels=1)
    tgt = c["target"].to(dev)
    _run_model(m, c, dev, lambda o: P.rel_l2_loss(o, tgt, size_average=False))


def test_golden_fno3d_and_observer(golden):
    import pde_policylearning_b200 as P
    dev = _dev()
    c = golden("a3_fno3d")
    _run_model(P.FNO3d(4, 4, 4, 6, in_channels=2, out_channels=1), c, dev)
    c = golden("a9_fno2d_observer")
    _run_model(P.FNO2dObserver(6, 6, 8), c, dev)


def test_golden_rno(golden):
    import pde_policylearning_b200 as P
    dev = _dev()
    c = golden("a5_rno_cell")
    _run_model(P.RNO_cell(6, 6, 4, 4, 6), c, dev)
    c = golden("a5_rno2d_L1")
    _run_model(P.RNO2d(4, 4, 6, 0, layer_num=1).eval(), c, dev, gtol=2e-4)
    c = golden("a5_rno2d_L2")
    _run_model(P.RNO2d(4, 4, 6, 1, layer_num=2).eval(), c, dev, gtol=2e-4)


def test_golden_pinobserver(golden):
    import pde_policylearning_b200 as P
    from oracle import restated as rs
    dev = _dev()
    c = golden("a7_pinobserver2d")
    m = P.PINObserver2d(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4, act="gelu",
                        pad_ratio=0.0625)
    u, re = c["u"].to(dev), c["inputs"][1].to(dev)
    forcing = P.get_forcing(8, device=dev)
    assert torch.equal(forcing.cpu(), c["forcing"])

    def loss_fn(o):
        # the product's PINO loss (pino_loss.py: DFT-matrix contractions, no torch.fft) against the reference's fixtures
        data = P.rel_l2_loss(o.reshape(2, 8, 8, 17), u, True)
        lic, lf = P.channelflow_pino_loss(o, u[..., 0], forcing, 1 / re, c["t_interval"])
        return 5.0 * data + lf + lic

    with torch.no_grad():
        ref_out = c["out"].to(dev)
        lic, lf = P.channelflow_pino_loss(ref_out, u[..., 0], forcing, 1 / re, c["t_interval"])
        assert abs(lic.item() - c["loss_ic"].item()) <= 1e-5 * abs(c["loss_ic"].item())
        assert abs(lf.item() - c["loss_f"].item()) <= 1e-5 * abs(c["loss_f"].item())
        assert rel(P.fdm_ns_vorticity(ref_out.reshape(2, 8, 8, 17), 1 / re, c["t_interval"]), c["Du"]) < TOL

    _run_model(m, c, dev, loss_fn, gtol=2e-4)
    # inference path (fused head) gives the same output
    with torch.no_grad():
        out = m(*[t.to(dev) for t in c["inputs"]])
    assert rel(out, c["out"]) < TOL


# --------------------------------------------------------------------------------------------
# BASELINE-size checks: restated torch.fft oracle on the same device + size-independent properties
# --------------------------------------------------------------------------------------------
def test_cfg1_full_size_vs_closed_form():
    """BASELINE config 1: FactorizedSpectralConv(32,32,(16,16)) on (8,32,64,64), fwd+bwd."""
    import pde_policylearning_b200 as P
    from oracle import closed_form as cf
    dev = _dev()
    torch.manual_seed(11)
    m = P.SpectralConv(32, 32, (16, 16), n_layers=1, factorization=None, implementation="factorized", fft_norm="forward")
    x = torch.randn(8, 32, 64, 64)
    gy = torch.randn(8, 32, 64, 64)
    geom = cf.geom_neuralop((64, 64), (16, 16), "forward")
    corners = [w.tensor.detach() for w in m.weight]
    y64, _, _ = cf.spectral_conv_forward(geom, x, corners, m.bias.detach()[0].flatten())
    dx64, dW64, db64 = cf.spectral_conv_backward(geom, x, corners, gy, has_bias=True)
    m = m.to(dev)
    xd = x.to(dev).requires_grad_(True)
    y = m(xd)
    gs = torch.autograd.grad(y, [xd, m.weight[0].tensor, m.weight[1].tensor, m.bias], gy.to(dev))
    assert rel(y, y64) < TOL
    assert rel(gs[0], dx64) < TOL
    assert rel(gs[1], dW64[0]) < TOL and rel(gs[2], dW64[1]) < TOL
    assert rel(gs[3].flatten(), db64) < TOL


def test_cfg2_fno2d_full_size_vs_restated():
    """BASELINE config 2 (batch 8 of the 64): FNO2d(12,12,32) 128x128 fwd+bwd against the restated
    reference algorithm (torch.fft + einsum, float64) on the same inputs."""
    import pde_policylearning_b200 as P
    from oracle import restated as rs
    dev = _dev()
    torch.manual_seed(12)
    m = P.FNO2d(12, 12, 32, in_channels=3, out_channels=1).to(dev)
    x = torch.randn(8, 3, 128, 128, device=dev)
    tgt = torch.randn(8, 1, 128, 128, device=dev)
    out = m(x)
    loss = P.rel_l2_loss(out, tgt, size_average=False)
    names = [n for n, _ in m.named_parameters()]
    gs = torch.autograd.grad(loss, [p for _, p in m.named_parameters()])
    sd = {}
    for k, v in m.state_dict().items():
        v = v.detach()
        sd[k] = (v.to(torch.complex128) if v.is_complex() else v.double()).requires_grad_(True)
    out64 = rs.fno_forward(sd, x.double(), (12, 12))
    loss64 = rs.lp_rel(out64, tgt.double(), size_average=False)
    gs64 = torch.autograd.grad(loss64, [sd[n] for n in names])
    assert rel(out, out64) < TOL
    assert abs(loss.item() - loss64.item()) < 1e-5 * abs(loss64.item())
    for n, a, b in zip(names, gs, gs64):
        assert rel(a, b) < 5e-5, n


def test_properties_full_size():
    """Size-independent properties at BASELINE config 2/3/4 shapes: linearity, the adjoint identity
    <conv(x), g> == <x, conv^T(g)>, translation equivariance and the DC-mode bias gradient."""
    import pde_policylearning_b200 as P
    dev = _dev()
    torch.manual_seed(13)
    cases = [
        (P.SpectralConv(32, 32, (12, 12), bias=False, factorization=None, implementation="factorized",
                        fft_norm="forward"), (16, 32, 128, 128)),
        (P.RnoSpectralConv2d(34, 34, 12, 12), (32, 34, 32, 32)),
        (P.PinoSpectralConv3d(16, 16, 8, 8, 8), (1, 16, 32, 32, 73)),
    ]
    for m, shape in cases:
        m = m.to(dev)
        x1 = torch.randn(*shape, device=dev, requires_grad=True)
        x2 = torch.randn(*shape, device=dev)
        y1 = m(x1)
        y2 = m(x2)
        y12 = m(2.0 * x1.detach() - 3.0 * x2)
        assert rel(y12, 2.0 * y1.detach() - 3.0 * y2) < TOL, "linearity"
        g = torch.randn_like(y1)
        (dx,) = torch.autograd.grad(y1, x1, g)
        lhs = (y1.detach().double() * g.double()).sum().item()
        rhs = (x1.detach().double() * dx.double()).sum().item()
        assert abs(lhs - rhs) < 1e-5 * max(abs(lhs), abs(rhs), 1e-3 * y1.detach().double().norm().item() * g.double().norm().item()), "adjoint"
        # circular shift along the last axis commutes with the convolution
        ys = m(torch.roll(x2, shifts=5, dims=-1))
        assert rel(ys, torch.roll(y2, shifts=5, dims=-1)) < TOL, "translation equivariance"


# --------------------------------------------------------------------------------------------
# tcgen05 tile kernel (tc_pointwise.cu): same C-ABI call, tensor-core path vs CUDA-core path vs float64
# --------------------------------------------------------------------------------------------
TC_CASES = [
    # grid, half, norm, ci, co, B, act
    ((128, 128), (6, 6), "forward", 32, 32, 3, "gelu"),
    ((64, 64), (8, 8), "forward", 32, 32, 2, None),
    ((16, 16), (4, 4), "forward", 16, 16, 2, "gelu"),
    ((32, 64), (5, 7), "backward", 3, 20, 2, "relu"),
    ((128, 128), (6, 6), "ortho", 8, 40, 1, "tanh"),
]


@pytest.mark.parametrize("case", TC_CASES, ids=lambda c: "x".join(map(str, c[0])) + f"-c{c[3]}-{c[4]}")
def test_tensor_core_tile_kernel(case):
    from oracle import closed_form as cf
    from pde_policylearning_b200 import ops
    grid, half, norm, ci, co, B, act = case
    dev = _dev()
    torch.manual_seed(11)
    g64 = cf.SpecGeom(nin=grid, half=half, norm=norm)
    plan = ops.get_plan(ops.SpecGeom(nin=grid, half=half, norm=norm), dev)
    sf, si = g64.scales()
    x = torch.randn(B, ci, *grid)
    yh = torch.randn(B, co, *plan.kept, dtype=torch.cfloat)
    w = torch.randn(co, ci)
    bias = torch.randn(co)
    dzt = torch.randn(B, co, *grid)
    f = {"gelu": torch.nn.functional.gelu, "relu": torch.relu, "tanh": torch.tanh, None: lambda t: t}[act]
    z64 = cf.idft_trunc(g64, yh.to(torch.complex128), si) + torch.einsum("oi,bi...->bo...", w.double(), x.double()) \
        + bias.double().reshape(1, -1, 1, 1)
    y64 = f(z64)
    zz = dzt.double().requires_grad_(True)
    torch.nn.functional.gelu(zz).sum().backward()
    y64_d = z64 * zz.grad
    xd, yhd, wd, bd, dzd = x.to(dev), yh.to(dev), w.to(dev), bias.to(dev), dzt.to(dev)
    outs = {}
    try:
        for mode in (True, False):
            assert ops.set_tensor_core_mode(mode) == mode
            n0 = ops.tensor_core_launches()
            z = torch.empty(B, co, *grid, device=dev)
            y = ops.dft_inverse(plan, 0, yhd, ops.make_epilogue(bias=bd, pw_w=wd, pw_x=xd, preact=z, act=act))
            yd = ops.dft_inverse(plan, 0, yhd, ops.make_epilogue(bias=bd, pw_w=wd, pw_x=xd, dact_z=dzd, dact="gelu"))
            assert (ops.tensor_core_launches() - n0 == 2) == mode, "tensor-core kernel did not run when expected"
            outs[mode] = (rel(z, z64), rel(y, y64), rel(yd, y64_d))
    finally:
        ops.set_tensor_core_mode(True)
    for mode, errs in outs.items():
        assert max(errs) < TOL, (mode, errs)


@pytest.mark.parametrize("case", [(2, 32, 32, (128, 128)), (1, 256, 32, (128, 64)), (3, 20, 3, (32, 32)), (2, 34, 34, (32, 32)),
                                  (1, 136, 40, (16, 16, 8))], ids=str)
def test_tensor_core_wgrad(case):
    """tc_wgrad.cu through b2no_pw_wgrad: dW, db vs float64, tensor-core and CUDA-core paths."""
    from pde_policylearning_b200 import ops
    B, co, ci, grid = case
    dev = _dev()
    torch.manual_seed(5)
    g = torch.randn(B, co, *grid, device=dev)
    x = torch.randn(B, ci, *grid, device=dev) + 0.5
    dw64 = torch.einsum("bo...,bi...->oi", g.double(), x.double())
    db64 = g.double().sum(dim=[0] + list(range(2, g.dim())))
    try:
        for mode in (True, False):
            ops.set_tensor_core_mode(mode)
            n0 = ops.tensor_core_launches()
            dw, db = ops.pw_wgrad(g, x, need_bias=True)
            assert (ops.tensor_core_launches() > n0) == mode
            assert rel(dw, dw64) < TOL and rel(db, db64) < TOL, (mode, rel(dw, dw64), rel(db, db64))
    finally:
        ops.set_tensor_core_mode(True)


@pytest.mark.parametrize("case", [(2, 32, 256, (128, 128), "gelu", False), (2, 34, 136, (32, 32), "relu", False),
                                  (2, 64, 128, (16, 16, 8), "gelu", True), (1, 8, 16, (16, 8), "tanh", False)], ids=str)
def test_tensor_core_mlp_head(case):
    """tc_mlp.cu: fused Ci -> hidden -> act -> 1 head, forward and backward, vs float64 autograd."""
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops
    B, ci, hid, grid, act, per_sample = case
    dev = _dev()
    torch.manual_seed(6)
    nd = len(grid)
    x = torch.randn(B, ci, *grid, device=dev, requires_grad=True)
    w1 = (torch.randn(hid, ci, device=dev) * 0.3).requires_grad_(True)
    b1 = torch.randn(*((B, hid) if per_sample else (hid,)), device=dev, requires_grad=True)
    w2 = (torch.randn(1, hid, device=dev) * 0.3).requires_grad_(True)
    b2 = torch.randn(1, device=dev, requires_grad=True)
    gout = torch.randn(B, 1, *grid, device=dev)
    f = {"gelu": torch.nn.functional.gelu, "relu": torch.relu, "tanh": torch.tanh}[act]
    xd, w1d, b1d, w2d, b2d = (t.detach().double().requires_grad_(True) for t in (x, w1, b1, w2, b2))
    bshape = (B, hid) + (1,) * nd if per_sample else (1, hid) + (1,) * nd
    h = f(torch.einsum("ji,bi...->bj...", w1d, xd) + b1d.reshape(bshape))
    ref = torch.einsum("oj,bj...->bo...", w2d, h) + b2d.reshape((1, 1) + (1,) * nd)
    gref = torch.autograd.grad(ref, [xd, w1d, b1d, w2d, b2d], gout.double())
    n0 = ops.tensor_core_launches()
    out = P.mlp_head(x, w1, b1, w2, b2, act)
    gs = torch.autograd.grad(out, [x, w1, b1, w2, b2], gout)
    assert ops.tensor_core_launches() - n0 >= 2, "fused tensor-core head did not run"
    assert rel(out, ref) < TOL
    for name, a, b in zip(("dx", "dw1", "db1", "dw2", "db2"), gs, gref):
        assert rel(a, b) < 2e-5, (name, rel(a, b))


@pytest.mark.parametrize("case", [(2, 32, 256, (128, 128), "gelu", False), (9, 32, 256, (128, 128), "gelu", True),
                                  (3, 20, 200, (16, 24), "gelu", False), (1, 8, 16, (16, 8), "tanh", False),
                                  (2, 16, 128, (8, 16, 4), "relu", True), (5, 32, 128, (64, 64), "gelu", False)], ids=str)
def test_head_backward_one_kernel(case):
    """tc_head_bwd.cu: gx, dW1, db1, dw2 of the Ci -> hidden -> act -> 1 head from ONE kernel (the hidden-channel gradient never
    reaches memory), vs float64 autograd; optional act'(dz) factor on gx; one / several tiles per CTA; padded channels / hidden."""
    from pde_policylearning_b200 import ops
    B, ci, hid, grid, act, with_dact = case
    dev = _dev()
    torch.manual_seed(8)
    nd = len(grid)
    assert ops.mlp_head_bwd_fused_supported(ci, hid, math.prod(grid))
    x = torch.randn(B, ci, *grid, device=dev)
    w1 = torch.randn(hid, ci, device=dev) * 0.3
    b1 = torch.randn(hid, device=dev)
    w2 = torch.randn(hid, device=dev) * 0.3
    g = torch.randn(B, 1, *grid, device=dev)
    dz = torch.randn(B, ci, *grid, device=dev) if with_dact else None
    f = {"gelu": torch.nn.functional.gelu, "relu": torch.relu, "tanh": torch.tanh}[act]
    xd, w1d, b1d, w2d = (t.double().requires_grad_(True) for t in (x, w1, b1, w2))
    h = f(torch.einsum("ji,bi...->bj...", w1d, xd) + b1d.reshape((1, hid) + (1,) * nd))
    ref = torch.einsum("j,bj...->b...", w2d, h).unsqueeze(1)
    gx64, dw164, db164, dw264 = torch.autograd.grad(ref, [xd, w1d, b1d, w2d], g.double())
    if with_dact:
        zd = dz.double().requires_grad_(True)
        gx64 = gx64 * torch.autograd.grad(torch.nn.functional.gelu(zd).sum(), zd)[0]
    n0 = ops.tensor_core_launches()
    gx, dw1, db1, dw2, db2 = ops.mlp_head_bwd_fused(x, w1, b1, w2, g, act, dact_z=dz, dact="gelu" if with_dact else None)
    assert ops.tensor_core_launches() == n0 + 1
    errs = dict(gx=rel(gx, gx64), dw1=rel(dw1, dw164), db1=rel(db1, db164), dw2=rel(dw2, dw264),
                db2=abs(float(db2) - float(g.double().sum())) / float(g.double().abs().sum()))
    print("head backward (one kernel)", case, {k: f"{v:.2e}" for k, v in errs.items()})
    for k, v in errs.items():
        assert v < 2e-5, (k, v)


# --------------------------------------------------------------------------------------------
# fused Adam (csrc/optim.cu) and the CUDA-graph training step
# --------------------------------------------------------------------------------------------
def test_fused_adam_matches_torch_adam():
    """Same update rule as torch.optim.Adam(lr, weight_decay) incl. complex parameters (run_pde_observers.py:134)."""
    import pde_policylearning_b200 as P
    dev = _dev()
    torch.manual_seed(21)
    shapes = [((7, 5), False), ((3,), False), ((4, 3, 2, 2), True), ((1,), False), ((130,), False)]
    mk = lambda: [torch.nn.Parameter(torch.randn(*s, dtype=torch.cfloat if c else torch.float32, device=dev)) for s, c in shapes]
    torch.manual_seed(22)
    pa = mk()
    pb = [torch.nn.Parameter(p.detach().clone()) for p in pa]
    ref = torch.optim.Adam(pb, lr=3e-3, weight_decay=1e-4)
    opt = P.FusedAdam(pa, lr=3e-3, weight_decay=1e-4)
    for it in range(5):
        opt.zero_grad()
        ref.zero_grad()
        for a, b in zip(pa, pb):
            g = torch.randn_like(a)
            a.grad.copy_(g)
            b.grad = g.clone()
        opt.step()
        ref.step()
    for a, b in zip(pa, pb):
        assert rel(a.detach(), b.detach()) < 1e-6


def test_graphed_train_step_matches_eager():
    """GraphedTrainStep (one CUDA graph per step) follows the same trajectory as the eager step."""
    import pde_policylearning_b200 as P
    dev = _dev()

    def build():
        torch.manual_seed(31)
        m = P.FNO2dObserver(6, 6, 8).to(dev)
        return m, P.FusedAdam(m.parameters(), lr=1e-3, weight_decay=1e-4)

    torch.manual_seed(32)
    xs = [torch.randn(4, 16, 16, 1, device=dev) for _ in range(3)]
    ts = [torch.randn(4, 1, 16, 16, device=dev) for _ in range(3)]
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
    assert int(o2.step_counter.item()) == 3


def test_grad_bucket_gather_and_loss_tail():
    """zero_grad(set_to_none=True) -> backward assigns fresh gradient tensors -> ONE gather kernel fills the flat bucket
    (unused parameters become zeros, complex gradients as (re, im)); LpLoss tail runs on the device."""
    import pde_policylearning_b200 as P
    dev = _dev()
    torch.manual_seed(41)
    a = torch.nn.Parameter(torch.randn(5, 3, device=dev))
    b = torch.nn.Parameter(torch.randn(4, 2, dtype=torch.cfloat, device=dev))
    c = torch.nn.Parameter(torch.randn(7, device=dev))          # never used: its slot must read zero
    opt = P.FusedAdam([a, b, c], lr=1e-3)
    opt.bucket.flat.fill_(123.0)                                # stale content must not survive
    opt.zero_grad(set_to_none=True)
    assert a.grad is None and b.grad is None
    x = torch.randn(6, 5, 3, device=dev)
    y = torch.randn(6, 4, 2, device=dev)
    out = torch.cat([(x * a).flatten(1), (y * b).abs().flatten(1)], dim=1)
    tgt = torch.randn_like(out)
    loss = P.rel_l2_loss(out, tgt, size_average=True)
    ref = ((out.double() - tgt.double()).flatten(1).norm(dim=1) / tgt.double().flatten(1).norm(dim=1)).mean()
    assert abs(loss.item() - ref.item()) < 1e-6 * abs(ref.item())
    ga, gb = torch.autograd.grad(ref, [a, b], retain_graph=True)
    loss.backward()
    opt.sync_grads()
    flat = opt.bucket.flat
    o = opt.bucket.offsets
    assert a.grad.data_ptr() == flat.data_ptr() + 4 * o[0]     # gradients are views of the bucket again
    assert rel(flat[o[0]:o[0] + 15].reshape(5, 3), ga) < 1e-5
    assert rel(torch.view_as_complex(flat[o[1]:o[1] + 16].reshape(4, 2, 2)), gb) < 1e-5
    assert float(flat[o[2]:o[2] + 7].abs().max()) == 0.0


def test_host_batch_pipeline_matches_direct_steps():
    """HostBatchPipeline (H2D of batch i+1 on a copy stream while step i runs) follows the same trajectory as feeding
    the same pinned batches to the graphed step one by one."""
    import pde_policylearning_b200 as P
    dev = _dev()

    def build():
        torch.manual_seed(51)
        m = P.FNO2dObserver(6, 6, 8).to(dev)
        o = P.FusedAdam(m.parameters(), lr=1e-3, weight_decay=1e-4)
        return m, o

    torch.manual_seed(52)
    xs = [torch.randn(4, 16, 16, 1).pin_memory() for _ in range(5)]
    ts = [torch.randn(4, 1, 16, 16).pin_memory() for _ in range(5)]
    loss_fn = lambda o, t: P.rel_l2_loss(o, t, size_average=False)
    m1, o1 = build()
    s1 = P.GraphedTrainStep(m1, loss_fn, o1, (xs[0].to(dev),), ts[0].to(dev))
    direct = [s1((x,), t).item() for x, t in zip(xs, ts)]
    m2, o2 = build()
    s2 = P.GraphedTrainStep(m2, loss_fn, o2, (xs[0].to(dev),), ts[0].to(dev))
    piped = [l.item() for l in P.HostBatchPipeline(s2).run(((x,), t) for x, t in zip(xs, ts))]
    for u, v in zip(direct, piped):
        assert abs(u - v) <= 1e-6 * abs(u), (direct, piped)
    assert rel(o2.flat_param, o1.flat_param) < 1e-6
    # deferred read-back: same losses, every step delivered
    m3, o3 = build()
    s3 = P.GraphedTrainStep(m3, loss_fn, o3, (xs[0].to(dev),), ts[0].to(dev))
    late = list(P.HostBatchPipeline(s3).run_losses(((x,), t) for x, t in zip(xs, ts)))
    assert len(late) == len(direct)
    for u, v in zip(direct, late):
        assert abs(u - v) <= 1e-6 * abs(u), (direct, late)
    s1.close()
    s2.close()
    s3.close()


# ---------------------------------------------------------------------------------------------
# round 2: tensor-core mixing, gate epilogue, the regrouped RNO layer, launch-evidence assertions
# ---------------------------------------------------------------------------------------------
MIX_CASES = [
    # grid, half, ci, co, batch, real-pair weights
    ((32, 32), (12, 12), 34, 34, 256, True),      # cfg3 RNO conv
    ((32, 32), (12, 12), 34, 68, 130, True),      # gate-stacked weights, ragged last tile
    ((16, 16), (4, 5), 10, 3, 200, False),        # odd channel counts (padding rows / columns)
    ((8, 8, 8), (2, 2, 3), 8, 8, 128, False),     # 3-D mode map (4 corners)
    ((64,), (9,), 16, 24, 128, False),            # 1-D
]


@pytest.mark.parametrize("case", MIX_CASES, ids=lambda c: "x".join(map(str, c[0])) + f"-{c[2]}to{c[3]}-b{c[4]}")
def test_tensor_core_mixing(case):
    """tc_mix.cu through b2no_mix / b2no_mix_dw (large batch): Yh, its adjoint, dW (plain and accumulated) vs complex128,
    on the tensor-core and the CUDA-core kernels."""
    from oracle import closed_form as cf
    from pde_policylearning_b200 import ops
    grid, half, ci, co, B, pairs = case
    dev = _dev()
    torch.manual_seed(5)
    g64 = cf.SpecGeom(nin=grid, half=half, norm="ortho")
    plan = ops.get_plan(ops.SpecGeom(nin=grid, half=half, norm="ortho"), dev)
    nc = 2 ** (len(grid) - 1)
    corners = [torch.randn(ci, co, *half, dtype=torch.cfloat) for _ in range(nc)]
    W = cf.gather_weight(g64, corners)
    xh = torch.randn(B, ci, *plan.kept, dtype=torch.cfloat)
    gyh = torch.randn(B, co, *plan.kept, dtype=torch.cfloat)
    y64 = torch.einsum("bi...,io...->bo...", xh.to(torch.complex128), W)
    gx64 = torch.einsum("bo...,io...->bi...", gyh.to(torch.complex128), W.conj())
    dW64 = cf.scatter_weight_grad(g64, torch.einsum("bi...,bo...->io...", xh.to(torch.complex128).conj(), gyh.to(torch.complex128)),
                                  [tuple(c.shape) for c in corners])
    cd = [(torch.view_as_real(c).contiguous() if pairs else c).to(dev) for c in corners]
    xhd, gyhd = xh.to(dev), gyh.to(dev)
    try:
        for mode in (True, False):
            assert ops.set_tensor_core_mode(mode) == mode
            n0 = ops.tensor_core_launches()
            y = ops.mix(plan, 0, xhd, cd, ci, co)
            gx = ops.mix(plan, 1, gyhd, cd, ci, co)
            gx2 = ops.mix(plan, 1, gyhd, cd, ci, co, out=gx.clone(), accumulate=True)
            dW = ops.mix_dw(plan, xhd, gyhd, cd, needs_zero=True)
            acc = [d.clone() for d in dW]
            ops.mix_dw(plan, xhd, gyhd, cd, needs_zero=False, out=acc, accumulate=True)
            assert (ops.tensor_core_launches() - n0 == 5) == mode, "tensor-core mixing kernel did not run when expected"
            as_c = lambda t: t if t.is_complex() else torch.view_as_complex(t.contiguous())
            errs = [rel(y, y64), rel(gx, gx64), rel(gx2, 2 * gx64)] + [rel(as_c(d), r) for d, r in zip(dW, dW64)] \
                + [rel(as_c(d), 2 * r) for d, r in zip(acc, dW64)]
            assert max(errs) < TOL, (mode, errs)
    finally:
        ops.set_tensor_core_mode(True)


def test_gate_epilogue_and_cell_backward_kernels():
    """The GRU update of rno.py:259 as the inverse-transform epilogue (gate_z / gate_h / strided mul), on the tile kernel and
    the CUDA-core kernel, and the two fused cell-backward kernels, vs float64."""
    from oracle import closed_form as cf
    from pde_policylearning_b200 import ops
    dev = _dev()
    torch.manual_seed(3)
    B, C, n, m = 3, 34, 32, 12
    g64 = cf.SpecGeom(nin=(n, n), half=(m, m), norm="ortho")
    plan = ops.get_plan(ops.SpecGeom(nin=(n, n), half=(m, m), norm="ortho"), dev)
    _, si = g64.scales()
    yh = torch.randn(B, C, *plan.kept, dtype=torch.cfloat)
    rh, h, add = torch.randn(B, C, n, n), torch.randn(B, C, n, n), torch.randn(B, C, n, n)
    zz2 = torch.rand(B, 2 * C, n, n)
    w = torch.randn(C, C) * 0.2
    a64 = cf.idft_trunc(g64, yh.to(torch.complex128), si) + torch.einsum("oi,bi...->bo...", w.double(), rh.double()) + add.double()
    hn64 = (1 - zz2[:, :C].double()) * h.double() + zz2[:, C:].double() * torch.nn.functional.selu(a64)
    yhd, rhd, hd, addd, zd, wd = (t.to(dev) for t in (yh, rh, h, add, zz2, w))
    try:
        for mode in (True, False):
            ops.set_tensor_core_mode(mode)
            ah = torch.empty(B, C, n, n, device=dev)
            hn = ops.dft_inverse(plan, 0, yhd, ops.make_epilogue(pw_w=wd, pw_x=rhd, add=addd, act="selu", preact=ah,
                                                                mul=zd[:, C:], gate_z=zd[:, :C], gate_h=hd))
            assert rel(ah, a64) < TOL and rel(hn, hn64) < TOL, (mode, rel(ah, a64), rel(hn, hn64))
    finally:
        ops.set_tensor_core_mode(True)
    # fused backward kernels
    g = torch.randn(B, C, n, n)
    ahc = a64.float()
    z, z2 = zz2[:, :C].double(), zz2[:, C:].double()
    a = ahc.double().requires_grad_(True)
    hh = torch.nn.functional.selu(a)
    (dselu,) = torch.autograd.grad(hh.sum(), a)
    g_zz2 = torch.empty(B, 2 * C, n, n, device=dev)
    g_ah = torch.empty(B, C, n, n, device=dev)
    g_h = ops.rno_cell_bwd(g.to(dev), hd, zd, ahc.to(dev), g_zz2, g_ah)
    gd = g.double()
    assert rel(g_zz2[:, :C], -gd * h.double() * z * (1 - z)) < TOL
    assert rel(g_zz2[:, C:], gd * hh.detach() * z2 * (1 - z2)) < TOL
    assert rel(g_ah, gd * z2 * dselu) < TOL and rel(g_h, gd * (1 - z)) < TOL
    ar = torch.randn(B, C, n, n)
    r = torch.sigmoid(ar.double())
    g_ar = torch.empty(B, C, n, n, device=dev)
    gh0 = torch.randn(B, C, n, n)
    ghd = gh0.to(dev).clone()
    ops.rno_reset_bwd(g.to(dev), hd, ar.to(dev), g_ar, ghd)
    assert rel(g_ar, gd * h.double() * r * (1 - r)) < TOL and rel(ghd, gh0.double() + gd * r) < TOL


def test_rno_layer_regrouped_vs_reference_composition():
    """cfg3 layer shape (width 34, modes 12, 32x32), B = 128 so that the tensor-core mixing runs: the regrouped layer
    (functional.RnoLayerFn) against autograd through the un-regrouped composition of the same kernels' FourierLayer2d
    calls -- outputs, dx, dh0 and every parameter gradient."""
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops
    dev = _dev()
    torch.manual_seed(0)
    layer = P.RNO_layer(34, 34, 12, 12, 34, return_sequences=False).to(dev)
    B, T = 128, 3
    x = torch.randn(B, T, 34, 32, 32, device=dev, requires_grad=True)
    h0 = torch.randn(B, 34, 32, 32, device=dev, requires_grad=True)
    n0 = ops.tensor_core_launches()
    out = layer(x, h0)
    gy = torch.randn_like(out)
    params = list(layer.parameters())
    got = torch.autograd.grad(out, [x, h0] + params, gy, allow_unused=True)
    assert ops.tensor_core_launches() > n0
    cell = layer.cell
    h = h0
    for t in range(T):
        xt = x[:, t]
        z = torch.sigmoid(cell.f1(xt) + cell.f2(h, extra_bias=cell.b1))
        z2 = torch.sigmoid(cell.f7(xt) + cell.f8(h, extra_bias=cell.b4))
        r = torch.sigmoid(cell.f3(xt) + cell.f4(h, extra_bias=cell.b2))
        hh = torch.nn.functional.selu(cell.f5(xt) + cell.f6(r * h, extra_bias=cell.b3))
        h = (1 - z) * h + z2 * hh
    ref = torch.autograd.grad(h, [x, h0] + params, gy, allow_unused=True)
    assert rel(out, h) < TOL, rel(out, h)
    names = ["x", "h0"] + [n for n, _ in layer.named_parameters()]
    worst = 0.0
    for n, a, b in zip(names, got, ref):
        if b is None:               # bias_h is not reached when h0 is given
            continue
        assert a is not None, n
        e = rel(a, b)
        worst = max(worst, e)
        assert e < 5e-5, (n, e)
    print(f"regrouped RNO layer: worst relative gradient error {worst:.2e}")


def test_dft_forward_runs_on_tensor_cores_at_bench_shapes():
    """Launch evidence: at the cfg2 plane shape b2no_dft_forward must take the tcgen05 kernel (k_fwd_tc), at the cfg3 shape
    (32 x 32 planes) the one-launch warp-per-plane kernel, never the two CUDA-core stages -- a silent fallback would pass every
    numeric test at several times the cost."""
    from pde_policylearning_b200 import ops
    dev = _dev()
    for grid, half, norm, C in (((128, 128), (6, 6), "forward", 32), ((32, 32), (12, 12), "ortho", 34)):
        plan = ops.get_plan(ops.SpecGeom(nin=grid, half=half, norm=norm), dev)
        x = torch.randn(4, C, *grid, device=dev)
        for which in (0, 1):
            n0, l0 = ops.tensor_core_launches(), ops.launch_count()
            ops.dft_forward(plan, which, x)
            if grid == (32, 32):
                # small planes: ONE launch of the warp-per-plane kernel (k_fwd_plane32), not the two CUDA-core stages
                assert ops.tensor_core_launches() == n0 and ops.launch_count() == l0 + 1, (grid, which)
            else:
                assert ops.tensor_core_launches() == n0 + 1, (grid, which)
        spec = torch.randn(4, C, *plan.kept, dtype=torch.cfloat, device=dev)
        w = torch.randn(C, C, device=dev)
        n0 = ops.tensor_core_launches()
        ops.dft_inverse(plan, 0, spec, ops.make_epilogue(pw_w=w, pw_x=x))
        assert ops.tensor_core_launches() == n0 + 1, (grid, "inverse")


def test_golden_pino_family_mirrors(golden):
    """SURVEY 8f rank 4: PINObserverFullField (+ PlanePredHead), PolicyModel2D, pino_models.fourier2d.FNO2d on the CUDA path
    against the reference's fixtures a10-a12 (outputs, loss, every parameter gradient)."""
    import pde_policylearning_b200 as P
    dev = _dev()
    kw = dict(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4, act="gelu", pad_ratio=0.0625)
    w = [_run_model(P.PINObserverFullField(plane_num=3, **kw), golden("a10_pinobserver_fullfield"), dev, gtol=2e-4),
         _run_model(P.PolicyModel2D(**kw), golden("a11_policy_model2d"), dev, gtol=2e-4),
         _run_model(P.PinoFNO2d(modes1=[4] * 3, modes2=[3] * 3, fc_dim=12, layers=[6, 8, 8, 5], in_dim=3, out_dim=2, act="gelu",
                                pad_ratio=[0.125, 0.0625]), golden("a12_pino_fno2d"), dev, gtol=2e-4),
         _run_model(P.PinoFNO2d(modes1=[4] * 2, modes2=[3] * 2, fc_dim=8, layers=[4, 6, 4], in_dim=3, out_dim=1, act="gelu"),
                    golden("a12_pino_fno2d_nopad"), dev, gtol=2e-4)]
    print("worst relative gradient errors (full-field, policy, pino fno2d, pino fno2d no pad):", ["%.1e" % e for e in w])
    # inference (no_grad) path of the trunk: per-sample Reynolds bias in the fused head == training path
    c = golden("a10_pinobserver_fullfield")
    m = P.PINObserverFullField(plane_num=3, **kw)
    m.load_state_dict(c["state_dict"])
    m = m.to(dev)
    with torch.no_grad():
        assert rel(m(*[t.to(dev) for t in c["inputs"]]), c["out"]) < TOL


def test_pinobserver_per_sample_bias_odd_width():
    """ADVICE r1: a trunk whose last width has no fused-head kernel (20 channels) with B > 1 and distinct Reynolds numbers --
    eval (no_grad) output must equal the train-mode output (the Reynolds term is per sample)."""
    import pde_policylearning_b200 as P
    dev = _dev()
    torch.manual_seed(2)
    m = P.PINObserver2d(modes1=[2] * 2, modes2=[2] * 2, modes3=[2] * 2, fc_dim=12, layers=[20] * 3, act="gelu",
                        pad_ratio=0.0625).to(dev)
    a = torch.randn(3, 8, 8, 9, 4, device=dev)
    re = torch.tensor([100.0, 300.0, 500.0], device=dev)
    out_train = m(a, re)
    with torch.no_grad():
        out_eval = m(a, re)
    assert rel(out_eval, out_train) < TOL
    assert rel(out_train[0], out_train[2]) > 1e-3         # the Reynolds number does enter


@pytest.mark.parametrize("N,T,B", [(64, 9, 2), (16, 5, 3), (8, 17, 2)], ids=str)
def test_pino_residual_fused_kernels_vs_composition(N, T, B):
    """csrc/pino_loss.cu (fused FDM_NS_vorticity + both relative-L2 losses + hand-derived backward) against the float64
    composition of DFT-matrix products with autograd (pino_loss.fdm_ns_vorticity): Du, loss_ic, loss_f and d loss / d w."""
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops, pino_loss
    dev = _dev()
    torch.manual_seed(4)
    w = torch.randn(B, N, N, T, dtype=torch.float64)
    w = torch.fft.irfft2(torch.fft.rfft2(w, dim=(1, 2)) * torch.exp(-0.05 * torch.arange(N // 2 + 1, dtype=torch.float64) ** 2).reshape(1, 1, -1, 1),
                         s=(N, N), dim=(1, 2))                      # smooth in y so that the residual is O(1)
    u0 = torch.randn(B, N, N, dtype=torch.float64)
    forcing = P.get_forcing(N).double()
    nu = 1.0 / torch.tensor([100.0 + 150.0 * i for i in range(B)], dtype=torch.float64)
    ti = 0.5
    w64 = w.clone().requires_grad_(True)
    du64 = pino_loss.fdm_ns_vorticity(w64, nu, ti)
    relm = lambda a, b: (torch.linalg.vector_norm((a - b).reshape(B, -1), dim=1) / torch.linalg.vector_norm(b.reshape(B, -1), dim=1)).mean()
    lic64 = relm(w64[..., 0], u0)
    lf64 = relm(du64, forcing.expand(B, N, N, T - 2))
    (dw64,) = torch.autograd.grad(0.7 * lic64 + 1.3 * lf64, w64)
    wd = w.float().to(dev).requires_grad_(True)
    lic, lf = P.channelflow_pino_loss(wd, u0.float().to(dev), forcing.float().to(dev), nu.float().to(dev), ti)
    (dw,) = torch.autograd.grad(0.7 * lic + 1.3 * lf, wd)
    assert abs(lic.item() - lic64.item()) <= 2e-6 * abs(lic64.item()), (lic.item(), lic64.item())
    assert abs(lf.item() - lf64.item()) <= 1e-5 * abs(lf64.item()), (lf.item(), lf64.item())
    assert rel(dw, dw64) < 2e-5, rel(dw, dw64)
    with torch.no_grad():
        du = P.fdm_ns_vorticity(wd.detach(), nu.float().to(dev), ti)
    assert rel(du, du64) < TOL, rel(du, du64)


def test_single_pass_tf32_mode_within_2e2():
    """g1: the reduced-precision tensor-core mode (one kind::tf32 MMA per product instead of the 3xTF32 triple) -- FNO2d
    block stack, RNO conv and the projection head stay within the north star's 2e-2 of the float64 restatement, and the
    mode really changes the arithmetic (error above the fp32-mode level)."""
    import pde_policylearning_b200 as P
    from oracle import restated as rs
    dev = _dev()
    torch.manual_seed(9)
    obs = P.FNO2dObserver(12, 12, 32).to(dev)
    p = torch.randn(4, 128, 128, 1, device=dev)
    tgt = torch.randn(4, 1, 128, 128, device=dev)
    sd = {k: (v.detach().cpu().to(torch.complex128) if v.is_complex() else v.detach().cpu().double()) for k, v in obs.state_dict().items()}
    ref = rs.fno2d_observer_forward(sd, p.cpu().double(), 12)
    errs = {}
    try:
        for mode in ("fp32", "tf32"):
            assert P.set_precision(mode) == mode
            out = obs(p)
            loss = P.rel_l2_loss(out, tgt, size_average=False)
            gs = torch.autograd.grad(loss, list(obs.parameters()))
            assert all(torch.isfinite(g).all() for g in gs)
            errs[mode] = rel(out, ref)
    finally:
        P.set_precision("fp32")
    print("FNO2dObserver 128x128 output error vs float64:", {k: f"{v:.2e}" for k, v in errs.items()})
    assert errs["tf32"] < 2e-2
    assert errs["tf32"] > 3 * errs["fp32"]


@pytest.mark.parametrize("m", [(3, 3, 4), (3, 2, 8)], ids=str)
def test_3d_layer_pointwise_on_tensor_cores(m):
    """PINO layer shape class (3-D, rows that are not multiples of the pixel tile): spectral conv + Conv1d(k=1) + bias +
    GELU with the 1x1 convolution on the tcgen05 tile kernel (transform result handed over through `add`), y, dx and
    parameter gradients vs the float64 closed form; the tile kernel must actually run."""
    import pde_policylearning_b200 as P
    from oracle import closed_form as cf
    from pde_policylearning_b200 import ops
    dev = _dev()
    torch.manual_seed(6)
    # 8 * 8 * 18 = 1152 = 9 * 128 pixels, rows of 18.  The second case (8 kept last-dim modes, 32768 rows) takes the kernels
    # of the PINO shape: k_r2c_rows32 (lane = row) and k_c2r_plain8
    B, C = 2, 16
    grid = (8, 8, 18) if m[2] != 8 else (32, 32, 18)
    conv = P.PinoSpectralConv3d(C, C, *m)
    w = torch.randn(C, C, 1) * 0.3
    bias = torch.randn(C)
    x = torch.randn(B, C, *grid)
    gy = torch.randn(B, C, *grid)
    g64 = cf.geom_pino3d(grid, *m)
    corners = [c.detach().clone() for c in conv.corners()]
    x64 = x.double().requires_grad_(True)
    w64, b64 = w.double().requires_grad_(True), bias.double().requires_grad_(True)
    sf, si = g64.scales()
    W = cf.gather_weight(g64, corners)
    z64 = cf.idft_trunc(g64, torch.einsum("bi...,io...->bo...", cf.dft_trunc(g64, x64, sf), W), si) \
        + torch.einsum("oi,bi...->bo...", w64[:, :, 0], x64) + b64.reshape(1, -1, 1, 1, 1)
    y64 = torch.nn.functional.gelu(z64)
    dx64, dw64, db64 = torch.autograd.grad(y64, [x64, w64, b64], gy.double())
    conv = conv.to(dev)
    xd = x.to(dev).requires_grad_(True)
    wd, bd = w.to(dev).requires_grad_(True), bias.to(dev).requires_grad_(True)
    n0 = ops.tensor_core_launches()
    y = conv.forward_fused(xd, bias=bd, pw_weight=wd, act="gelu")
    assert ops.tensor_core_launches() > n0, "the 3-D layer's 1x1 conv did not reach the tile kernel"
    dx, dw, db = torch.autograd.grad(y, [xd, wd, bd], gy.to(dev))
    errs = dict(y=rel(y, y64), dx=rel(dx, dx64), dw=rel(dw, dw64), db=rel(db, db64))
    assert max(errs.values()) < TOL, errs


def test_pinobserver_training_through_fused_head():
    """The PINO tail in training: fused head (per-sample Reynolds bias, hidden never materialised) vs the composition of
    two pointwise convs with the Reynolds term as a 1-channel map -- output and every parameter gradient."""
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import functional as Fn, ops
    dev = _dev()
    torch.manual_seed(8)
    m = P.PINObserver2d(modes1=[3] * 2, modes2=[3] * 2, modes3=[3] * 2, fc_dim=32, layers=[16] * 3, act="gelu",
                        pad_ratio=0.0625).to(dev)
    a = torch.randn(3, 8, 8, 14, 4, device=dev)             # 14 + 1 + 1 padded time steps: 8 * 8 * 16 = 1024 pixels
    re = torch.tensor([120.0, 260.0, 480.0], device=dev)
    gy = torch.randn(3, 8, 8, 14, 1, device=dev)
    params = list(m.parameters())
    n0 = ops.tensor_core_launches()
    assert Fn.mlp_head_fused_available(torch.empty(3, 16, 8, 8, 16, device=dev), m.fc1.weight, m.fc2.weight, None, True)
    out = m(a, re)
    g1 = torch.autograd.grad(out, params, gy)
    assert ops.tensor_core_launches() > n0
    saved = Fn.mlp_head_fused_available
    Fn.mlp_head_fused_available = lambda *args, **kw: False
    try:
        out2 = m(a, re)
        g2 = torch.autograd.grad(out2, params, gy)
    finally:
        Fn.mlp_head_fused_available = saved
    assert rel(out, out2) < TOL
    worst = max(rel(x, y) for x, y in zip(g1, g2))
    assert worst < 5e-5, worst


@pytest.mark.parametrize("ci,ci2,co", [(64, 1, 128), (128, 0, 64), (72, 0, 34)], ids=str)
def test_tile_kernel_single_a_buffer(ci, ci2, co):
    """Wide 1x1 convolutions whose double-buffered TMEM operand does not fit 512 columns (PINO tail 64 -> 128 with the
    Reynolds map, its dx 128 -> 64, the RNO gate dx 68 -> 34) run the tile kernel with ONE operand buffer instead of
    dropping to the CUDA-core kernel."""
    from pde_policylearning_b200 import ops
    dev = _dev()
    torch.manual_seed(12)
    B, grid = 2, (16, 32)
    x = torch.randn(B, ci, *grid)
    w = torch.randn(co, ci) * 0.2
    bias = torch.randn(co)
    z64 = torch.einsum("oi,bi...->bo...", w.double(), x.double()) + bias.double().reshape(1, -1, 1, 1)
    kw = {}
    if ci2:
        x2 = torch.randn(B, ci2, *grid)
        w2 = torch.randn(co, ci2)
        z64 = z64 + torch.einsum("oi,bi...->bo...", w2.double(), x2.double())
        kw = dict(pw2_w=w2.to(dev), pw2_x=x2.to(dev))
    n0 = ops.tensor_core_launches()
    y = ops.pointwise(B, co, grid, dev, ops.make_epilogue(bias=bias.to(dev), pw_w=w.to(dev), pw_x=x.to(dev), act="gelu", **kw))
    assert ops.tensor_core_launches() == n0 + 1, "tile kernel did not run"
    assert rel(y, torch.nn.functional.gelu(z64)) < TOL


def _sd_as(m, real_dtype):
    cdt = torch.complex128 if real_dtype == torch.float64 else torch.complex64
    sd = {}
    for k, v in m.state_dict().items():
        v = v.detach()
        sd[k] = (v.to(cdt) if v.is_complex() else v.to(real_dtype)).clone().requires_grad_(True)
    return sd


def _check_vs_ref32(names, gs, gs64, gs32, floor, what):
    """Every parameter gradient against the float64 restatement: within `floor`, or -- for gradients that are sums with
    heavy cancellation at full size -- within 4x what the reference's OWN fp32 arithmetic (the restated torch.fft / einsum
    algorithm run in float32 on the same inputs) achieves against float64."""
    worst, worst32 = 0.0, 0.0
    for n, a, b64, b32 in zip(names, gs, gs64, gs32):
        e, e32 = rel(a, b64), rel(b32, b64)
        worst, worst32 = max(worst, e), max(worst32, e32)
        assert e < max(floor, 4.0 * e32), (what, n, e, e32)
    return worst, worst32


def test_cfg3_rno_full_size_vs_restated():
    """BASELINE config 3 shape: RNO2dObserver(12,12,34, layer_num 1) on B = 256 trajectories of 32x32 planes (T = 4 frames of
    the 100: 7 recurrent cell steps + 4 regressor calls, every kernel at its bench shape incl. the tensor-core mixing),
    `.eval()`; output, loss and every parameter gradient against the restated reference algorithm in float64."""
    import pde_policylearning_b200 as P
    from oracle import restated as rs
    dev = _dev()
    torch.manual_seed(13)
    m = P.RNO2dObserver(12, 12, 34, 0, layer_num=1).to(dev).eval()
    B, T = 256, 4
    x = torch.randn(B, T, 32, 32, 1, device=dev)
    tgt = torch.randn(B, 32, 32, 1, device=dev)
    out = m(x)
    loss = P.rel_l2_loss(out.reshape(B, -1), tgt.reshape(B, -1), size_average=False)
    names = [n for n, _ in m.named_parameters()]
    gs = torch.autograd.grad(loss, [p for _, p in m.named_parameters()])
    res = {}
    for dt in (torch.float64, torch.float32):
        sd = _sd_as(m, dt)
        o = rs.rno2d_forward(sd, x.to(dt), 12, 12, 34, recurrent_index=0, layer_num=1)
        l = rs.lp_rel(o.reshape(B, -1), tgt.to(dt).reshape(B, -1), size_average=False)
        res[dt] = (o, l, torch.autograd.grad(l, [sd[n] for n in names]))
    out64, loss64, gs64 = res[torch.float64]
    eo = rel(out, out64)
    worst, worst32 = _check_vs_ref32(names, gs, gs64, res[torch.float32][2], 2e-4, "cfg3")
    print(f"cfg3 full size: output {eo:.2e} (reference fp32 arithmetic: {rel(res[torch.float32][0], out64):.2e}), loss "
          f"{abs(loss.item() - loss64.item()) / abs(loss64.item()):.2e}, worst gradient {worst:.2e} (reference fp32: {worst32:.2e})")
    assert eo < 2e-5, eo
    assert abs(loss.item() - loss64.item()) < 1e-5 * abs(loss64.item())


def test_cfg4_pino_full_size_vs_restated():
    """BASELINE config 4 shape: PINObserver2d (4 x 64 channels, modes 8, fc 128, pad 0.0625) on ONE 64x64x65 sample with
    the training loss 5 data + f + ic (train_pino.py:87-107; fused residual-loss kernels, fused head); output, the
    loss and every parameter gradient against the restated reference algorithm in float64."""
    import pde_policylearning_b200 as P
    from oracle import restated as rs
    dev = _dev()
    torch.manual_seed(14)
    m = P.PINObserver2d(modes1=[8] * 4, modes2=[8] * 4, modes3=[8] * 4, fc_dim=128, layers=[64] * 5, act="gelu",
                        pad_ratio=0.0625).to(dev)
    S, T = 64, 65
    a_in = torch.randn(1, S, S, T, 4, device=dev)
    u = torch.randn(1, S, S, T, device=dev)
    re = torch.tensor([250.0], device=dev)
    forcing = P.get_forcing(S, device=dev)
    out = m(a_in, re)
    loss = P.pino_training_loss(m, a_in, re, u, forcing, 5.0, 1.0, 1.0, 0.5)
    names = [n for n, _ in m.named_parameters()]
    gs = torch.autograd.grad(loss, [p for _, p in m.named_parameters()])
    res = {}
    for dt in (torch.float64, torch.float32):
        sd = _sd_as(m, dt)
        o = rs.pinobserver2d_forward(sd, a_in.to(dt), re.to(dt), [8] * 4, [8] * 4, [8] * 4, [64] * 5, 0.0625)
        o4 = o.reshape(1, S, S, T)
        lic, lf = rs.channelflow_pino_loss(o4, a_in[:, :, :, 0, -1].to(dt), forcing.to(dt), 1.0 / re.to(dt), 0.5)
        l = 5.0 * rs.lp_rel(o4, u.to(dt)) + lf + lic
        res[dt] = (o, l, torch.autograd.grad(l, [sd[n] for n in names]))
    out64, loss64, gs64 = res[torch.float64]
    eo = rel(out, out64)
    worst, worst32 = _check_vs_ref32(names, gs, gs64, res[torch.float32][2], 2e-4, "cfg4")
    print(f"cfg4 full size: output {eo:.2e} (reference fp32 arithmetic: {rel(res[torch.float32][0], out64):.2e}), loss "
          f"{abs(loss.item() - loss64.item()) / abs(loss64.item()):.2e}, worst gradient {worst:.2e} (reference fp32: {worst32:.2e})")
    assert eo < 2e-5, eo
    assert abs(loss.item() - loss64.item()) < 2e-5 * abs(loss64.item())


def test_mode_major_spectrum_layout():
    """b2no_geom.spec_layout = 1 (kept modes outermost): every op of the RNO layer -- forward DFT, its adjoint twin, mixing,
    adjoint mixing (plain and accumulated), dW (plain and accumulated), inverse with epilogue -- gives bit-for-bit the same
    numbers as the default layout (same kernels, different addressing), at the cfg3 layer shape."""
    from pde_policylearning_b200 import ops
    dev = _dev()
    torch.manual_seed(21)
    g0 = ops.SpecGeom(nin=(32, 32), half=(12, 12), norm="ortho")
    p0, p1 = ops.get_plan(g0, dev), ops.get_plan(g0.with_layout(1), dev)
    B, C = 160, 34
    assert p1.layout_supported(B, C)
    mm = lambda s: s.permute(2, 3, 0, 1).contiguous()            # (B, C, Kx, Ky) -> (Kx, Ky, B, C)
    x = torch.randn(B, C, 32, 32, device=dev)
    w = [torch.randn(C, 2 * C, 12, 12, 2, device=dev) * 0.1 for _ in range(2)]
    pw = torch.randn(2 * C, C, device=dev) * 0.2
    add = torch.randn(B, 2 * C, 32, 32, device=dev)
    for which in (0, 1):
        a, b = ops.dft_forward(p0, which, x), ops.dft_forward(p1, which, x)
        assert b.shape == (24, 12, B, C) and torch.equal(mm(a), b), which
    xh0 = ops.dft_forward(p0, 0, x)
    xh1 = mm(xh0)
    y0, y1 = ops.mix(p0, 0, xh0, w, C, 2 * C), ops.mix(p1, 0, xh1, w, C, 2 * C)
    assert y1.shape == (24, 12, B, 2 * C) and rel(y1, mm(y0)) < 1e-7
    gx0, gx1 = ops.mix(p0, 1, y0, w, C, 2 * C), ops.mix(p1, 1, y1, w, C, 2 * C)
    assert rel(gx1, mm(gx0)) < 1e-7
    acc1 = ops.mix(p1, 1, y1, w, C, 2 * C, out=gx1.clone(), accumulate=True)
    assert rel(acc1, 2 * mm(gx0)) < 1e-6
    d0 = ops.mix_dw(p0, xh0, y0, w, needs_zero=False)
    d1 = ops.mix_dw(p1, xh1, y1, w, needs_zero=False)
    assert all(rel(a, b) < 1e-6 for a, b in zip(d1, d0))
    ops.mix_dw(p1, xh1, y1, w, needs_zero=False, out=d1, accumulate=True)
    assert all(rel(a, 2 * b) < 1e-6 for a, b in zip(d1, d0))
    e = lambda: ops.make_epilogue(pw_w=pw, pw_x=x, add=add, act="sigmoid")
    z0, z1 = ops.dft_inverse(p0, 0, y0, e()), ops.dft_inverse(p1, 0, mm(y0), e())
    assert torch.equal(z0, z1)
