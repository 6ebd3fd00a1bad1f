"""Projection heads with 2..4 output channels on the fused head kernels (b2no_mlp_head_fwd_multi / b2no_mlp_head_bwd_multi,
functional.MlpHeadMultiFn): the ops against float64 autograd of the composed definition, the routing of mlp_head and of the
PINO tail, whole models against the float64 restatements, a captured training step, the memory the hidden tensor no longer
takes, and (on the CPU, with the emulated ops) the host logic against the reference fixtures."""
import contextlib
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ops_emulator as emu  # noqa: E402

ACTS = {"gelu": F.gelu, "relu": F.relu, "tanh": torch.tanh}
PINO_KW = dict(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4, act="gelu", pad_ratio=0.0625)


def rel(a, b):
    cv = lambda t: t.detach().cpu().to(torch.complex128 if t.is_complex() else torch.float64)
    a, b = cv(a), cv(b)
    den = torch.linalg.vector_norm(b).item()
    return torch.linalg.vector_norm(a - b).item() / (den if den > 0 else 1.0)


def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _head_ref(x, w1, b1, w2, b2, act):
    """The composed definition (tfno.py:34-38): Conv(C->H) -> act -> Conv(H->O), b1 (H) or per sample (B, H)."""
    nd = x.dim() - 2
    z = torch.einsum("ji,bi...->bj...", w1, x)
    z = z + (b1.reshape((1, -1) + (1,) * nd) if b1.dim() == 1 else b1.reshape(b1.shape + (1,) * nd))
    return torch.einsum("oj,bj...->bo...", w2, ACTS[act](z)) + b2.reshape((1, -1) + (1,) * nd)


def _ff_inputs(B, X, T, seed, dev="cpu"):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(B, X, X, T, 4, generator=g)
    re = torch.tensor([100.0 + 200.0 * i for i in range(B)])
    return a.to(dev), re.to(dev)


def _restated_fullfield(sd, a, re):
    """float64 PINObserverFullField (oracle/restated.py) with autograd leaves for every state_dict entry."""
    from oracle import restated as rs
    leaves = {k: (v.detach().cpu().to(torch.complex128 if v.is_complex() else torch.float64)).requires_grad_(True)
              for k, v in sd.items()}
    out = rs.pinobserver_fullfield_forward(leaves, a.double().cpu(), re.double().cpu(), PINO_KW["modes1"], PINO_KW["modes2"],
                                           PINO_KW["modes3"], PINO_KW["layers"], PINO_KW["pad_ratio"])
    return out, leaves


# float64 definitions of the multi-output head ops (include/b2no.h), on top of the emulated ops of ops_emulator.py
def _emu_multi_supported(x, hidden, out_channels):
    """Shape rule of b2no_mlp_head_bwd_multi_supported, without the device's shared-memory budget."""
    return 2 <= out_channels <= 4 and x.shape[1] <= 64 and hidden <= 512 and math.prod(x.shape[2:]) % 128 == 0


def _emu_z(x, w1, b1):
    nd = x.dim() - 2
    z = torch.einsum("ji,bi...->bj...", w1.double(), x.double())
    if b1 is not None:
        z = z + (b1.double().reshape((1, -1) + (1,) * nd) if b1.dim() == 1 else b1.double().reshape(b1.shape + (1,) * nd))
    return z


def _emu_act_grad(z, act):
    z = z.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        (g,) = torch.autograd.grad(ACTS[act](z).sum(), z)
    return g


def _emu_fwd_multi(x, w1, b1, w2, b2, act="gelu"):
    """b2no_mlp_head_fwd_multi: out[b,o] = b2[o] + sum_j w2[o,j] act(z1[b,j])."""
    nd = x.dim() - 2
    y = torch.einsum("oj,bj...->bo...", w2.double(), ACTS[act](_emu_z(x, w1, b1)))
    if b2 is not None:
        y = y + b2.double().reshape((1, -1) + (1,) * nd)
    return y.float()


def _emu_bwd_multi(x, w1, b1, w2, g, act="gelu", want_gz=True, dact_z=None, dact=None):
    """b2no_mlp_head_bwd_multi: (gx, gz | None, dw2 (O, hidden))."""
    z = _emu_z(x, w1, b1)
    f = _emu_act_grad(z, act) * torch.einsum("oj,bo...->bj...", w2.double(), g.double())
    gx = torch.einsum("ji,bj...->bi...", w1.double(), f)
    if dact_z is not None:
        gx = gx * _emu_act_grad(dact_z.double(), dact)
    dw2 = torch.einsum("bo...,bj...->oj", g.double(), ACTS[act](z))
    return gx.float(), (f.float() if want_gz else None), dw2.float()


@contextlib.contextmanager
def _emulated(supported=_emu_multi_supported):
    """ops_emulator.installed() plus the multi-output head ops (host-logic tests on the CPU)."""
    import pde_policylearning_b200.ops as ops
    names = ("mlp_head_multi_supported", "mlp_head_fwd_multi", "mlp_head_bwd_multi")
    saved = {n: getattr(ops, n) for n in names}
    with emu.installed():
        try:
            for n, f in zip(names, (supported, _emu_fwd_multi, _emu_bwd_multi)):
                setattr(ops, n, f)
            yield
        finally:
            for n, f in saved.items():
                setattr(ops, n, f)


class _Counting:
    """Counts the calls of the multi-output head ops (the route mlp_head / the PINO tail took)."""

    def __init__(self, ops):
        self.ops, self.n_fwd, self.n_bwd = ops, 0, 0

    def __enter__(self):
        self.fwd, self.bwd = self.ops.mlp_head_fwd_multi, self.ops.mlp_head_bwd_multi

        def fwd(*a, **k):
            self.n_fwd += 1
            return self.fwd(*a, **k)

        def bwd(*a, **k):
            self.n_bwd += 1
            return self.bwd(*a, **k)

        self.ops.mlp_head_fwd_multi, self.ops.mlp_head_bwd_multi = fwd, bwd
        return self

    def __exit__(self, *exc):
        self.ops.mlp_head_fwd_multi, self.ops.mlp_head_bwd_multi = self.fwd, self.bwd


# ------------------------------------------------------------------------------------------------------------------------
# CPU: host logic with the emulated ops
# ------------------------------------------------------------------------------------------------------------------------
def test_fullfield_fixture_through_the_multi_output_route_emulated(golden):
    """PINObserverFullField (plane_num = 3: a 3-output tail with the per-sample Reynolds bias) through MlpHeadMultiFn against
    the reference fixture a10: output and every parameter gradient.  The fixture's padded grid (8 x 8 x 11) is not a multiple
    of 128 pixels, which the kernels need, so the shape rule is widened here to reach the route with the fixture's data."""
    import pde_policylearning_b200 as P
    import pde_policylearning_b200.ops as ops
    c = golden("a10_pinobserver_fullfield")
    with _emulated(supported=lambda x, hidden, n_out: 2 <= n_out <= 4), _Counting(ops) as cnt:
        m = P.PINObserverFullField(plane_num=3, **PINO_KW)
        m.load_state_dict(c["state_dict"])
        out = m(*c["inputs"])
        assert rel(out, c["out"]) < 2e-5
        gs = torch.autograd.grad(out.square().mean(), [p for _, p in m.named_parameters()])
        with torch.no_grad():
            assert rel(m(*c["inputs"]), c["out"]) < 2e-5
    assert (cnt.n_fwd, cnt.n_bwd) == (2, 1)
    for (n, _), g in zip(m.named_parameters(), gs):
        assert rel(g, c["grads"][n]) < 1e-4, (n, rel(g, c["grads"][n]))


def test_fno2d_two_outputs_emulated():
    """FNO2d(out_channels=2): Projection -> mlp_head -> MlpHeadMultiFn (emulated ops) against the float64 restatement
    (oracle/restated.py::fno_forward), output and every parameter gradient."""
    import pde_policylearning_b200 as P
    import pde_policylearning_b200.ops as ops
    from oracle import restated as rs
    torch.manual_seed(5)
    x = torch.randn(2, 3, 16, 16)
    with _emulated(), _Counting(ops) as cnt:
        m = P.FNO2d(6, 6, 8, in_channels=3, out_channels=2, lifting_channels=16, projection_channels=16)
        out = m(x)
        gs = torch.autograd.grad(out.square().sum(), [p for _, p in m.named_parameters()])
    assert (cnt.n_fwd, cnt.n_bwd) == (1, 1)
    leaves = {k: v.detach().to(torch.complex128 if v.is_complex() else torch.float64).requires_grad_(True)
              for k, v in m.state_dict().items()}
    ref = rs.fno_forward(leaves, x.double(), (6, 6))
    rgs = torch.autograd.grad(ref.square().sum(), list(leaves.values()))
    rg = dict(zip(leaves.keys(), rgs))
    assert out.shape == (2, 2, 16, 16) and rel(out, ref) < 1e-6
    for (n, _), g in zip(m.named_parameters(), gs):
        r = rg[n]
        g = torch.view_as_real(g) if g.is_complex() and not r.is_complex() else g
        assert rel(g, r) < 1e-5, (n, rel(g, r))


# ------------------------------------------------------------------------------------------------------------------------
# GPU: ops
# ------------------------------------------------------------------------------------------------------------------------
OP_CASES = [(o, ci, h) for o in (2, 3, 4) for ci in (8, 16, 32, 64) for h in (128, 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32", 2e-2)])
@pytest.mark.parametrize("per_sample", [False, True], ids=["b1", "b1_per_sample"])
@pytest.mark.parametrize("act", ["gelu", "relu", "tanh"])
@pytest.mark.parametrize("case", OP_CASES, ids=lambda c: f"O{c[0]}-ci{c[1]}-h{c[2]}")
def test_multi_output_head_ops(case, act, per_sample, precision, tol):
    """out, gx, dW1, db1, dW2, db2 of mlp_head (-> MlpHeadMultiFn) and gx with the dact_z chaining of mlp_head_bwd_multi,
    against float64 autograd of the composed head; the fused kernels ran (two tensor-core launches: forward, backward pass
    over the pixel tiles).  ci = 64 with hidden = 256 exceeds the backward's shared memory: it declines, and mlp_head composes
    two pointwise convs with the same result.

    ReLU in the single-pass TF32 mode: the pre-activation carries TF32 rounding (~1e-3), so ReLU' flips for the hidden units
    whose |z1| is below it, and each flipped unit contributes its full-size gradient: gx, dW1 and db1 (the gradients through
    ReLU') measure ~2e-2 against float64 on these inputs, and are held to 5e-2 there; everything else to 2e-2."""
    import pde_policylearning_b200.functional as Fn
    from pde_policylearning_b200 import ops
    O, ci, hidden = case
    dev = _dev()
    torch.manual_seed(11)
    B, grid = 2, (16, 24)
    x = torch.randn(B, ci, *grid)
    w1 = torch.randn(hidden, ci) / ci ** 0.5
    b1 = 0.3 * torch.randn(B, hidden) if per_sample else 0.3 * torch.randn(hidden)
    w2 = torch.randn(O, hidden) / hidden ** 0.5
    b2 = torch.randn(O)
    g = torch.randn(B, O, *grid)
    dz = torch.randn(B, ci, *grid)
    ts = [t.double().requires_grad_(True) for t in (x, w1, b1, w2, b2)]
    ref = _head_ref(*ts, act)
    rgs = torch.autograd.grad(ref, ts, g.double())
    dts = [t.to(dev).requires_grad_(True) for t in (x, w1, b1, w2, b2)]
    supported = ops.mlp_head_multi_supported(dts[0], hidden, O)
    assert supported == (not (ci == 64 and hidden == 256)), "support rule changed"
    if not supported and per_sample:
        assert ops.mlp_head_bwd_multi(dts[0].detach(), dts[1].detach(), dts[2].detach(), dts[3].detach(), g.to(dev), act) is None
        return                                  # the composed path has no per-sample bias
    try:
        ops.set_precision(precision)
        n0 = ops.tensor_core_launches()
        out = Fn.mlp_head(*dts, act)
        gs = torch.autograd.grad(out, dts, g.to(dev))
        n_tc = ops.tensor_core_launches() - n0
        res = None
        if supported:
            res = ops.mlp_head_bwd_multi(dts[0].detach(), dts[1].detach(), dts[2].detach(), dts[3].detach(), g.to(dev), act,
                                         want_gz=False, dact_z=dz.to(dev), dact="gelu")
    finally:
        ops.set_precision("fp32")
    assert rel(out, ref) < tol, ("out", rel(out, ref))
    tol_dact = 5e-2 if (act == "relu" and precision == "tf32") else tol
    for name, a, b in zip(("gx", "dW1", "db1", "dW2", "db2"), gs, rgs):
        t = tol_dact if name in ("gx", "dW1", "db1") else tol
        assert a.shape == b.shape and rel(a, b) < t, (name, rel(a, b))
    if supported:
        assert n_tc >= 2, n_tc                   # forward + backward pass (+ the weight-gradient kernel when it is eligible)
        dzd = dz.double().requires_grad_(True)
        (dgelu,) = torch.autograd.grad(F.gelu(dzd).sum(), dzd)
        assert res is not None and res[1] is None and rel(res[0], rgs[0] * dgelu) < tol_dact, rel(res[0], rgs[0] * dgelu)


@pytest.mark.gpu
def test_five_outputs_decline_and_compose():
    """O = 5 is outside the fused kernels: the ops decline, having written nothing, and mlp_head composes two pointwise
    convs with the right answer."""
    import pde_policylearning_b200.functional as Fn
    from pde_policylearning_b200 import ops
    dev = _dev()
    torch.manual_seed(12)
    x, w1, b1 = torch.randn(2, 16, 16, 16), torch.randn(64, 16) / 4, torch.randn(64)
    w2, b2, g = torch.randn(5, 64) / 8, torch.randn(5), torch.randn(2, 5, 16, 16)
    xd, w1d, b1d, w2d, gd = (t.to(dev) for t in (x, w1, b1, w2, g))
    assert not ops.mlp_head_multi_supported(xd, 64, 5)
    assert not Fn.mlp_head_fused_available(xd, w1d, w2d, b1d, True)
    n0 = ops.tensor_core_launches()
    assert ops.mlp_head_fwd_multi(xd, w1d, b1d, w2d, b2.to(dev)) is None
    assert ops.mlp_head_bwd_multi(xd, w1d, b1d, w2d, gd) is None
    assert ops.tensor_core_launches() == n0
    ts = [t.double().requires_grad_(True) for t in (x, w1, b1, w2, b2)]
    ref = _head_ref(*ts, "gelu")
    rgs = torch.autograd.grad(ref, ts, g.double())
    dts = [t.to(dev).requires_grad_(True) for t in (x, w1, b1, w2, b2)]
    out = Fn.mlp_head(*dts, "gelu")
    gs = torch.autograd.grad(out, dts, gd)
    assert rel(out, ref) < 1e-5
    for a, b in zip(gs, rgs):
        assert rel(a, b) < 1e-5


# ------------------------------------------------------------------------------------------------------------------------
# GPU: models
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fullfield_fused_tail_vs_restated(golden):
    """PINObserverFullField(plane_num = 3) with the fixture a10's parameters on a 8 x 8 x 14 grid (padded to 16: 1024 pixels,
    so the fused tail runs): output, loss and every parameter gradient against float64 autograd of the restated reference
    (oracle/restated.py), in training and under no_grad."""
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops
    dev = _dev()
    c = golden("a10_pinobserver_fullfield")
    a, re = _ff_inputs(2, 8, 14, seed=21)
    ref, leaves = _restated_fullfield(c["state_dict"], a, re)
    rloss = ref.square().mean()
    rgs = dict(zip(leaves.keys(), torch.autograd.grad(rloss, list(leaves.values()))))
    m = P.PINObserverFullField(plane_num=3, **PINO_KW)
    m.load_state_dict(c["state_dict"])
    m = m.to(dev)
    with _Counting(ops) as cnt:
        out = m(a.to(dev), re.to(dev))
        loss = out.square().mean()
        gs = torch.autograd.grad(loss, [p for _, p in m.named_parameters()])
        with torch.no_grad():
            out_ng = m(a.to(dev), re.to(dev))
    assert (cnt.n_fwd, cnt.n_bwd) == (2, 1), (cnt.n_fwd, cnt.n_bwd)
    assert out.shape == (2, 3, 8, 8, 14)
    assert rel(out, ref) < 1e-5 and rel(out_ng, ref) < 1e-5, (rel(out, ref), rel(out_ng, ref))
    assert abs(loss.item() - rloss.item()) <= 2e-5 * abs(rloss.item())
    for (n, _), g in zip(m.named_parameters(), gs):
        r = rgs[n]
        g = torch.view_as_real(g) if g.is_complex() and not r.is_complex() else g
        assert rel(g, r) < 2e-4, (n, rel(g, r))


@pytest.mark.gpu
def test_fno2d_two_outputs_vs_restated():
    """FNO2d(out_channels = 2): the Projection runs the fused multi-output head; output and every parameter gradient
    against float64 autograd of the restated reference."""
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops
    from oracle import restated as rs
    dev = _dev()
    torch.manual_seed(6)
    x = torch.randn(2, 3, 32, 32)
    m = P.FNO2d(8, 8, 16, in_channels=3, out_channels=2, lifting_channels=32, projection_channels=64).to(dev)
    with _Counting(ops) as cnt:
        out = m(x.to(dev))
        gs = torch.autograd.grad(out.square().sum(), [p for _, p in m.named_parameters()])
    assert (cnt.n_fwd, cnt.n_bwd) == (1, 1)
    leaves = {k: v.detach().cpu().to(torch.complex128 if v.is_complex() else torch.float64).requires_grad_(True)
              for k, v in m.state_dict().items()}
    ref = rs.fno_forward(leaves, x.double(), (8, 8))
    rg = dict(zip(leaves.keys(), torch.autograd.grad(ref.square().sum(), list(leaves.values()))))
    assert rel(out, ref) < 1e-5, rel(out, ref)
    for (n, _), g in zip(m.named_parameters(), gs):
        r = rg[n]
        g = torch.view_as_real(g) if g.is_complex() and not r.is_complex() else g
        assert rel(g, r) < 1e-4, (n, rel(g, r))


@pytest.mark.gpu
def test_graphed_fullfield_step_matches_eager():
    """GraphedTrainStep of PINObserverFullField (fused 3-output tail inside the captured graph) follows the eager steps."""
    import pde_policylearning_b200 as P
    from pde_policylearning_b200 import ops
    dev = _dev()

    def build():
        torch.manual_seed(41)
        m = P.PINObserverFullField(plane_num=3, **PINO_KW).to(dev)
        return m, P.FusedAdam(m.parameters(), lr=1e-3)

    data = [_ff_inputs(2, 8, 14, seed=30 + i, dev=dev) for i in range(3)]
    tgts = [torch.randn(2, 3, 8, 8, 14, generator=torch.Generator().manual_seed(40 + i)).to(dev) for i in range(3)]
    loss_fn = lambda o, t: P.rel_l2_loss(o, t, size_average=False)
    m1, o1 = build()
    eager = []
    with _Counting(ops) as cnt:
        for (a, re), t in zip(data, tgts):
            o1.zero_grad()
            loss = loss_fn(m1(a, re), t)
            loss.backward()
            o1.step()
            eager.append(loss.item())
    assert cnt.n_bwd == 3
    m2, o2 = build()
    step = P.GraphedTrainStep(m2, loss_fn, o2, data[0], tgts[0])
    graphed = [step((a, re), t).item() for (a, re), t in zip(data, tgts)]
    for a, b in zip(eager, graphed):
        assert abs(a - b) < 1e-5 * abs(a), (eager, graphed)
    assert rel(o2.flat_param, o1.flat_param) < 1e-5


@pytest.mark.gpu
def test_fullfield_training_step_peak_memory():
    """One training step of PINObserverFullField at a cfg4-like size (B = 4, fc_dim 128, 64 x 64 x 65 padded to 73,
    plane_num = 3): the peak memory of the fused tail is below the composed tail's by at least one fc_dim-wide hidden
    tensor (B x 128 x 64 x 64 x 73 fp32 = 612 MB)."""
    import pde_policylearning_b200 as P
    import pde_policylearning_b200.functional as Fn
    dev = _dev()
    B, S, T = 4, 64, 65
    torch.manual_seed(50)
    m = P.PINObserverFullField(plane_num=3, modes1=[8] * 4, modes2=[8] * 4, modes3=[8] * 4, fc_dim=128, layers=[64] * 5,
                               act="gelu", pad_ratio=0.0625).to(dev)
    a = torch.randn(B, S, S, T, 4, device=dev)
    re = torch.linspace(100.0, 500.0, B, device=dev)
    hidden_bytes = B * 128 * S * S * 73 * 4

    def peak():
        m.zero_grad(set_to_none=True)
        torch.cuda.synchronize(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        loss = m(a, re).square().mean()
        loss.backward()
        torch.cuda.synchronize(dev)
        return torch.cuda.max_memory_allocated(dev) - base, loss.item()

    assert Fn.mlp_head_fused_available(torch.empty(B, 64, S, S, 73, device=dev), m.observer_head.fc1.weight,
                                       m.observer_head.fc2.weight, None, True)
    peak(), peak()                                      # plans and workspaces allocated once
    fused, loss_f = peak()
    saved = Fn.mlp_head_fused_available
    try:
        Fn.mlp_head_fused_available = lambda *a, **k: False
        peak()
        composed, loss_c = peak()
    finally:
        Fn.mlp_head_fused_available = saved
    print(f"peak memory of one step: fused {fused / 2**20:.0f} MiB, composed {composed / 2**20:.0f} MiB, "
          f"hidden tensor {hidden_bytes / 2**20:.0f} MiB")
    assert abs(loss_f - loss_c) <= 1e-5 * abs(loss_c)
    assert composed - fused >= hidden_bytes, (fused, composed, hidden_bytes)
