"""Instance and group norm in FNO blocks, computed on the kept-mode spectrum (b2no_spec_norm_fwd / b2no_spec_norm_bwd,
functional.SpectralBlockFn / FNOStackFn with a norm, FNOBlocks(norm=...), convert_).

CPU: the spectral mean / variance / gradient identities against the float64 closed form, the host logic of the normed
blocks with emulated ops against a float64 restatement that normalises in real space (F.group_norm / F.instance_norm),
state_dict keys and convert_.  GPU: the ops against float64 autograd, FNO2d at the cfg2 shape, the per-layer route against
the stack route, and a captured training step."""
import contextlib
import itertools
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ops_emulator as emu  # noqa: E402
from oracle import closed_form as cf  # noqa: E402
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
# float64 statement of the spectral normalisation (include/b2no.h, csrc/spec_norm.cu), from the closed-form geometry
# ------------------------------------------------------------------------------------------------------------------------
def norm_table(g: cf.SpecGeom):
    """Per flat kept mode: (mirror, c) -- c = c(k_d) of the inverse; mirror = flat index of the kept mode at frequency -k
    when c == 1 and that mode is kept, else -1."""
    d = g.ndim
    rows = [g.rows(j) for j in range(d)]
    pos = [{r[0]: i for i, r in enumerate(rows[j])} for j in range(d)]
    K = g.kept()
    N, Np = g.nfft[-1], g.nout[-1]
    mirror, cs = [], []
    for idx in itertools.product(*[range(k) for k in K]):
        f = idx[-1]
        c = 2
        if f == 0 or (Np % 2 == 0 and f == Np // 2):
            c = 1
        if f >= Np // 2 + 1 or f >= N // 2 + 1:
            c = 0
        m = -1
        if c == 1:
            mi = []
            for j in range(d - 1):
                r = pos[j].get((g.nfft[j] - rows[j][idx[j]][0]) % g.nfft[j])
                if r is None:
                    break
                mi.append(r)
            else:
                m = 0
                for j in range(d - 1):
                    m = m * K[j] + mi[j]
                m = m * K[-1] + f
        mirror.append(m)
        cs.append(c)
    return torch.tensor(mirror), torch.tensor(cs, dtype=RD)


def spectral_moments(g: cf.SpecGeom, yh, bias=None):
    """(mean, var) over the output grid of s = s_i Re IDFT_trunc(yh) + bias, per (b, c), from the kept modes alone."""
    mirror, c = norm_table(g)
    si = g.scales()[1]
    B, C = yh.shape[:2]
    y = yh.reshape(B, C, -1)
    a = y + torch.where(mirror >= 0, y[..., mirror.clamp(min=0)].conj(), torch.zeros_like(y))
    S = 0.5 * si * c * a
    w = torch.where(mirror >= 0, 1.0, 2.0).to(RD)
    var = (w * S.abs().square())[..., 1:].sum(-1)
    mean = si * y[..., 0].real
    if bias is not None:
        mean = mean + bias.reshape(1, -1)
    return mean, var


def spec_norm_ref(g: cf.SpecGeom, yh, bias, gamma, beta, groups, eps):
    """The normalised spectrum of b2no_spec_norm_fwd, in float64 (differentiable)."""
    B, C = yh.shape[:2]
    si = g.scales()[1]
    mu, var = spectral_moments(g, yh, bias)
    cg = C // groups
    mu_g = mu.reshape(B, groups, cg).mean(-1)
    var_g = (var.reshape(B, groups, cg) + (mu.reshape(B, groups, cg) - mu_g[..., None]).square()).mean(-1)
    r = (var_g + eps).rsqrt().repeat_interleave(cg, dim=1)
    gam = torch.ones(C, dtype=RD) if gamma is None else gamma.to(RD)
    bet = torch.zeros(C, dtype=RD) if beta is None else beta.to(RD)
    y = yh.reshape(B, C, -1)
    dc = (gam * (mu - mu_g.repeat_interleave(cg, dim=1)) * r + bet) / si
    out = torch.cat((dc.to(CD)[..., None], (gam * r)[..., None] * y[..., 1:]), dim=-1)
    return out.reshape(yh.shape)


# ------------------------------------------------------------------------------------------------------------------------
# CPU: the identities
# ------------------------------------------------------------------------------------------------------------------------
GEOMS = [
    cf.SpecGeom(nin=(16,), half=(5,), norm="backward"),
    cf.SpecGeom(nin=(12,), half=(7,), norm="forward"),                 # kept last-dim Nyquist
    cf.SpecGeom(nin=(16, 12), half=(4, 3), norm="forward"),
    cf.SpecGeom(nin=(15, 11), half=(5, 6), norm="ortho"),              # odd grids
    cf.SpecGeom(nin=(8, 10), half=(4, 6), norm="backward"),            # h = N/2, kept Nyquist
    cf.SpecGeom(nin=(9, 8), half=(6, 5), norm="forward"),              # 2h > N, kept Nyquist
    cf.SpecGeom(nin=(8, 7, 6), half=(3, 4, 4), norm="ortho"),          # 2h > N on dim 1, kept Nyquist
    cf.SpecGeom(nin=(6, 8, 9), half=(3, 2, 3), norm="backward"),       # h = N/2
]


@pytest.mark.parametrize("g", GEOMS, ids=lambda g: f"{g.nin}-{g.half}-{g.norm}")
def test_spectral_moments_match_the_grid(g):
    """mean / variance over the grid of IDFT_trunc(yh) + bias, and the gradient of the variance, from the kept modes."""
    torch.manual_seed(0)
    B, C = 3, 4
    yh = torch.randn((B, C) + g.kept(), dtype=CD, requires_grad=True)
    bias = torch.randn(C, dtype=RD)
    si = g.scales()[1]
    s = cf.idft_trunc(g, yh, si) + bias.reshape((1, -1) + (1,) * g.ndim)
    dims = tuple(range(2, 2 + g.ndim))
    mean_g, var_g = s.mean(dims), s.var(dims, unbiased=False)
    mean, var = spectral_moments(g, yh, bias)
    assert rel(mean, mean_g) < 1e-13 and rel(var, var_g) < 1e-13
    w = torch.randn(B, C, dtype=RD)
    (ga,) = torch.autograd.grad((var_g * w).sum(), yh)
    # d var / d yh_k = 2 s_i c(k_d) S_k (k != 0), 0 at DC
    mirror, c = norm_table(g)
    y = yh.detach().reshape(B, C, -1)
    S = 0.5 * si * c * (y + torch.where(mirror >= 0, y[..., mirror.clamp(min=0)].conj(), torch.zeros_like(y)))
    gb = 2 * si * c * S * w[..., None]
    gb[..., 0] = 0
    assert rel(gb, ga.reshape(B, C, -1)) < 1e-13


@pytest.mark.parametrize("g", GEOMS[2:6], ids=lambda g: f"{g.nin}-{g.half}-{g.norm}")
@pytest.mark.parametrize("groups", [1, 2, 4])
def test_normalised_spectrum_is_group_norm_of_the_conv_output(g, groups):
    """IDFT_trunc of the normalised spectrum (no bias) equals F.group_norm of IDFT_trunc(yh) + bias."""
    torch.manual_seed(1)
    B, C = 2, 4
    yh = torch.randn((B, C) + g.kept(), dtype=CD)
    bias, gamma, beta = torch.randn(C, dtype=RD), torch.randn(C, dtype=RD), torch.randn(C, dtype=RD)
    si = g.scales()[1]
    s = cf.idft_trunc(g, yh, si) + bias.reshape((1, -1) + (1,) * g.ndim)
    out = cf.idft_trunc(g, spec_norm_ref(g, yh, bias, gamma, beta, groups, 1e-5), si)
    assert rel(out, F.group_norm(s, groups, gamma, beta, 1e-5)) < 1e-12


# ------------------------------------------------------------------------------------------------------------------------
# the emulated ops and the float64 restatement of the normed FNO
# ------------------------------------------------------------------------------------------------------------------------
def _emu_spec_norm_fwd(plan, spec, bias, gamma, beta, groups, eps):
    g = plan.cf
    d = lambda t: None if t is None else t.detach().to(RD)
    out = spec_norm_ref(g, spec.to(CD), d(bias), d(gamma), d(beta), groups, eps)
    C = spec.shape[1]
    z = torch.zeros(C, dtype=RD)
    # what the backward needs besides spec and gamma: [bias | beta | eps]
    stats = torch.cat((z if bias is None else d(bias), z if beta is None else d(beta), torch.tensor([eps], dtype=RD)))
    return out.to(torch.complex64), stats


def _emu_spec_norm_bwd(plan, spec, gspec, stats, gamma, groups, need_bias, need_affine, db_out=None):
    C = spec.shape[1]
    bias, bet, eps = stats[:C], stats[C:2 * C], float(stats[2 * C])
    affine = gamma is not None
    yh = spec.to(CD).requires_grad_(True)
    leaves = [t.detach().to(RD).clone().requires_grad_(True) for t in (bias, gamma if affine else bias, bet)]
    with torch.enable_grad():
        out = spec_norm_ref(plan.cf, yh, leaves[0], leaves[1] if affine else None, leaves[2] if affine else None,
                            groups, eps)
        gy, db, dg, dbt = torch.autograd.grad(out, [yh] + leaves, gspec.to(CD), allow_unused=True)
    f32 = lambda t: None if t is None else t.to(torch.float32)
    db = f32(db) if need_bias else None
    if db is not None and db_out is not None:
        db_out.copy_(db)
        db = db_out
    return gy.to(torch.complex64), db, f32(dg) if need_affine else None, f32(dbt) if need_affine else None


@contextlib.contextmanager
def _emulated():
    """ops_emulator.installed() plus the spectral-normalisation ops."""
    import pde_policylearning_b200.ops as ops
    names = ("spec_norm_fwd", "spec_norm_bwd")
    saved = {n: getattr(ops, n) for n in names}
    with emu.installed():
        try:
            ops.spec_norm_fwd, ops.spec_norm_bwd = _emu_spec_norm_fwd, _emu_spec_norm_bwd
            yield
        finally:
            for n, f in saved.items():
                setattr(ops, n, f)


def fno_normed_forward(sd, x, n_modes, norm, n_layers=4, fft_norm="forward", eps=1e-5):
    """oracle/restated.py::fno_forward with the block norm of fno_block.py:142-150 in real space:
    y_l = act_l(Norm_l(SpectralConv_l(x) + bias_l) + skip_l x)."""
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
        y = rs.neuralop_spectral_conv(x, corners, bias[l].reshape(-1), n_modes, fft_norm)
        if norm == "instance_norm":
            y = F.instance_norm(y, eps=eps)
        else:
            y = F.group_norm(y, 1, g(f"fno_blocks.norm.{l}.weight"), g(f"fno_blocks.norm.{l}.bias"), eps)
        x = y + skip
        if l < n_layers - l:
            x = F.gelu(x)
    x = F.gelu(conv1x1(x, g("projection.fc1.weight"), g("projection.fc1.bias")))
    return conv1x1(x, g("projection.fc2.weight"), g("projection.fc2.bias"))


def _randomise_norms(m, seed):
    """Non-trivial norm weights / biases (the constructor's are ones / zeros)."""
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if ".norm." in n:
                p.copy_(torch.randn(p.shape, generator=gen).to(p.device) * 0.5 + (1.0 if n.endswith("weight") else 0.0))


def _restated_grads(m, x, norm, n_modes, dev="cpu", weight=None):
    leaves = {k: v.detach().to(dev).to(CD if v.is_complex() else RD).requires_grad_(True) for k, v in m.state_dict().items()}
    ref = fno_normed_forward(leaves, x.detach().to(dev).double(), n_modes, norm)
    loss = ref.square().sum() if weight is None else (ref * weight.to(dev).double()).sum()
    gs = torch.autograd.grad(loss, list(leaves.values()))
    return ref, dict(zip(leaves.keys(), gs))


# ------------------------------------------------------------------------------------------------------------------------
# CPU: host logic
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("norm", ["instance_norm", "group_norm"])
@pytest.mark.parametrize("dims", [2, 3])
def test_fno_with_norm_emulated(norm, dims):
    """FNO2d / FNO3d with each norm through FNOStackFn (emulated ops) against the real-space float64 restatement: output
    and every gradient, the norm weights / biases and the conv bias included; FNOBlocks' per-layer route agrees."""
    import pde_policylearning_b200 as P
    torch.manual_seed(7)
    if dims == 2:
        n_modes, x = (6, 6), torch.randn(2, 3, 12, 10)
        m = P.FNO2d(6, 6, 8, in_channels=3, out_channels=1, lifting_channels=16, projection_channels=16, norm=norm)
    else:
        n_modes, x = (4, 4, 4), torch.randn(2, 3, 6, 8, 7)
        m = P.FNO3d(4, 4, 4, 6, in_channels=3, out_channels=1, lifting_channels=8, projection_channels=8, norm=norm)
    _randomise_norms(m, 3)
    params = [p for _, p in m.named_parameters()]
    with _emulated():
        out = m(x)
        gs = torch.autograd.grad(out.square().sum(), params)
        h = m.lifting(x)
        for l in range(m.n_layers):
            h = m.fno_blocks(h, l)
        out_l = m.projection(h)
        gs_l = torch.autograd.grad(out_l.square().sum(), params)
    ref, rg = _restated_grads(m, x, norm, n_modes)
    assert rel(out, ref) < 1e-6 and rel(out_l, ref) < 1e-6
    names = [n for n, _ in m.named_parameters()]
    if norm == "group_norm":
        assert any(".norm." in n for n in names)
    for n, g, gl in zip(names, gs, gs_l):
        if n == "fno_blocks.convs.bias" and norm == "instance_norm":
            # the bias cancels in the instance statistics: its gradient is zero (to rounding in the restatement)
            assert rg[n].abs().max() < 1e-10 and g.abs().max() < 1e-6 and gl.abs().max() < 1e-6
            continue
        assert rel(g, rg[n]) < 1e-5, (n, rel(g, rg[n]))
        assert rel(gl, rg[n]) < 1e-5, (n, rel(gl, rg[n]))


def test_state_dict_keys():
    import pde_policylearning_b200 as P
    for norm, extra in ((None, []), ("instance_norm", []),
                        ("group_norm", [f"fno_blocks.norm.{l}.{k}" for l in range(4) for k in ("weight", "bias")])):
        keys = set(P.FNO2d(6, 6, 8, norm=norm).state_dict())
        base = set(P.FNO2d(6, 6, 8).state_dict())
        assert keys == base | set(extra), norm
    b = P.FNOBlocks(8, 8, (4, 4), n_layers=2, norm="instance_norm")
    assert isinstance(b.norm[1], torch.nn.InstanceNorm2d) and not b.norm[1].affine and not b.norm[1].track_running_stats
    b = P.FNOBlocks(8, 8, (4, 4, 4), n_layers=2, norm="group_norm")
    assert isinstance(b.norm[0], torch.nn.GroupNorm) and b.norm[0].num_groups == 1 and b.norm[0].affine
    with pytest.raises(NotImplementedError):
        P.FNO2d(6, 6, 8, norm="ada_in")
    with pytest.raises(ValueError):
        P.FNO2d(6, 6, 8, norm="batch_norm")


def _as_reference_blocks(blocks, norm_modules):
    """A stand-in of the reference's FNOBlocks: the reference's class name, outside this package, with its norm list."""
    cls = type("FNOBlocks", (type(blocks),), {"__module__": "reference_stand_in", "preactivation": False})
    blocks.__class__ = cls
    blocks.norm = norm_modules
    return blocks


@pytest.mark.parametrize("kind", ["instance", "instance_affine", "group", "group2", "batch", "instance_running"])
def test_convert_reuses_norm_modules(kind):
    """convert_ swaps a reference FNOBlocks with instance / group norms for the native block, re-using the same norm
    modules (state_dict keys and Parameters unchanged); other norms leave the block in torch."""
    import pde_policylearning_b200 as P
    nn = torch.nn
    C = 8
    make = {"instance": lambda: nn.InstanceNorm2d(C), "instance_affine": lambda: nn.InstanceNorm2d(C, affine=True),
            "group": lambda: nn.GroupNorm(1, C), "group2": lambda: nn.GroupNorm(4, C), "batch": lambda: nn.BatchNorm2d(C),
            "instance_running": lambda: nn.InstanceNorm2d(C, track_running_stats=True)}[kind]
    m = P.FNO2d(4, 4, C, n_layers=2)
    norms = nn.ModuleList([make() for _ in range(2)])
    _as_reference_blocks(m.fno_blocks, norms)
    keys, before = list(m.state_dict().keys()), dict(m.named_parameters())
    c = P.convert_(m)
    assert list(c.state_dict().keys()) == keys
    assert all(p is before[k] for k, p in c.named_parameters())
    native = type(c.fno_blocks).__module__.startswith("pde_policylearning_b200")
    assert native == (kind not in ("batch", "instance_running"))
    if native:
        assert c.fno_blocks.norm is norms


@pytest.mark.skipif(not ref_loader.available(), reason="B2NO_REFERENCE_ROOT does not name a checkout of the reference")
@pytest.mark.parametrize("norm", ["instance_norm", "group_norm"])
def test_reference_fno2d_with_norm(norm):
    """The unmodified reference FNO2d(norm=...) against the real-space restatement, and convert_ re-using its norms; with the
    emulated ops the converted model reproduces the reference."""
    import pde_policylearning_b200 as P
    ref = ref_loader.load()
    torch.manual_seed(11)
    r = ref.FNO2d(6, 6, 8, in_channels=3, out_channels=1, lifting_channels=16, projection_channels=16, norm=norm)
    _randomise_norms(r, 5)
    x = torch.randn(2, 3, 12, 12)
    with torch.no_grad():
        y_ref = r(x)
    sd = {k: v.detach().to(CD if v.is_complex() else RD) for k, v in r.state_dict().items()}
    assert rel(y_ref, fno_normed_forward(sd, x.double(), (6, 6), norm)) < 1e-5
    norms = r.fno_blocks.norm
    c = P.convert_(r)
    assert type(c.fno_blocks).__module__.startswith("pde_policylearning_b200") and c.fno_blocks.norm is norms
    with _emulated(), torch.no_grad():
        assert rel(c(x), y_ref) < 1e-5


# ------------------------------------------------------------------------------------------------------------------------
# GPU: the ops
# ------------------------------------------------------------------------------------------------------------------------
OP_CASES = [
    # (nin, n_modes of the neuralop conv, fft_norm, B, C)
    ((128, 128), (12, 12), "forward", 64, 32),          # cfg2: 64 x 32 x 72 modes
    ((16,), (10,), "backward", 5, 6),
    ((15, 11), (10, 12), "ortho", 3, 12),
    ((32, 32, 32), (32, 32, 32), "forward", 4, 64),     # FNO3d: K = 32 * 32 * 16 = 16384 (every row kept)
    ((24, 20, 16), (16, 16, 16), "backward", 1, 16),    # K = 16 * 16 * 8 = 2048
]


@pytest.mark.gpu
@pytest.mark.parametrize("affine", [False, True], ids=["plain", "affine"])
@pytest.mark.parametrize("gsel", ["1", "C", "div"])
@pytest.mark.parametrize("case", OP_CASES, ids=lambda c: f"{c[0]}-B{c[3]}-C{c[4]}")
def test_spec_norm_ops(case, gsel, affine):
    """spec_norm_fwd / spec_norm_bwd against float64 autograd of the spectral statement: the normalised spectrum, gYh, the
    conv-bias gradient and the norm weight / bias gradients."""
    from pde_policylearning_b200 import ops
    dev = _dev()
    nin, n_modes, fft_norm, B, C = case
    groups = {"1": 1, "C": C, "div": 2 if C % 4 else 4}[gsel]
    g = cf.geom_neuralop(nin, n_modes, fft_norm)
    plan = ops.get_plan(ops.SpecGeom(g.nin, g.half, g.norm), dev)
    gen = torch.Generator().manual_seed(B * 1000 + C + groups)
    yh = torch.randn((B, C) + g.kept(), dtype=CD, generator=gen)
    # a realistic spectrum: a DC term comparable to the fluctuation
    yh.reshape(B, C, -1)[..., 0] *= 3.0 * math.sqrt(plan.modes)
    bias = torch.randn(C, dtype=RD, generator=gen)
    gamma = torch.randn(C, dtype=RD, generator=gen) * 0.5 + 1 if affine else None
    beta = torch.randn(C, dtype=RD, generator=gen) if affine else None
    gout = torch.randn((B, C) + g.kept(), dtype=CD, generator=gen)
    leaves = [t.clone().requires_grad_(True) for t in (yh, bias)] + \
        ([gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)] if affine else [])
    ref = spec_norm_ref(g, leaves[0], leaves[1], leaves[2] if affine else None, leaves[3] if affine else None, groups, 1e-5)
    rg = torch.autograd.grad(ref, leaves, gout)
    f32 = lambda t: None if t is None else t.to(torch.float32).to(dev).contiguous()
    c64 = lambda t: t.to(torch.complex64).to(dev).contiguous()
    out, stats = ops.spec_norm_fwd(plan, c64(yh), f32(bias), f32(gamma), f32(beta), groups, 1e-5)
    # the DC imaginary part is not read by the inverse transform: compare what the output grid sees
    outr, refr = out.cpu().to(CD).reshape(B, C, -1), ref.detach().reshape(B, C, -1)
    assert rel(outr[..., 1:], refr[..., 1:]) < 1e-5
    assert rel(outr[..., 0].real, refr[..., 0].real) < 1e-5
    gy, db, dgam, dbet = ops.spec_norm_bwd(plan, c64(yh), c64(gout), stats, f32(gamma), groups, True, affine)
    assert rel(gy, rg[0]) < 1e-5, rel(gy, rg[0])
    if groups == C:
        assert db.abs().max().item() <= 1e-6 * max(1.0, rg[0].abs().max().item())
    else:
        assert rel(db, rg[1]) < 1e-5, rel(db, rg[1])
    if affine:
        assert rel(dgam, rg[2]) < 1e-5 and rel(dbet, rg[3]) < 1e-5


@pytest.mark.gpu
def test_spec_norm_declines_mode_major_plans():
    from pde_policylearning_b200 import ops
    dev = _dev()
    plan = ops.get_plan(ops.SpecGeom((64, 64), (6, 6), "forward", layout=1), dev)
    spec = torch.zeros(plan.spec_shape(2, 4), dtype=torch.complex64, device=dev)
    with pytest.raises(RuntimeError, match="unsupported"):
        ops.spec_norm_fwd(plan, spec, None, None, None, 1, 1e-5)


# ------------------------------------------------------------------------------------------------------------------------
# GPU: models
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("norm", ["instance_norm", "group_norm"])
def test_fno2d_cfg2_with_norm(norm):
    """FNO2d(12, 12, 32, norm=...) at the cfg2 shape (batch 64, 128 x 128) against the real-space float64 restatement (run on
    the GPU in float64): output and every gradient; the per-layer route (FNOBlocks(x, i)) agrees with the stack route."""
    import pde_policylearning_b200 as P
    dev = _dev()
    torch.manual_seed(21)
    m = P.FNO2d(12, 12, 32, in_channels=3, out_channels=1, norm=norm)
    _randomise_norms(m, 9)
    m = m.to(dev)
    x = torch.randn(64, 3, 128, 128, device=dev)
    w = torch.randn(64, 1, 128, 128, device=dev)
    params = [p for _, p in m.named_parameters()]
    out = m(x)
    gs = torch.autograd.grad((out * w).sum(), params)
    h = m.lifting(x)
    for l in range(m.n_layers):
        h = m.fno_blocks(h, l)
    out_l = m.projection(h)
    gs_l = torch.autograd.grad((out_l * w).sum(), params)
    ref, rg = _restated_grads(m, x, norm, (12, 12), dev=dev, weight=w)
    assert rel(out, ref) < 5e-5 and rel(out_l, out) < 1e-5
    for (n, _), g, gl in zip(m.named_parameters(), gs, gs_l):
        r = rg[n]
        if n == "fno_blocks.convs.bias" and norm == "instance_norm":
            assert g.abs().max().item() <= 1e-6 and gl.abs().max().item() <= 1e-6, n
            continue
        assert rel(g, r) < 5e-5, (n, rel(g, r))
        assert rel(gl, g) < 5e-5, (n, rel(gl, g))


@pytest.mark.gpu
def test_graphed_train_step_with_norm_matches_eager():
    """GraphedTrainStep of an FNO2d with group norm follows the same trajectory as the eager step."""
    import pde_policylearning_b200 as P
    dev = _dev()

    def build():
        torch.manual_seed(31)
        m = P.FNO2d(6, 6, 16, in_channels=3, out_channels=1, norm="group_norm")
        _randomise_norms(m, 4)
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
