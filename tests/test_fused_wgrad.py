"""The dx pass of a 2-D FNO layer with the 1x1 weight gradient computed in the same pass (b2no_dft_inverse_wgrad,
k_pw_tc<MODE, true>): dW and db against float64, dx against the two-launch path, the fall-back for shapes the fused pass
does not take, and (on the CPU, with the emulated ops) the host routing of FNOStackFn against the reference fixture."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ops_emulator as emu  # noqa: E402


def rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    den = torch.linalg.vector_norm(b).item()
    return torch.linalg.vector_norm(a - b).item() / (den if den > 0 else 1.0)


# grid, half, B, co (gradient channels), ci (input / dx channels)
CASES = [((128, 128), (12, 12), 2, 32, 32), ((64, 64), (8, 8), 2, 32, 32), ((64, 64), (6, 6), 3, 20, 20),
         ((64, 64), (8, 8), 2, 34, 34), ((64, 64), (8, 8), 2, 20, 34)]


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32", 2e-2)])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "x".join(map(str, c[0])) + f"-co{c[3]}-ci{c[4]}")
def test_fused_dx_pass_weight_gradient(case, precision, tol):
    from pde_policylearning_b200 import ops
    grid, half, B, co, ci = case
    dev = torch.device("cuda", 0)
    torch.manual_seed(3)
    plan = ops.get_plan(ops.SpecGeom(nin=grid, half=half, norm="forward"), dev)
    gxh = torch.randn(plan.spec_shape(B, ci), dtype=torch.cfloat, device=dev)
    g = torch.randn(B, co, *grid, device=dev)
    x = torch.randn(B, ci, *grid, device=dev) + 0.5
    w = torch.randn(co, ci, device=dev)
    dw64 = torch.einsum("bo...,bi...->oi", g.double(), x.double())
    db64 = g.double().sum(dim=[0, 2, 3])
    epi = ops.make_epilogue(pw_w=w, pw_x=g, pw_transposed=True)
    try:
        ops.set_precision(precision)
        n0 = ops.tensor_core_launches()
        r = ops.dft_inverse_wgrad(plan, 1, gxh, epi, x, need_bias=True)
        assert r is not None, "fused pass declined an eligible shape"
        assert ops.tensor_core_launches() - n0 == 1
        y, dw, db = r
        n0 = ops.tensor_core_launches()
        y_ref = ops.dft_inverse(plan, 1, gxh, epi)
        dw_ref, db_ref = ops.pw_wgrad(g, x, need_bias=True)
        assert ops.tensor_core_launches() - n0 == 2
    finally:
        ops.set_precision("fp32")
    assert rel(y, y_ref) < 1e-6, rel(y, y_ref)
    assert rel(dw, dw64) < tol and rel(db, db64) < tol, (rel(dw, dw64), rel(db, db64))
    assert rel(dw, dw_ref) < tol and rel(db, db_ref) < tol


@pytest.mark.gpu
def test_fused_pass_declines_ineligible_shapes():
    """More than 64 gradient channels, a 3-D plan, the dx pass that multiplies by GELU'(z): nothing is computed and the
    caller keeps the two launches."""
    from pde_policylearning_b200 import ops
    dev = torch.device("cuda", 0)
    torch.manual_seed(4)
    for grid, half, co, ci, dact in (((64, 64), (8, 8), 72, 32, None), ((16, 16, 8), (4, 4, 3), 8, 8, None),
                                     ((64, 64), (8, 8), 32, 32, "gelu")):
        plan = ops.get_plan(ops.SpecGeom(nin=grid, half=half), dev)
        gxh = torch.randn(plan.spec_shape(2, ci), dtype=torch.cfloat, device=dev)
        g = torch.randn(2, co, *grid, device=dev)
        x = torch.randn(2, ci, *grid, device=dev)
        dz = torch.randn(2, ci, *grid, device=dev) if dact else None
        epi = ops.make_epilogue(pw_w=torch.randn(co, ci, device=dev), pw_x=g, pw_transposed=True, dact_z=dz, dact=dact)
        n0 = ops.tensor_core_launches()
        assert ops.dft_inverse_wgrad(plan, 1, gxh, epi, x, need_bias=True) is None
        assert ops.tensor_core_launches() == n0


def _stack_grads(width, fused, B=2, grid=(64, 64), modes=(8, 8), layers=3):
    assert layers == 3
    import pde_policylearning_b200.functional as Fn
    from pde_policylearning_b200 import ops
    dev = torch.device("cuda", 0)
    torch.manual_seed(7)
    geom = ops.SpecGeom(nin=grid, half=modes)
    x = torch.randn(B, width, *grid, device=dev, requires_grad=True)
    bias = (0.1 * torch.randn(layers, width, 1, 1, device=dev)).requires_grad_(True)
    params = []
    for _ in range(layers):
        pw = (torch.randn(width, width, 1, 1, device=dev) / width ** 0.5).requires_grad_(True)
        corners = [(0.05 * torch.randn(width, width, *modes, dtype=torch.cfloat, device=dev)).requires_grad_(True)
                   for _ in range(2)]
        params.append((pw, corners))
    acts = ["gelu", None, None]        # dx passes: layer 2 and layer 0 without GELU'(z) (fused), layer 1 with it
    saved = Fn._fused_wgrad_ok
    try:
        if not fused:
            Fn._fused_wgrad_ok = lambda g: False
        y = Fn.fno_stack(x, geom, bias, params, acts)
        n0 = ops.tensor_core_launches()
        leaves = [x, bias] + [t for pw, cs in params for t in [pw] + cs]
        grads = torch.autograd.grad(y.square().sum(), leaves)
        return grads, ops.tensor_core_launches() - n0
    finally:
        Fn._fused_wgrad_ok = saved


@pytest.mark.gpu
@pytest.mark.parametrize("width,eligible", [(32, True), (72, False)])
def test_fno_stack_backward_uses_the_fused_pass(width, eligible):
    """FNOStackFn: the same gradients with and without the fused pass; one tensor-core launch fewer per fused dx pass
    (two of the three) when the width is eligible, the same launches when it is not."""
    g_fused, n_fused = _stack_grads(width, True)
    g_ref, n_ref = _stack_grads(width, False)
    for a, b in zip(g_fused, g_ref):
        assert rel(a, b) < 1e-5, rel(a, b)
    assert n_ref - n_fused == (2 if eligible else 0), (n_ref, n_fused)


def test_fno_stack_routing_with_emulated_ops(golden):
    """Host logic: FNOStackFn's fused branch (dx, dWp and dbias[l] from one call) against the reference fixture, with
    every op replaced by its float64 definition."""
    import pde_policylearning_b200 as P
    import pde_policylearning_b200.functional as Fn
    import pde_policylearning_b200.ops as ops
    calls = []

    def dft_inverse_wgrad(plan, which, spec, epi, x, need_bias, db_out=None):
        calls.append(x.shape)
        y = emu.dft_inverse(plan, which, spec, epi)
        dw, db = emu.pw_wgrad(epi["pw_x"], x, need_bias, db_out)
        return y, dw, db

    c = golden("a3_fno2d")
    saved, saved_op = Fn._fused_wgrad_ok, ops.dft_inverse_wgrad
    with emu.installed():
        try:
            Fn._fused_wgrad_ok = lambda g: True
            ops.dft_inverse_wgrad = dft_inverse_wgrad
            mod = P.FNO2d(8, 8, 16, in_channels=3, out_channels=1)
            mod.load_state_dict(c["state_dict"])
            out = mod(*c["inputs"])
            assert rel(out, c["out"]) < 2e-5
            loss = P.rel_l2_loss(out, c["target"], size_average=False)
            names = [n for n, _ in mod.named_parameters()]
            gs = torch.autograd.grad(loss, [p for _, p in mod.named_parameters()])
        finally:
            Fn._fused_wgrad_ok = saved
            ops.dft_inverse_wgrad = saved_op
    assert len(calls) > 0
    for n, g in zip(names, gs):
        assert rel(g, c["grads"][n]) < 1e-4, (n, rel(g, c["grads"][n]))
