"""CPU, only where B2NO_REFERENCE_ROOT names a checkout of the reference: the oracle against the UNMODIFIED reference
on freshly seeded inputs -- the direct pin.  tests/test_oracle_golden.py makes the same kind of check through committed
fixtures, on other cases: the shapes below (the (16, 12) and (9, 14) grids, the 3-D (8, 6, 10) grid, the restated models at
these sizes, the residual at n = 16) are compared with the reference only here."""
import pytest
import torch

from oracle import closed_form as cf
from oracle import ref_loader
from oracle import restated as rs

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason="B2NO_REFERENCE_ROOT does not name a checkout of the reference")

TOL = 2e-6


@pytest.fixture(scope="module")
def ref():
    return ref_loader.load()


@pytest.mark.parametrize("ci,co,modes,grid,norm", [(3, 5, (6, 4), (16, 12), "forward"), (4, 4, (8, 8), (16, 16), "backward"),
                                                   (2, 3, (4, 6), (9, 14), "ortho"), (2, 2, (4, 4, 4), (8, 6, 10), "forward")])
def test_closed_form_vs_reference_neuralop_conv(ref, ci, co, modes, grid, norm):
    """spectral_convolution.py:303-347 (the class FNOBlocks builds) on random inputs: y, dx, dW, dbias."""
    torch.manual_seed(7)
    m = ref.FactorizedSpectralConv(ci, co, modes, n_layers=1, factorization=None, implementation="factorized", fft_norm=norm)
    x = torch.randn(2, ci, *grid, requires_grad=True)
    gy = torch.randn(2, co, *grid)
    y = m(x)
    params = dict(m.named_parameters())
    wn = sorted((k for k in params if k.startswith("weight.")), key=lambda k: int(k.split(".")[1]))
    gs = torch.autograd.grad(y, [x, params["bias"]] + [params[k] for k in wn], gy)
    geom = cf.geom_neuralop(grid, modes, norm)
    corners = [ref_loader_complex(params[k]) for k in wn]
    y64, _, _ = cf.spectral_conv_forward(geom, x.detach(), corners, params["bias"].detach()[0].flatten())
    assert cf.rel_l2(y64, y) < TOL
    dx, dW, db = cf.spectral_conv_backward(geom, x.detach(), corners, gy, has_bias=True)
    assert cf.rel_l2(dx, gs[0]) < TOL
    assert cf.rel_l2(db, gs[1].flatten()) < TOL
    for g64, g in zip(dW, gs[2:]):
        assert cf.rel_l2(g64, ref_loader_complex(g)) < TOL


def ref_loader_complex(t):
    t = t.detach()
    return t if t.is_complex() else torch.view_as_complex(t.contiguous())


def test_closed_form_vs_reference_rno_and_pino_conv(ref):
    """rno.py:60-77 and basics.py:114-143 on random inputs."""
    torch.manual_seed(8)
    m = ref.RnoSpectralConv2d(3, 4, 5, 3)
    x = torch.randn(2, 3, 12, 12, requires_grad=True)
    gy = torch.randn(2, 4, 12, 12)
    y = m(x)
    gs = torch.autograd.grad(y, [x] + list(m.parameters()), gy)
    geom = cf.geom_rno((12, 12), 5, 3)
    corners = [cf.rno_pairs_to_complex(p.detach()) for p in m.parameters()]
    y64, _, _ = cf.spectral_conv_forward(geom, x.detach(), corners)
    dx, dW, _ = cf.spectral_conv_backward(geom, x.detach(), corners, gy)
    assert cf.rel_l2(y64, y) < TOL and cf.rel_l2(dx, gs[0]) < TOL
    for g64, g in zip(dW, gs[1:]):
        assert cf.rel_l2(torch.view_as_real(g64), g) < TOL
    p3 = ref.PinoSpectralConv3d(2, 3, 3, 2, 3)
    x3 = torch.randn(2, 2, 8, 6, 9, requires_grad=True)
    y3 = p3(x3)
    gy3 = torch.randn_like(y3)
    g3 = torch.autograd.grad(y3, [x3, p3.weights1, p3.weights2, p3.weights3, p3.weights4], gy3)
    geom3 = cf.geom_pino3d((8, 6, 9), 3, 2, 3)
    c3 = cf.pino_corners_to_canonical(*[w.detach() for w in (p3.weights1, p3.weights2, p3.weights3, p3.weights4)])
    y64, _, _ = cf.spectral_conv_forward(geom3, x3.detach(), c3)
    dx3, _, _ = cf.spectral_conv_backward(geom3, x3.detach(), c3, gy3)
    assert cf.rel_l2(y64, y3) < TOL and cf.rel_l2(dx3, g3[0]) < TOL


def test_restated_models_vs_reference(ref):
    """The model-level restatements (the CPU 'port' bench.py times on the GPU box) on random inputs."""
    torch.manual_seed(9)
    obs = ref_loader.RefFNO2dObserver(6, 6, 8)
    p = torch.randn(2, 16, 16, 1)
    sd = {k: v.detach() for k, v in obs.state_dict().items()}
    assert cf.rel_l2(rs.fno2d_observer_forward(sd, p, 6), obs(p)) < 5e-6
    r = ref.RNO2d(4, 4, 6, 0, layer_num=1).eval()
    x = torch.randn(2, 3, 12, 12, 1)
    assert cf.rel_l2(rs.rno2d_forward({k: v.detach() for k, v in r.state_dict().items()}, x, 4, 4, 6), r(x)) < 5e-6
    pm = ref.PINObserver2d(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4, act="gelu", pad_ratio=0.0625)
    a, re = torch.randn(2, 8, 8, 9, 4), torch.tensor([150.0, 450.0])
    out = pm(a, re)
    assert cf.rel_l2(rs.pinobserver2d_forward({k: v.detach() for k, v in pm.state_dict().items()}, a, re, [3] * 3, [3] * 3, [3] * 3, [8] * 4), out) < 5e-6


def test_pino_residual_vs_reference(ref):
    """diff_control_env.py:5-60 against the restatement AND the product's DFT-matrix form (pino_loss.py, pure torch ops)."""
    import pde_policylearning_b200 as P
    torch.manual_seed(10)
    w = torch.randn(2, 16, 16, 7)
    v = 1.0 / torch.tensor([120.0, 380.0])
    du = ref.FDM_NS_vorticity(w, v, 0.5)
    assert cf.rel_l2(rs.fdm_ns_vorticity(w, v, 0.5), du) < 5e-6
    assert cf.rel_l2(P.fdm_ns_vorticity(w, v, 0.5), du) < 5e-6
    assert torch.equal(P.get_forcing(16), ref.get_forcing(16))
    lic, lf = ref.Channelflow_PINO_loss(w.unsqueeze(-1), w[..., 0] * 0.9, ref.get_forcing(16), v, 0.5)
    lic2, lf2 = rs.channelflow_pino_loss(w.unsqueeze(-1), w[..., 0] * 0.9, rs.get_forcing(16), v, 0.5)
    assert abs(lic.item() - lic2.item()) < 1e-5 * abs(lic.item()) and abs(lf.item() - lf2.item()) < 1e-5 * abs(lf.item())
