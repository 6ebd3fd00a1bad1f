"""CPU: the oracle (closed form + restated models) against the committed golden vectors, which were produced
by the UNMODIFIED reference (tests/golden/make_golden.py).  This is what pins the oracle where no
checkout of the reference is at hand."""
import pytest
import torch

from oracle import closed_form as cf
from oracle import restated as rs

TOL = 2e-6  # fp32 reference noise is ~1e-7; the oracle is float64


def _corners_a1(case):
    ws = sorted((k for k in case["params"] if k.startswith("weight.")), key=lambda k: int(k.split(".")[1]))
    return [case["params"][k] for k in ws], ws


A1 = ["2d_forward", "2d_backward", "2d_ortho", "1d_forward", "3d_forward", "2d_overlap", "2d_oddgrid",
      "2d_scale_half", "2d_scale_2", "2d_cfg1_small"]


@pytest.mark.parametrize("name", A1)
def test_closed_form_neuralop(golden, name):
    c = golden("a1_neuralop_conv")[name]
    x = c["x"]
    scale = c["kw"].get("output_scaling_factor")
    geom = cf.geom_neuralop(tuple(x.shape[2:]), c["n_modes"], c["fft_norm"],
                            None if scale is None else (scale,) * (x.dim() - 2))
    corners, names = _corners_a1(c)
    bias = c["params"]["bias"][0].flatten()
    y, _, _ = cf.spectral_conv_forward(geom, x, corners, bias)
    assert cf.rel_l2(y, c["y"]) < TOL
    dx, dW, db = cf.spectral_conv_backward(geom, x, corners, c["gy"], has_bias=True)
    assert cf.rel_l2(dx, c["dx"]) < TOL
    for n, g in zip(names, dW):
        assert cf.rel_l2(g, c["grads"][n]) < TOL
    assert cf.rel_l2(db, c["grads"]["bias"].flatten()) < TOL


def test_closed_form_layer_index(golden):
    c = golden("a1_neuralop_conv")["2d_layer_index2"]
    geom = cf.geom_neuralop((12, 12), c["n_modes"], c["fft_norm"])
    corners = [c["params"]["weight.4.tensor"], c["params"]["weight.5.tensor"]]
    y, _, _ = cf.spectral_conv_forward(geom, c["x"], corners, c["params"]["bias"][2].flatten())
    assert cf.rel_l2(y, c["y"]) < TOL


@pytest.mark.parametrize("name", ["square", "cfg3_small", "tall", "short"])
def test_closed_form_rno(golden, name):
    c = golden("a4_rno_conv")[name]
    x = c["x"]
    geom = cf.geom_rno(tuple(x.shape[2:]), *c["modes"])
    corners = [cf.rno_pairs_to_complex(c["params"][f"fourier_weight.{i}"]) for i in range(2)]
    y, _, _ = cf.spectral_conv_forward(geom, x, corners)
    assert cf.rel_l2(y, c["y"]) < TOL
    dx, dW, _ = cf.spectral_conv_backward(geom, x, corners, c["gy"])
    assert cf.rel_l2(dx, c["dx"]) < TOL
    for i in range(2):
        assert cf.rel_l2(torch.view_as_real(dW[i]), c["grads"][f"fourier_weight.{i}"]) < TOL


@pytest.mark.parametrize("name", ["basic", "zpad", "cfg4_small"])
def test_closed_form_pino(golden, name):
    c = golden("a6_pino_conv")[name]
    x = c["x"]
    geom = cf.geom_pino3d(tuple(x.shape[2:]), *c["modes"])
    corners = cf.pino_corners_to_canonical(*[c["params"][f"weights{k}"] for k in (1, 2, 3, 4)])
    y, _, _ = cf.spectral_conv_forward(geom, x, corners)
    assert cf.rel_l2(y, c["y"]) < TOL
    dx, dW, _ = cf.spectral_conv_backward(geom, x, corners, c["gy"])
    assert cf.rel_l2(dx, c["dx"]) < TOL
    back = {1: dW[0], 2: dW[2], 3: dW[1], 4: dW[3]}
    for k in (1, 2, 3, 4):
        assert cf.rel_l2(back[k], c["grads"][f"weights{k}"]) < TOL


def _grads(out, sd, names):
    return torch.autograd.grad(out, [sd[n] for n in names])


def test_restated_fno2d(golden):
    c = golden("a3_fno2d")
    sd = {k: v.clone().requires_grad_(True) for k, v in c["state_dict"].items()}
    x, tgt = c["inputs"][0], c["target"]
    out = rs.fno_forward(sd, x, c["n_modes"])
    assert cf.rel_l2(out, c["out"]) < 5e-6
    loss = rs.lp_rel(out, tgt, size_average=False)
    assert abs(loss.item() - c["loss"].item()) < 1e-5 * abs(c["loss"].item())
    names = list(c["grads"])
    for n, g in zip(names, _grads(loss, sd, names)):
        assert cf.rel_l2(g, c["grads"][n]) < 2e-5, n


def test_restated_observer_and_fno3d(golden):
    c = golden("a9_fno2d_observer")
    out = rs.fno2d_observer_forward(c["state_dict"], c["inputs"][0], c["modes"])
    assert cf.rel_l2(out, c["out"]) < 5e-6
    c = golden("a3_fno3d")
    out = rs.fno_forward(c["state_dict"], c["inputs"][0], c["n_modes"])
    assert cf.rel_l2(out, c["out"]) < 5e-6


@pytest.mark.parametrize("name,L,ri", [("a5_rno2d_L1", 1, 0), ("a5_rno2d_L2", 2, 1)])
def test_restated_rno2d(golden, name, L, ri):
    c = golden(name)
    out = rs.rno2d_forward(c["state_dict"], c["inputs"][0], c["modes"], c["modes"], c["width"], ri, L)
    assert cf.rel_l2(out, c["out"]) < 5e-6


def test_restated_rno_cell(golden):
    c = golden("a5_rno_cell")
    out = rs.rno_cell(c["state_dict"], "", c["inputs"][0], c["inputs"][1], 4, 4)
    assert cf.rel_l2(out, c["out"]) < 5e-6


def test_restated_pino(golden):
    c = golden("a7_pinobserver2d")
    a, re = c["inputs"]
    out = rs.pinobserver2d_forward(c["state_dict"], a, re, [3] * 3, [3] * 3, [3] * 3, [8] * 4)
    assert cf.rel_l2(out, c["out"]) < 5e-6
    lic, lf = rs.channelflow_pino_loss(out, c["u"][..., 0], rs.get_forcing(8), 1 / re, c["t_interval"])
    assert abs(lic.item() - c["loss_ic"].item()) < 1e-5 * abs(c["loss_ic"].item())
    assert abs(lf.item() - c["loss_f"].item()) < 1e-5 * abs(c["loss_f"].item())
    # same input as the reference used (the residual amplifies 1e-7 input noise through d/dt and the Laplacian)
    Du = rs.fdm_ns_vorticity(c["out"].reshape(2, 8, 8, 17), 1 / re, c["t_interval"])
    assert cf.rel_l2(Du, c["Du"]) < 5e-6


def test_restated_pino_fullfield_and_policy(golden):
    """SURVEY 8f rank 4: the other consumers of the PINO trunk (pinobserver.py:276-463), fixtures from the unmodified
    reference -- output AND every parameter gradient of the restatement."""
    for name, fwd in (("a10_pinobserver_fullfield", rs.pinobserver_fullfield_forward),
                      ("a11_policy_model2d", rs.policy_model2d_forward)):
        c = golden(name)
        a, re = c["inputs"]
        sd = {k: v.clone().requires_grad_(True) for k, v in c["state_dict"].items()}
        out = fwd(sd, a, re, [3] * 3, [3] * 3, [3] * 3, [8] * 4)
        assert out.shape == c["out"].shape
        assert cf.rel_l2(out, c["out"]) < 5e-6, name
        names = list(c["grads"].keys())
        gs = torch.autograd.grad(out.square().mean(), [sd[n] for n in names])
        for n, g in zip(names, gs):
            assert cf.rel_l2(g, c["grads"][n]) < 5e-5, (name, n)      # fp32 round-off of two op orders on 1e-9-sized gradients
    assert golden("a10_pinobserver_fullfield")["out"].shape == (2, 3, 8, 8, 9)      # planes first (pinobserver.py:360)


def test_restated_pino_fno2d(golden):
    """libs/models/pino_models/fourier2d.FNO2d (8f rank 4), with and without the two-sided zero padding."""
    for name, m1, m2, layers in (("a12_pino_fno2d", [4] * 3, [3] * 3, [6, 8, 8, 5]), ("a12_pino_fno2d_nopad", [4] * 2, [3] * 2, [4, 6, 4])):
        c = golden(name)
        sd = {k: v.clone().requires_grad_(True) for k, v in c["state_dict"].items()}
        out = rs.pino_fno2d_forward(sd, c["inputs"][0], m1, m2, layers, c.get("pad_ratio", (0.0, 0.0)))
        assert out.shape == c["out"].shape
        assert cf.rel_l2(out, c["out"]) < 5e-6, name
        names = list(c["grads"].keys())
        gs = torch.autograd.grad(out.square().mean(), [sd[n] for n in names])
        for n, g in zip(names, gs):
            assert cf.rel_l2(g, c["grads"][n]) < 5e-5, (name, n)
