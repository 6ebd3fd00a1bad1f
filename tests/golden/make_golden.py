"""Generates tests/golden/*.pt from the UNMODIFIED reference (B2NO_REFERENCE_ROOT names a checkout of it).

    B2NO_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py

Each fixture stores seeded inputs, the reference module's parameters, and the reference's own outputs
and autograd gradients (fp32, CPU); the three conv fixtures (a1, a4, a6) store their seed instead of
their inputs, which tests/seeded_inputs.py replays; run this script again if that replay stops matching (a torch
upgrade that changes the CPU generator).  The reference has no golden vectors of its own (SURVEY.md 8c), so
these files ARE the pin: the oracle (oracle/closed_form.py, oracle/restated.py) and the CUDA path are
both tested against them.  Shapes follow the reference tests (neuralop/models/tests/
test_spectral_convolution.py:89-168 -- 12 per dim, channels 3/10/11, modes (4,5,2)/(4,5)/(5,)) plus small
variants of the five BASELINE configs.
"""
import os
import sys
import warnings

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
warnings.filterwarnings("ignore")

from oracle import ref_loader  # noqa: E402
import seeded_inputs  # noqa: E402

SEEDS = {"a1_neuralop_conv": 1234, "a4_rno_conv": 1235, "a6_pino_conv": 1236}


def _grads(y, inputs, gy):
    return [g.detach().clone() for g in torch.autograd.grad(y, inputs, gy)]


def conv_case(mod, x, extra=None):
    x = x.clone().requires_grad_(True)
    y = mod(x)
    gy = torch.randn_like(y)
    names = [n for n, _ in mod.named_parameters()]
    params = [p for _, p in mod.named_parameters()]
    gs = _grads(y, [x] + params, gy)
    d = dict(x=x.detach().clone(), y=y.detach().clone(), gy=gy, dx=gs[0],
             params={n: p.detach().clone() for n, p in zip(names, params)},
             grads={n: g for n, g in zip(names, gs[1:])})
    if extra:
        d.update(extra)
    return d


def model_case(mod, inputs, loss_fn=None, extra=None):
    out = mod(*inputs)
    loss = (out.square().mean() if loss_fn is None else loss_fn(out))
    names = [n for n, _ in mod.named_parameters()]
    params = [p for _, p in mod.named_parameters()]
    gs = torch.autograd.grad(loss, params)
    d = dict(inputs=[t.detach().clone() for t in inputs], out=out.detach().clone(), loss=loss.detach().clone(),
             state_dict={k: v.detach().clone() for k, v in mod.state_dict().items()},
             grads={n: g.detach().clone() for n, g in zip(names, gs)})
    if extra:
        d.update(extra)
    return d


def main():
    ref = ref_loader.load()
    out = {}

    # ---- a1: FactorizedSpectralConv (generic N-D) ------------------------------------------
    torch.manual_seed(SEEDS["a1_neuralop_conv"])
    cases = {}
    for name, (ci, co, modes, grid, norm, kw) in {
        "2d_forward": (3, 11, (4, 5), (12, 12), "forward", {}),
        "2d_backward": (3, 11, (4, 5), (12, 12), "backward", {}),
        "2d_ortho": (10, 11, (4, 5), (12, 12), "ortho", {}),
        "1d_forward": (3, 11, (5,), (12,), "forward", {}),
        "3d_forward": (3, 10, (4, 5, 2), (12, 12, 12), "forward", {}),
        "2d_overlap": (3, 4, (12, 6), (8, 12), "forward", {}),
        "2d_oddgrid": (4, 4, (6, 6), (9, 11), "forward", {}),
        "2d_scale_half": (3, 4, (8, 6), (16, 12), "forward", {"output_scaling_factor": 0.5}),
        "2d_scale_2": (3, 4, (8, 6), (16, 12), "forward", {"output_scaling_factor": 2}),
        "2d_cfg1_small": (8, 8, (16, 16), (32, 32), "forward", {}),
    }.items():
        m = ref.FactorizedSpectralConv(ci, co, modes, n_layers=1, factorization=None,
                                       implementation="factorized", fft_norm=norm, **kw)
        x = torch.randn(2, ci, *grid)
        cases[name] = conv_case(m, x, dict(n_modes=modes, fft_norm=norm, kw=kw))
    # multi-layer joint indexing: weight index = 2*layer + corner (spectral_convolution.py:337)
    m = ref.FactorizedSpectralConv(4, 4, (6, 6), n_layers=3, factorization=None,
                                   implementation="factorized", fft_norm="forward")
    x = torch.randn(2, 4, 12, 12)
    cases["2d_layer_index2"] = dict(x=x, y=m(x, 2).detach(), n_modes=(6, 6), fft_norm="forward",
                                    params={n: p.detach().clone() for n, p in m.named_parameters()})
    out["a1_neuralop_conv"] = cases

    # ---- a4: rno.SpectralConv2d -------------------------------------------------------------
    torch.manual_seed(SEEDS["a4_rno_conv"])
    cases = {}
    for name, (ci, co, m1, m2, grid) in {
        "square": (5, 6, 4, 3, (12, 12)),
        "cfg3_small": (34, 34, 6, 6, (16, 16)),
        "tall": (5, 6, 4, 3, (15, 12)),
        "short": (5, 6, 4, 3, (9, 12)),
    }.items():
        m = ref.RnoSpectralConv2d(ci, co, m1, m2)
        x = torch.randn(2, ci, *grid)
        cases[name] = conv_case(m, x, dict(modes=(m1, m2)))
    out["a4_rno_conv"] = cases

    # ---- a6: PINO SpectralConv3d ------------------------------------------------------------
    torch.manual_seed(SEEDS["a6_pino_conv"])
    cases = {}
    for name, (ci, co, ms, grid) in {
        "basic": (4, 5, (3, 2, 4), (8, 8, 9)),
        "zpad": (4, 5, (3, 2, 6), (8, 8, 9)),
        "cfg4_small": (8, 8, (4, 4, 4), (16, 16, 19)),
    }.items():
        m = ref.PinoSpectralConv3d(ci, co, *ms)
        x = torch.randn(2, ci, *grid)
        cases[name] = conv_case(m, x, dict(modes=ms))
    out["a6_pino_conv"] = cases

    # ---- a3/a9: FNO2d + observer + rel-L2 -----------------------------------------------------
    torch.manual_seed(1237)
    m = ref.FNO2d(8, 8, 16, in_channels=3, out_channels=1)
    x = torch.randn(3, 3, 24, 24)
    tgt = torch.randn(3, 1, 24, 24)
    lp = lambda o: (torch.norm((o - tgt).reshape(3, -1), 2, 1) / torch.norm(tgt.reshape(3, -1), 2, 1)).sum()
    out["a3_fno2d"] = model_case(m, [x], lp, dict(target=tgt, n_modes=(8, 8), hidden=16))
    obs = ref_loader.RefFNO2dObserver(6, 6, 8)
    p = torch.randn(2, 16, 16, 1)
    out["a9_fno2d_observer"] = model_case(obs, [p], None, dict(modes=6, width=8))
    m3 = ref.FNO3d(4, 4, 4, 6, in_channels=2, out_channels=1)
    out["a3_fno3d"] = model_case(m3, [torch.randn(2, 2, 8, 8, 10)], None, dict(n_modes=(4, 4, 4), hidden=6))

    # ---- a5: RNO2d (eval: dropout off, Q4) ----------------------------------------------------
    torch.manual_seed(1238)
    r = ref.RNO2d(4, 4, 6, 0, layer_num=1).eval()
    x = torch.randn(2, 3, 12, 12, 1)
    out["a5_rno2d_L1"] = model_case(r, [x], None, dict(modes=4, width=6, layer_num=1))
    r2 = ref.RNO2d(4, 4, 6, 1, layer_num=2).eval()
    out["a5_rno2d_L2"] = model_case(r2, [x], None, dict(modes=4, width=6, layer_num=2, recurrent_index=1))
    cell = ref.RNO_cell(6, 6, 4, 4, 6)
    xx, hh = torch.randn(2, 6, 12, 12), torch.randn(2, 6, 12, 12)
    out["a5_rno_cell"] = model_case(cell, [xx, hh], None, {})

    # ---- a7/a8: PINObserver2d + Channelflow PINO loss -----------------------------------------
    torch.manual_seed(1239)
    pm = ref.PINObserver2d(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4,
                           act="gelu", pad_ratio=0.0625)
    a = torch.randn(2, 8, 8, 17, 4)
    re = torch.tensor([100.0, 300.0])
    u = torch.randn(2, 8, 8, 17)
    forcing = ref.get_forcing(8)

    def pino_loss(o):
        data = ref.LpLoss(size_average=True)(o.reshape(2, 8, 8, 17), u)
        lic, lf = ref.Channelflow_PINO_loss(o, u[..., 0], forcing, 1 / re, 0.5)
        return 5.0 * data + lf + lic

    d = model_case(pm, [a, re], pino_loss, dict(u=u, forcing=forcing, t_interval=0.5))
    o = pm(a, re)
    lic, lf = ref.Channelflow_PINO_loss(o, u[..., 0], forcing, 1 / re, 0.5)
    d["loss_ic"], d["loss_f"] = lic.detach(), lf.detach()
    d["Du"] = ref.FDM_NS_vorticity(o.reshape(2, 8, 8, 17), 1 / re, 0.5).detach()
    out["a7_pinobserver2d"] = d

    # ---- 8f rank 4: the other consumers of the PINO trunk (pinobserver.py:276-463) ----------------
    torch.manual_seed(1240)
    ff = ref.PINObserverFullField(plane_num=3, modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4,
                                  act="gelu", pad_ratio=0.0625)
    a = torch.randn(2, 8, 8, 9, 4)
    re = torch.tensor([180.0, 420.0])
    out["a10_pinobserver_fullfield"] = model_case(ff, [a, re], None, dict(plane_num=3))
    pol = ref.PolicyModel2D(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4, act="gelu",
                            pad_ratio=0.0625)
    d0 = model_case(pol, [a, re], None, {})           # as constructed: every parameter zero (pinobserver.py:432-433)
    assert float(d0["out"].abs().max()) == 0.0
    with torch.no_grad():
        for prm in pol.parameters():                   # a trained policy: random parameters of the reference's init scale
            if prm.is_complex():
                prm.copy_(torch.view_as_complex(torch.rand(*prm.shape, 2)) / 64.0)
            else:
                prm.copy_(torch.randn_like(prm) * 0.2)
    out["a11_policy_model2d"] = model_case(pol, [a, re], None, {})

    # ---- 8f rank 4: libs/models/pino_models/fourier2d.FNO2d (basics.SpectralConv2d, two-sided padding) -----
    torch.manual_seed(1241)
    f2 = ref.PinoFNO2d(modes1=[4] * 3, modes2=[3] * 3, fc_dim=12, layers=[6, 8, 8, 5], in_dim=3, out_dim=2, act="gelu",
                       pad_ratio=[0.125, 0.0625])
    out["a12_pino_fno2d"] = model_case(f2, [torch.randn(2, 16, 12, 3)], None, dict(pad_ratio=[0.125, 0.0625]))
    f2n = ref.PinoFNO2d(modes1=[4] * 2, modes2=[3] * 2, fc_dim=8, layers=[4, 6, 4], in_dim=3, out_dim=1, act="gelu")
    out["a12_pino_fno2d_nopad"] = model_case(f2n, [torch.randn(2, 10, 14, 3)], None, {})

    only = os.environ.get("GOLDEN_ONLY")               # e.g. GOLDEN_ONLY=a10,a11: write just the new fixtures
    for k, v in out.items():
        if only and not any(k.startswith(p) for p in only.split(",")):
            continue
        path = os.path.join(HERE, k + ".pt")
        torch.save(seeded_inputs.strip(k, SEEDS[k], v) if k in SEEDS else v, path)
        print(k, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
