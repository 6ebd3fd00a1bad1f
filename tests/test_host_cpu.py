"""CPU: host-side logic, the C ABI surface, state_dict / drop-in contracts.  No compute calls, except the one bench.py test marked gpu."""
import ctypes
import os
import re

import pytest
import torch

from oracle import ref_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import subprocess
    from pde_policylearning_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    hdr = open(os.path.join(ROOT, "include", "b2no.h")).read()
    declared = set(re.findall(r"\b(b2no_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 19
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/b2no.h but not exported"
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
    defined = set(re.findall(r"\b(b2no_[a-z0-9_]+)$", nm, re.M))
    assert defined == declared, f"exported, not declared in include/b2no.h: {sorted(defined - declared)}"
    assert set(_lib.EXPORTS) == declared
    assert _lib.lib().b2no_version() == 5
    assert b"bad argument" in _lib.lib().b2no_error_string(-1)


def test_no_cpu_fallback():
    import pde_policylearning_b200 as P
    m = P.SpectralConv(3, 3, (4, 4), factorization=None, implementation="factorized")
    with pytest.raises(RuntimeError, match="no CPU fallback|only on CUDA"):
        m(torch.randn(1, 3, 8, 8))
    with pytest.raises(RuntimeError):
        P.pointwise_conv(torch.randn(1, 3, 8, 8), torch.randn(4, 3), None, None)
    with pytest.raises(RuntimeError):
        P.rel_l2_loss(torch.randn(2, 5), torch.randn(2, 5))


def test_unsupported_options_raise():
    import pde_policylearning_b200 as P
    with pytest.raises(NotImplementedError):
        P.SpectralConv(3, 3, (4, 4), factorization="cp")
    with pytest.raises(NotImplementedError):
        P.SpectralConv(3, 3, (4, 4), factorization=None, separable=True)
    with pytest.raises(ValueError):
        P.SpectralConv(3, 3, (4, 4), factorization=None, implementation="bogus")
    with pytest.raises(NotImplementedError):
        P.FNO((4, 4), 8, use_mlp=True)
    with pytest.raises(ValueError):
        P.SpectralConv(3, 3, (4, 4), factorization=None, incremental_n_modes=(2, 2, 2))


def test_state_dict_layout_matches_golden(golden):
    """Parameter names / shapes / dtypes are the reference's (SURVEY.md 8a.4)."""
    import pde_policylearning_b200 as P
    pairs = [
        (P.FNO2d(8, 8, 16, in_channels=3, out_channels=1), golden("a3_fno2d")["state_dict"]),
        (P.FNO3d(4, 4, 4, 6, in_channels=2, out_channels=1), golden("a3_fno3d")["state_dict"]),
        (P.FNO2dObserver(6, 6, 8), golden("a9_fno2d_observer")["state_dict"]),
        (P.RNO2d(4, 4, 6, 0, layer_num=1), golden("a5_rno2d_L1")["state_dict"]),
        (P.RNO2d(4, 4, 6, 1, layer_num=2), golden("a5_rno2d_L2")["state_dict"]),
        (P.RNO_cell(6, 6, 4, 4, 6), golden("a5_rno_cell")["state_dict"]),
        (P.PINObserver2d(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4, act="gelu",
                         pad_ratio=0.0625), golden("a7_pinobserver2d")["state_dict"]),
    ]
    for mod, sd in pairs:
        mine = {k: (tuple(v.shape), v.dtype) for k, v in mod.state_dict().items()}
        ref = {k: (tuple(v.shape), v.dtype) for k, v in sd.items()}
        assert mine == ref
        mod.load_state_dict(sd)


def test_real_view_checkpoint_loads():
    """tltorch >= 0.4 stores ComplexDense weights as a real view (..., 2): accept both (SURVEY 8a.4)."""
    import pde_policylearning_b200 as P
    m = P.SpectralConv(3, 4, (4, 4), factorization=None, implementation="factorized")
    sd = {k: (torch.view_as_real(v).clone() if v.is_complex() else v.clone()) for k, v in m.state_dict().items()}
    m2 = P.SpectralConv(3, 4, (4, 4), factorization=None, implementation="factorized")
    m2.load_state_dict(sd)
    assert torch.equal(m2.weight[0].tensor, m.weight[0].tensor)


def test_incremental_modes_and_quirks():
    import pde_policylearning_b200 as P
    m = P.SpectralConv(3, 4, (8, 6), factorization=None, implementation="factorized", n_layers=2)
    assert m.half_n_modes == [4, 3] and m.n_weights_per_layer == 2 and len(m.weight) == 4
    m.incremental_n_modes = (4, 4)
    assert m.half_n_modes == [2, 2]
    assert tuple(m._get_weight(1).shape) == (3, 4, 2, 2)
    blocks = P.FNOBlocks(8, 8, (4, 4), n_layers=4)
    # quirk Q1: activation iff index < n_layers - index  -> layers 0, 1 only
    assert [i < (blocks.n_layers - i) for i in range(4)] == [True, True, False, False]
    f = P.FNO2d(4, 4, 8, skip="soft-gating")    # quirk Q2: `skip=` is swallowed, skips stay linear
    assert isinstance(f.fno_blocks.fno_skips[0], torch.nn.Conv2d) and f.fno_blocks.fno_skips[0].bias is None
    r = P.RNO2d(3, 5, 6, 0, layer_num=1)
    assert r.modes1 == 5                         # quirk Q4
    assert r.regressor.spectral_conv[0].dropout.p == 0.3


def test_geometry_matches_oracle():
    from oracle import closed_form as cf
    from pde_policylearning_b200.ops import SpecGeom
    for nin, half, norm, nfft, nout in (((16, 12), (4, 3), "forward", None, None),
                                        ((15, 12), (4, 3), "ortho", (12, 12), (12, 12)),
                                        ((16, 12), (4, 3), "backward", None, (32, 24))):
        a = SpecGeom(nin, half, norm, nfft, nout).resolved()
        b = cf.SpecGeom(nin=nin, half=half, norm=norm, nfft=nfft, nout=nout)
        assert a.nfft == b.nfft and a.nout == b.nout
        assert a.scales() == pytest.approx(b.scales())


@pytest.mark.skipif(not ref_loader.available(), reason="B2NO_REFERENCE_ROOT does not name a checkout of the reference")
def test_convert_shares_parameters_with_reference_modules():
    import pde_policylearning_b200 as P
    ref = ref_loader.load()
    pino_kw = dict(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4, act="gelu", pad_ratio=0.0625)
    for build in (lambda: ref.FNO2d(12, 12, 32, in_channels=3, out_channels=1),
                  lambda: ref.RNO2d(12, 12, 34, 0, layer_num=1),
                  lambda: ref.PINObserver2d(**pino_kw),
                  # the other consumers of the PINO conv (pinobserver.py:276-463) are reached through convert_ as well
                  lambda: ref.PINObserverFullField(plane_num=3, **pino_kw),
                  lambda: ref.PolicyModel2D(**pino_kw)):
        r = build()
        before = {k: v.data_ptr() for k, v in r.named_parameters()}
        keys = list(r.state_dict().keys())
        c = P.convert_(r)
        assert {k: v.data_ptr() for k, v in c.named_parameters()} == before
        assert list(c.state_dict().keys()) == keys
        native = [m for m in c.modules() if type(m).__module__.startswith("pde_policylearning_b200")]
        assert native, "nothing was converted"


def test_convert_shares_parameters_with_stand_in_reference_modules(golden):
    """convert_ without the reference: every module of a native model is re-classed as a stand-in that carries the
    reference's class name (FactorizedSpectralConv, SpectralConv2d / 3d, FNOBlocks, ...) and lives outside this package,
    so convert_ sees what it sees in a reference model: class names and parameter layout.  The key list and shapes are
    pinned to the state_dicts the unmodified reference recorded in the fixtures.  convert_ must swap every spectral conv
    and every fusable container for a native module and keep the same Parameter objects and state_dict keys."""
    import pde_policylearning_b200 as P
    ref_names = {"SpectralConv": "FactorizedSpectralConv", "RnoSpectralConv2d": "SpectralConv2d",
                 "PinoSpectralConv3d": "SpectralConv3d", "PinoSpectralConv2d": "SpectralConv2d"}
    # what the reference's classes store and the native mirrors drop (they reject any other value at construction)
    ref_attrs = {"FNOBlocks": {"preactivation": False}}
    stand_ins = {}

    def as_reference(model):
        for m in model.modules():
            cls = type(m)
            if cls.__module__.startswith("pde_policylearning_b200"):
                if cls not in stand_ins:
                    stand_ins[cls] = type(ref_names.get(cls.__name__, cls.__name__), (cls,),
                                          {"__module__": "reference_stand_in", **ref_attrs.get(cls.__name__, {})})
                m.__class__ = stand_ins[cls]
        return model

    pino_kw = dict(modes1=[3] * 3, modes2=[3] * 3, modes3=[3] * 3, fc_dim=16, layers=[8] * 4, act="gelu", pad_ratio=0.0625)
    for build, fixture in ((lambda: P.FNO2d(8, 8, 16, in_channels=3, out_channels=1), "a3_fno2d"),
                           (lambda: P.RNO2d(4, 4, 6, 0, layer_num=1), "a5_rno2d_L1"),
                           (lambda: P.PINObserver2d(**pino_kw), "a7_pinobserver2d"),
                           (lambda: P.PINObserverFullField(plane_num=3, **pino_kw), "a10_pinobserver_fullfield"),
                           (lambda: P.PolicyModel2D(**pino_kw), "a11_policy_model2d")):
        r = as_reference(build())
        ref_sd = golden(fixture)["state_dict"]
        assert {k: tuple(v.shape) for k, v in r.state_dict().items()} == {k: tuple(v.shape) for k, v in ref_sd.items()}
        swapped = ("FactorizedSpectralConv", "SpectralConv2d", "SpectralConv3d", "FNOBlocks", "FourierLayer2d", "Lifting", "Projection")
        convs = [n for n, m in r.named_modules() if type(m).__name__ in swapped]
        assert convs and all(type(dict(r.named_modules())[n]).__module__ == "reference_stand_in" for n in convs)
        before = dict(r.named_parameters())
        keys = list(r.state_dict().keys())
        c = P.convert_(r)
        after = dict(c.named_parameters())
        assert after.keys() == before.keys() and all(after[k] is before[k] for k in before)
        assert list(c.state_dict().keys()) == keys
        mods = dict(c.named_modules())
        assert all(type(mods[n]).__module__.startswith("pde_policylearning_b200") for n in convs), fixture


def test_fast_erf_coefficients():
    """The rational erf used by the CUDA GELU (csrc/common.cuh::b2no_erf), restated in numpy float32:
    pins the coefficients and the accuracy claim without a GPU."""
    import numpy as np
    src = open(os.path.join(ROOT, "pde_policylearning_b200", "csrc", "common.cuh")).read()
    body = src[src.index("float b2no_erf"):src.index("return __fdividef")]
    nums = [float(t) for t in re.findall(r"-?\d\.\d+e-\d+", body)]
    assert len(nums) == 12
    a, b = nums[:7], nums[7:]
    x = np.clip(np.linspace(-6, 6, 400001), -4, 4).astype(np.float32)
    x2 = x * x
    p = np.full_like(x, a[0])
    for c in a[1:]:
        p = p * x2 + np.float32(c)
    q = np.full_like(x, b[0])
    for c in b[1:]:
        q = q * x2 + np.float32(c)
    approx = (x * p / q).astype(np.float64)
    ref = torch.erf(torch.linspace(-6, 6, 400001, dtype=torch.float64)).numpy()
    assert np.abs(approx - ref).max() < 6e-7


def test_gelu_with_gradient_formulation():
    """csrc/common.cuh::b2no_gelu2_both (Abramowitz-Stegun 7.1.26 on the Gaussian the derivative needs anyway), restated in
    numpy float32 with the coefficients read from the source: GELU and GELU' against float64 (F.gelu is the erf form)."""
    import numpy as np
    src = open(os.path.join(ROOT, "pde_policylearning_b200", "csrc", "common.cuh")).read()
    body = src[src.index("void b2no_gelu2_both"):src.index("float2 b2no_gelu2_grad")]
    nums = [float(t) for t in re.findall(r"b2no_f2\((-?\d+\.\d+)f\)", body)]
    p, one, a5, a4, a3, a2, a1, c, mh, ph, half, k = [np.float32(v) for v in nums]
    assert (one, mh, ph, half) == (1.0, -0.5, 0.5, 0.5)
    f = np.float32
    x = np.linspace(-12, 12, 400001).astype(f)
    t = (f(1) / (f(1) + p * np.abs(x))).astype(f)
    q = a5
    for a in (a4, a3, a2, a1):
        q = (q * t + a).astype(f)
    q = (q * t).astype(f)
    g = np.exp2(((x * x).astype(f) * c).astype(f)).astype(f)
    cdf = (half + np.copysign((ph + mh * (q * g).astype(f)).astype(f), x)).astype(f)
    val, grad = (x * cdf).astype(f), (cdf + (x * k).astype(f) * g).astype(f)
    x64 = torch.from_numpy(x.astype(np.float64)).requires_grad_(True)
    ref = torch.nn.functional.gelu(x64)
    (gref,) = torch.autograd.grad(ref.sum(), x64)
    assert np.abs(val - ref.detach().numpy()).max() < 6e-7
    assert np.abs(grad - gref.numpy()).max() < 6e-7


def test_pino_residual_matches_reference_fixture_and_oracle(golden):
    """Row a8 (diff_control_env.py:5-41) as DFT-matrix contractions: the residual of the reference's own output equals
    the Du the unmodified reference produced (fixture), and values + gradients equal the torch.fft restatement."""
    import pde_policylearning_b200 as P
    from oracle import restated as rs
    c = golden("a7_pinobserver2d")
    re = c["inputs"][1]
    du = P.fdm_ns_vorticity(c["out"].reshape(2, 8, 8, 17), 1 / re, c["t_interval"])
    assert float((du - c["Du"]).norm() / c["Du"].norm()) < 1e-5
    assert torch.equal(P.get_forcing(8), c["forcing"])
    torch.manual_seed(3)
    for n, t in ((16, 6), (64, 5)):
        w = torch.randn(2, n, n, t, dtype=torch.float64, requires_grad=True)
        v = torch.rand(2, dtype=torch.float64) * 0.01 + 0.002
        a = P.fdm_ns_vorticity(w, v, 0.5)
        b = rs.fdm_ns_vorticity(w, v, 0.5)
        assert float((a - b).norm() / b.norm()) < 1e-12
        g = torch.randn_like(a)
        (ga,) = torch.autograd.grad(a, w, g, retain_graph=True)
        (gb,) = torch.autograd.grad(b, w, g)
        assert float((ga - gb).norm() / gb.norm()) < 1e-12
    with pytest.raises(ValueError):
        P.fdm_ns_vorticity(torch.randn(1, 7, 7, 4), torch.ones(1), 1.0)


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference: ONE JSON line on stdout with the contract's keys (the CPU arm runs without a GPU)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=280)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "fno2d_fwd_bwd_samples_per_s" and d["unit"] == "samples/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_bench_rejects_bad_arguments():
    """--steps below 1, and --dump-outputs where no b200 training step is timed, end in an argument error."""
    import subprocess
    import sys
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-500:])


@pytest.mark.gpu
def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs writes the last timed step's loss, parameters and gradients as float32 .npy files (<= 64 MB
    in all); the same arguments give the same outputs (one step from the seeded weights on the seeded batch), and --steps
    sets how many timed steps ran before the dump.  Three bench.py --quick processes, ~12 s in all on one B200."""
    import json
    import subprocess
    import sys

    import numpy as np
    bench = os.path.join(ROOT, "bench.py")

    def run(out, steps):
        r = subprocess.run([sys.executable, bench, "--quick", "--steps", str(steps), "--warmup", "3", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=280)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["value"] > 0
        return {f.name[:-4]: np.load(f) for f in sorted(out.glob("*.npy"))}

    a, b, c = run(tmp_path / "a", 1), run(tmp_path / "b", 1), run(tmp_path / "c", 2)
    assert a.keys() == b.keys() == c.keys()
    assert "loss" in a and any(k.startswith("param.") for k in a) and any(k.startswith("grad.") for k in a)
    assert all(v.dtype == np.float32 for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20
    assert np.isfinite(a["loss"]).all()
    dist = lambda x, y: float(np.linalg.norm((x - y).ravel())) / max(float(np.linalg.norm(y.ravel())), 1e-30)
    worst = max((dist(a[k], b[k]), k) for k in a)
    assert worst[0] < 1e-4, worst
    assert max(dist(c[k], a[k]) for k in a if k.startswith("param.")) > 1e-6      # one more Adam step moved the weights


def test_bench_warmup_runs_a_fixed_number_of_steps():
    """The training step contains the gradient all-reduce at N > 1, so every untimed step before the timed region must be
    counted, not clocked: a time-based warm-up loop gave the ranks different numbers of collectives and the 8-GPU run hung."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    region = src[src.index("res_in = (graphed.static_in[0]"):src.index("l0 = ops.launch_count()")]
    assert "step(*res_in)" in region
    assert "perf_counter" not in region and "time.time" not in region and "while " not in region
