"""TEST INFRASTRUCTURE ONLY -- loader for the *unmodified* reference modules.

Only ``tests/``, ``tests/golden/make_golden.py``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import this file.
The product package (``pde_policylearning_b200``) never does.

The reference (a checkout of it, named by ``B2NO_REFERENCE_ROOT``) is pure Python/PyTorch but its ``neuralop`` half
imports ``tensorly`` / ``tltorch`` / ``torch_harmonics`` which are not installed and
cannot be installed (no network).  SURVEY.md Appendix A lists the exact third-party
surface the dense path touches; this file registers in-memory stand-ins for those
names (parameter *storage* only -- every arithmetic op stays ``torch.fft`` /
``torch.einsum``) and then imports the reference files from where they lie.  Nothing
is copied out of the checkout.

The reference is not part of this repository, so ``available()`` must be checked first;
what the tests need from it is turned into fixtures under ``tests/golden/`` by
``tests/golden/make_golden.py``.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

import torch
from torch import nn

REFERENCE_ROOT = os.environ.get("B2NO_REFERENCE_ROOT", "")


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "neuralop", "models"))


# --------------------------------------------------------------------------------------
# Stand-ins for tensorly / tltorch (dense ComplexDense storage only)
# --------------------------------------------------------------------------------------
class _DenseFactorizedTensor(nn.Module):
    """Holder of ONE complex64 parameter.

    Mirrors the subset of ``tltorch.FactorizedTensor`` that
    neuralop/models/spectral_convolution.py:126-134,253-269,276-280 touches:
    ``.new``, ``.normal_``, ``.to_tensor``, ``.name``, ``__getitem__``, ``from_tensor``.
    """

    name = "ComplexDense"

    def __init__(self, shape=None, tensor=None):
        super().__init__()
        if tensor is None:
            tensor = torch.zeros(*shape, dtype=torch.cfloat)
        self.tensor = nn.Parameter(tensor.to(torch.cfloat))
        self.shape = tuple(self.tensor.shape)

    @classmethod
    def new(cls, shape, rank=None, factorization="ComplexDense", fixed_rank_modes=None, **kw):
        f = str(factorization).lower()
        if not f.endswith("dense"):
            raise NotImplementedError(
                f"oracle stub supports dense weights only (got factorization={factorization!r}); "
                "CP/Tucker/TT arithmetic lives in tltorch which is absent -> parity unpinned for it"
            )
        return cls(shape=tuple(shape))

    @classmethod
    def from_tensor(cls, tensor, rank=None, factorization="ComplexDense", **kw):
        return cls(tensor=tensor.detach().clone())

    def normal_(self, mean=0.0, std=1.0):
        with torch.no_grad():
            # complex normal: torch fills real and imag parts (variance split like torch does)
            self.tensor.normal_(mean, std)
        return self

    def to_tensor(self):
        return self.tensor

    def __getitem__(self, idx):
        return self.tensor[idx]

    @property
    def ndim(self):
        return self.tensor.ndim


def _install_stubs() -> None:
    if "tensorly" in sys.modules and getattr(sys.modules["tensorly"], "__b2no_stub__", False):
        return
    tl = types.ModuleType("tensorly")
    tl.__b2no_stub__ = True
    tl.set_backend = lambda *a, **k: None
    tl.ndim = lambda x: x.ndim
    tl.einsum = lambda eq, *ops: torch.einsum(eq, *ops)
    plugins = types.ModuleType("tensorly.plugins")
    plugins.use_opt_einsum = lambda *a, **k: None
    tl.plugins = plugins

    tlt = types.ModuleType("tltorch")
    tlt.__b2no_stub__ = True
    ft = types.ModuleType("tltorch.factorized_tensors")
    core = types.ModuleType("tltorch.factorized_tensors.core")
    core.FactorizedTensor = _DenseFactorizedTensor
    ft.core = core
    tlt.factorized_tensors = ft
    tlt.FactorizedTensor = _DenseFactorizedTensor
    tlt.TensorizedTensor = object
    utils = types.ModuleType("tltorch.utils")
    utils.get_tensorized_shape = lambda *a, **k: None
    tlt.utils = utils

    th = types.ModuleType("torch_harmonics")
    th.RealSHT = object
    th.InverseRealSHT = object

    sys.modules.update({
        "tensorly": tl, "tensorly.plugins": plugins,
        "tltorch": tlt, "tltorch.factorized_tensors": ft,
        "tltorch.factorized_tensors.core": core, "tltorch.utils": utils,
        "torch_harmonics": th,
    })


def _install_namespace_packages() -> None:
    """Bypass neuralop/__init__.py and neuralop/models/__init__.py (they pull wandb, h5py,
    zarr, uno, ...): register empty packages whose __path__ points at the reference dirs."""
    for name, sub in (("neuralop", "neuralop"), ("neuralop.models", "neuralop/models")):
        if name in sys.modules:
            continue
        m = types.ModuleType(name)
        m.__path__ = [os.path.join(REFERENCE_ROOT, sub)]
        m.__b2no_stub__ = True
        sys.modules[name] = m


_loaded = {}


def load():
    """Returns a namespace with the reference classes on the hot path (SURVEY.md section 8a)."""
    if _loaded:
        return types.SimpleNamespace(**_loaded)
    if not available():
        raise RuntimeError(f"reference tree not present at {REFERENCE_ROOT}")
    _install_stubs()
    _install_namespace_packages()
    sc = importlib.import_module("neuralop.models.spectral_convolution")
    fb = importlib.import_module("neuralop.models.fno_block")
    tfno = importlib.import_module("neuralop.models.tfno")
    rno = importlib.import_module("neuralop.models.rno")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    # libs/__init__ chain: import the leaf files directly to avoid matlab/h5py imports.
    libs = types.ModuleType("libs"); libs.__path__ = [os.path.join(REFERENCE_ROOT, "libs")]
    sys.modules.setdefault("libs", libs)
    lm = types.ModuleType("libs.models"); lm.__path__ = [os.path.join(REFERENCE_ROOT, "libs/models")]
    sys.modules.setdefault("libs.models", lm)
    pm = types.ModuleType("libs.models.pino_models")
    pm.__path__ = [os.path.join(REFERENCE_ROOT, "libs/models/pino_models")]
    sys.modules.setdefault("libs.models.pino_models", pm)
    basics = importlib.import_module("libs.models.pino_models.basics")
    # pinobserver imports libs.DINo.network (torchdiffeq-free file) -- give it a stub if it fails
    try:
        pinobs = importlib.import_module("libs.models.pino_models.pinobserver")
    except Exception:  # pragma: no cover - depends on absent deps
        dn = types.ModuleType("libs.DINo"); dn.__path__ = []
        net = types.ModuleType("libs.DINo.network"); net.MultiplicativeNet = object
        sys.modules["libs.DINo"] = dn; sys.modules["libs.DINo.network"] = net
        pinobs = importlib.import_module("libs.models.pino_models.pinobserver")
    f2d = importlib.import_module("libs.models.pino_models.fourier2d")
    pu = types.ModuleType("libs.pino_utils"); pu.__path__ = [os.path.join(REFERENCE_ROOT, "libs/pino_utils")]
    sys.modules.setdefault("libs.pino_utils", pu)
    losses = importlib.import_module("libs.pino_utils.losses")
    envs = types.ModuleType("libs.envs"); envs.__path__ = [os.path.join(REFERENCE_ROOT, "libs/envs")]
    sys.modules.setdefault("libs.envs", envs)
    dce = importlib.import_module("libs.envs.diff_control_env")

    _loaded.update(
        FactorizedTensor=_DenseFactorizedTensor,
        spectral_convolution=sc, fno_block=fb, tfno=tfno, rno=rno, basics=basics,
        pinobserver=pinobs, losses=losses, diff_control_env=dce,
        FactorizedSpectralConv=sc.FactorizedSpectralConv,
        FactorizedSpectralConv1d=sc.FactorizedSpectralConv1d,
        FactorizedSpectralConv2d=sc.FactorizedSpectralConv2d,
        FactorizedSpectralConv3d=sc.FactorizedSpectralConv3d,
        FNOBlocks=fb.FNOBlocks, FNO=tfno.FNO, FNO1d=tfno.FNO1d, FNO2d=tfno.FNO2d, FNO3d=tfno.FNO3d,
        RnoSpectralConv2d=rno.SpectralConv2d, FourierLayer2d=rno.FourierLayer2d,
        RNO_cell=rno.RNO_cell, RNO_layer=rno.RNO_layer, RNO2d=rno.RNO2d,
        SpectralConvWithFC=rno.SpectralConvWithFC, SpectralRegressor=rno.SpectralRegressor,
        PinoSpectralConv3d=basics.SpectralConv3d, PinoSpectralConv2d=basics.SpectralConv2d,
        PinoSpectralConv1d=basics.SpectralConv1d,
        PINObserver2d=pinobs.PINObserver2d, MultiplicativeNet=pinobs.MultiplicativeNet,
        PINObserverFullField=pinobs.PINObserverFullField, PolicyModel2D=pinobs.PolicyModel2D,
        PinoFNO2d=f2d.FNO2d,
        LpLoss=losses.LpLoss, get_forcing=losses.get_forcing,
        Channelflow_PINO_loss=dce.Channelflow_PINO_loss, FDM_NS_vorticity=dce.FDM_NS_vorticity,
    )
    return types.SimpleNamespace(**_loaded)


class RefFNO2dObserver(nn.Module):
    """libs/models/fno_models.py:16-57 cannot be imported (matplotlib import at :7); this is the
    same 12 lines of glue expressed around the *reference* FNO2d so the observer-level oracle
    still runs the reference's FNO2d unmodified."""

    def __init__(self, modes1, modes2, width):
        super().__init__()
        ref = load()
        self.fno2d = ref.FNO2d(modes1, modes2, width, in_channels=3, out_channels=1)

    def forward(self, p_plane, v_plane=None):
        import numpy as np
        b, sx, sy = p_plane.shape[0], p_plane.shape[1], p_plane.shape[2]
        gx = torch.tensor(np.linspace(0, 1, sx), dtype=torch.float).reshape(1, sx, 1, 1).repeat([b, 1, sy, 1])
        gy = torch.tensor(np.linspace(0, 1, sy), dtype=torch.float).reshape(1, 1, sy, 1).repeat([b, sx, 1, 1])
        x = torch.cat((p_plane, gx.to(p_plane.device), gy.to(p_plane.device)), dim=-1).permute(0, 3, 1, 2)
        return self.fno2d(x)
