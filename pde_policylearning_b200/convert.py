"""convert_(model): swap the reference's spectral-conv modules inside an already built / loaded model for the
native ones, RE-USING the same nn.Parameter objects, so state_dict keys, optimizer state and whole-module
pickles (run_pde_observers.py:314, run_control.py:40) are unchanged (SURVEY.md 8b).

Recognised by class name + parameter layout (no import of the reference is needed):
  * FactorizedSpectralConv{,1d,2d,3d}  (neuralop/models/spectral_convolution.py)  -> SpectralConv
  * SpectralConv2d with ``fourier_weight`` (neuralop/models/rno.py:34-77)          -> RnoSpectralConv2d
  * SpectralConv3d with ``weights1..4``   (libs/models/pino_models/basics.py:99)   -> PinoSpectralConv3d
  * SpectralConv2d with ``weights1..2``   (libs/models/pino_models/basics.py:64)   -> PinoSpectralConv2d
With fuse=True the enclosing FNOBlocks / FourierLayer2d / Lifting / Projection are swapped as well so that the
skip, bias and activation run in the fused epilogue instead of separate PyTorch ops.
"""
from __future__ import annotations

import warnings

import torch
from torch import nn

from . import modules as M


def _is_dense(ref) -> bool:
    w = ref.weight[0] if isinstance(ref.weight, nn.ModuleList) else ref.weight
    name = getattr(w, "name", "dense")
    return str(name).lower().endswith("dense") and not getattr(ref, "separable", False)


def _convert_neuralop_conv(ref) -> nn.Module:
    new = M.SpectralConv.__new__(M.SpectralConv)
    nn.Module.__init__(new)
    for k in ("in_channels", "out_channels", "joint_factorization", "n_modes", "order", "half_total_n_modes",
              "rank", "factorization", "n_layers", "implementation", "output_scaling_factor", "fft_norm",
              "separable", "n_weights_per_layer"):
        setattr(new, k, getattr(ref, k))
    new.incremental_n_modes = ref.incremental_n_modes
    new.weight = ref.weight          # same container module, same Parameter objects
    new.bias = ref.bias
    new.train(ref.training)
    return new


def _convert_rno_conv(ref) -> nn.Module:
    new = M.RnoSpectralConv2d.__new__(M.RnoSpectralConv2d)
    nn.Module.__init__(new)
    for k in ("in_channels", "out_channels", "modes1", "modes2", "norm"):
        setattr(new, k, getattr(ref, k))
    new.fourier_weight = ref.fourier_weight
    new.train(ref.training)
    return new


def _convert_pino_conv(ref) -> nn.Module:
    new = M.PinoSpectralConv3d.__new__(M.PinoSpectralConv3d)
    nn.Module.__init__(new)
    for k in ("in_channels", "out_channels", "modes1", "modes2", "modes3", "scale"):
        setattr(new, k, getattr(ref, k))
    for k in range(1, 5):
        setattr(new, f"weights{k}", getattr(ref, f"weights{k}"))
    new.train(ref.training)
    return new


def _convert_pino_conv2d(ref) -> nn.Module:
    new = M.PinoSpectralConv2d.__new__(M.PinoSpectralConv2d)
    nn.Module.__init__(new)
    for k in ("in_channels", "out_channels", "modes1", "modes2", "scale"):
        setattr(new, k, getattr(ref, k))
    new.weights1, new.weights2 = ref.weights1, ref.weights2
    new.train(ref.training)
    return new


def _convert_fno_blocks(ref):
    ok = (not ref.preactivation and ref.fno_skip == "linear"
          and ref.output_scaling_factor is None and isinstance(ref.convs, M.SpectralConv))
    # two-layer GELU MLPs without dropout and soft-gating skips without bias run as Fn.channel_mlp (M.mlp_supported), and
    # not together with a norm; any other MLP keeps the block in torch
    mlp, mlp_skips = getattr(ref, "mlp", None), getattr(ref, "mlp_skips", None)
    if ok and mlp is not None:
        ok = (ref.norm is None and mlp_skips is not None and len(mlp) >= ref.n_layers and len(mlp_skips) >= ref.n_layers
              and all(M.mlp_supported(mlp[i], mlp_skips[i], ref.out_channels) for i in range(ref.n_layers)))
    # instance / group norms run on the spectrum (M.norm_args); any other norm keeps the block in torch
    if ok and ref.norm is not None:
        ok = len(ref.norm) >= ref.n_layers and all(M.norm_args(m, ref.out_channels) is not None for m in ref.norm)
    if not ok:
        return None
    new = M.FNOBlocks.__new__(M.FNOBlocks)
    nn.Module.__init__(new)
    for k in ("n_modes", "n_dim", "output_scaling_factor", "_incremental_n_modes", "in_channels", "out_channels",
              "n_layers", "joint_factorization", "non_linearity", "fno_skip", "mlp_skip", "fft_norm"):
        setattr(new, k, getattr(ref, k))
    new.convs = ref.convs
    new.fno_skips = ref.fno_skips
    new.mlp = mlp                    # the same MLP and gating modules (and Parameters), or None
    new.mlp_skips = mlp_skips if mlp is not None else None
    new.norm = ref.norm              # the same norm modules (and Parameters), or None
    new.train(ref.training)
    return new


def _convert_fourier_layer(ref):
    if not isinstance(ref.spec_conv, M.RnoSpectralConv2d):
        return None
    new = M.FourierLayer2d.__new__(M.FourierLayer2d)
    nn.Module.__init__(new)
    for k in ("modes1", "modes2", "width"):
        setattr(new, k, getattr(ref, k))
    new.spec_conv = ref.spec_conv
    new.norm_conv1d = ref.norm_conv1d
    new.train(ref.training)
    return new


def _convert_lifting(ref):
    new = M.Lifting.__new__(M.Lifting)
    nn.Module.__init__(new)
    new.in_channels, new.out_channels = ref.in_channels, ref.out_channels
    new.fc = ref.fc
    new.train(ref.training)
    return new


def _convert_projection(ref):
    try:
        M._act_name(ref.non_linearity)
    except NotImplementedError:
        return None
    new = M.Projection.__new__(M.Projection)
    nn.Module.__init__(new)
    for k in ("in_channels", "out_channels", "hidden_channels", "non_linearity"):
        setattr(new, k, getattr(ref, k))
    new.fc1, new.fc2 = ref.fc1, ref.fc2
    new.train(ref.training)
    return new


def _native(mod) -> bool:
    return type(mod).__module__.startswith(__package__)


def _swap(mod: nn.Module, fuse: bool):
    if _native(mod):
        return None
    name = type(mod).__name__
    if name in ("FactorizedSpectralConv", "FactorizedSpectralConv1d", "FactorizedSpectralConv2d",
                "FactorizedSpectralConv3d") and hasattr(mod, "half_n_modes"):
        if not _is_dense(mod):
            warnings.warn(f"convert_: leaving {name} with non-dense / separable weights untouched")
            return None
        if not 1 <= mod.order <= 3:
            return None
        return _convert_neuralop_conv(mod)
    if name == "SpectralConv2d" and hasattr(mod, "fourier_weight"):
        return _convert_rno_conv(mod)
    if name == "SpectralConv3d" and all(hasattr(mod, f"weights{k}") for k in range(1, 5)):
        return _convert_pino_conv(mod)
    if (name == "SpectralConv2d" and hasattr(mod, "weights1") and hasattr(mod, "weights2") and not hasattr(mod, "weights3")
            and getattr(mod.weights1, "is_complex", lambda: False)() and mod.weights1.dim() == 4):
        return _convert_pino_conv2d(mod)                      # libs/models/pino_models/basics.py:64-96
    if fuse:
        if name == "FNOBlocks" and hasattr(mod, "fno_skips"):
            return _convert_fno_blocks(mod)
        if name == "FourierLayer2d" and hasattr(mod, "norm_conv1d"):
            return _convert_fourier_layer(mod)
        if name == "Lifting" and hasattr(mod, "fc"):
            return _convert_lifting(mod)
        if name == "Projection" and hasattr(mod, "fc1") and hasattr(mod, "fc2"):
            return _convert_projection(mod)
    return None


def convert_(model: nn.Module, fuse: bool = True) -> nn.Module:
    """In-place conversion; returns the (possibly replaced) root module.  Children are converted first so
    that parents see native convs when deciding whether they can fuse."""
    for child_name, child in list(model.named_children()):
        new_child = convert_(child, fuse)
        if new_child is not child:
            setattr(model, child_name, new_child)
    new = _swap(model, fuse)
    return model if new is None else new
