"""Host-side mirror of the reference's operator interface for the SpectralConv hot path.

Same class roles, constructor signatures, parameter names / shapes and state_dict keys as the reference
(SURVEY.md 8a.4), so reference checkpoints load unchanged and the callers (run_pde_observers.py,
train_pino.py, run_control.py) can pick the layers up as drop-ins; the arithmetic runs in libb2no.so.

    SpectralConv{,1d,2d,3d}   <-> neuralop/models/spectral_convolution.py:143-457  FactorizedSpectralConv*
    FNOBlocks / Lifting / Projection / FNO / FNO{1,2,3}d <-> neuralop/models/{fno_block,tfno}.py
    RnoSpectralConv2d, FourierLayer2d, RNO_cell, RNO_layer, SpectralConvWithFC, SpectralRegressor, RNO2d
                              <-> neuralop/models/rno.py
    PinoSpectralConv3d, MultiplicativeNet, PINObserver2d <-> libs/models/pino_models/{basics,pinobserver}.py
    FNO2dObserver, RNO2dObserver, LpLoss <-> libs/models/{fno_models,rno_models}.py, libs/utilities3.py
"""
from __future__ import annotations

import itertools
import math
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from . import functional as Fn
from .ops import SpecGeom


# =============================================================================================
# neuralop family
# =============================================================================================
class ComplexDenseWeight(nn.Module):
    """Stands where tltorch's ComplexDense FactorizedTensor stands in the reference
    (spectral_convolution.py:253-268): one complex64 parameter registered as ``tensor`` so the state_dict
    key is ``...weight.<i>.tensor``.  Checkpoints that store the real view (..., 2) (newer tltorch) load too."""

    name = "ComplexDense"

    def __init__(self, shape):
        super().__init__()
        self.tensor = nn.Parameter(torch.zeros(*shape, dtype=torch.cfloat))

    @property
    def shape(self):
        return tuple(self.tensor.shape)

    def normal_(self, mean=0.0, std=1.0):
        with torch.no_grad():
            self.tensor.normal_(mean, std)
        return self

    def to_tensor(self):
        return self.tensor

    def __getitem__(self, idx):
        return self.tensor[idx]

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        key = prefix + "tensor"
        if key in state_dict and not state_dict[key].is_complex() and state_dict[key].shape[-1] == 2 \
                and tuple(state_dict[key].shape[:-1]) == tuple(self.tensor.shape):
            state_dict[key] = torch.view_as_complex(state_dict[key].contiguous())
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)


def _check_dense(factorization, separable, implementation):
    f = "dense" if factorization is None else str(factorization).lower()
    if f.startswith("complex"):
        f = f[len("complex"):]
    if f != "dense":
        raise NotImplementedError(
            f"factorization={factorization!r}: only dense spectral weights are implemented natively "
            "(CP/Tucker/TT arithmetic lives in tltorch; SURVEY.md 8c marks its parity unpinned)")
    if separable:
        raise NotImplementedError("separable spectral convolution is not implemented in the native path")
    if implementation not in ("factorized", "reconstructed"):
        raise ValueError(f'Got implementation={implementation!r}, expected "reconstructed" or "factorized"')


class SpectralConv(nn.Module):
    """Generic N-D (1-3) truncated Fourier convolution; constructor signature of
    FactorizedSpectralConv (spectral_convolution.py:183-187)."""

    def __init__(self, in_channels, out_channels, n_modes, incremental_n_modes=None, bias=True,
                 n_layers=1, separable=False, output_scaling_factor=None,
                 rank=0.5, factorization=None, implementation="reconstructed",
                 fixed_rank_modes=False, joint_factorization=False, decomposition_kwargs=dict(),
                 init_std="auto", fft_norm="backward"):
        super().__init__()
        _check_dense(factorization, separable, implementation)
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.joint_factorization = joint_factorization
        if isinstance(n_modes, int):
            n_modes = [n_modes]
        self.n_modes = n_modes
        self.order = len(n_modes)
        if not 1 <= self.order <= 3:
            raise NotImplementedError("native spectral conv supports 1, 2 or 3 spatial dims")
        self.half_total_n_modes = [m // 2 for m in n_modes]
        self.incremental_n_modes = incremental_n_modes
        self.rank = rank
        self.factorization = factorization
        self.n_layers = n_layers
        self.implementation = implementation
        self.separable = separable
        if output_scaling_factor is not None:
            if isinstance(output_scaling_factor, (float, int)):
                output_scaling_factor = [[float(output_scaling_factor)] * len(self.n_modes)] * n_layers
            elif isinstance(output_scaling_factor[0], (float, int)):
                output_scaling_factor = [[s] * len(self.n_modes) for s in output_scaling_factor]
        self.output_scaling_factor = output_scaling_factor
        init_std = (1 / (in_channels * out_channels)) if init_std == "auto" else 0.02  # quirk Q3
        self.fft_norm = fft_norm
        weight_shape = (in_channels, out_channels, *self.half_total_n_modes)
        self.n_weights_per_layer = 2 ** (self.order - 1)
        if joint_factorization:
            self.weight = ComplexDenseWeight((self.n_weights_per_layer * n_layers, *weight_shape))
            self.weight.normal_(0, init_std)
        else:
            self.weight = nn.ModuleList([ComplexDenseWeight(weight_shape)
                                         for _ in range(self.n_weights_per_layer * n_layers)])
            for w in self.weight:
                w.normal_(0, init_std)
        if bias:
            self.bias = nn.Parameter(init_std * torch.randn(*((n_layers, self.out_channels) + (1,) * self.order)))
        else:
            self.bias = None

    # ---- incremental modes (spectral_convolution.py:282-301) --------------------------------
    @property
    def incremental_n_modes(self):
        return self._incremental_n_modes

    @incremental_n_modes.setter
    def incremental_n_modes(self, incremental_n_modes):
        if incremental_n_modes is None:
            self._incremental_n_modes = None
            self.half_n_modes = [m // 2 for m in self.n_modes]
        else:
            if isinstance(incremental_n_modes, int):
                self._incremental_n_modes = [incremental_n_modes] * len(self.n_modes)
            elif len(incremental_n_modes) == len(self.n_modes):
                self._incremental_n_modes = incremental_n_modes
            else:
                raise ValueError(f"Provided {incremental_n_modes} for actual n_modes={self.n_modes}.")
            self.weight_slices = [slice(None)] * 2 + [slice(None, n // 2) for n in self._incremental_n_modes]
            self.half_n_modes = [m // 2 for m in self._incremental_n_modes]

    def _get_weight(self, index):
        w = self.weight[index]
        if not torch.is_tensor(w):
            w = w.to_tensor()
        if self.incremental_n_modes is not None:
            return w[tuple(self.weight_slices)]
        return w

    # ---- geometry -----------------------------------------------------------------------------
    def _geom(self, grid, indices) -> SpecGeom:
        nout = None
        if self.output_scaling_factor is not None:
            nout = tuple(int(round(s * r)) for s, r in zip(grid, self.output_scaling_factor[indices]))
        return SpecGeom(nin=tuple(grid), half=tuple(self.half_n_modes), norm=self.fft_norm, nout=nout)

    def corners(self, indices=0) -> List[torch.Tensor]:
        """itertools.product order == canonical corner order (spectral_convolution.py:330-337)."""
        return [self._get_weight(self.n_weights_per_layer * indices + i) for i in range(self.n_weights_per_layer)]

    def forward(self, x, indices=0):
        return self.forward_fused(x, indices)

    def forward_fused(self, x, indices=0, pw_weight=None, act=None, norm=None):
        """spectral conv + bias [-> norm] [+ 1x1 skip + activation] in one fused pass; norm: an nn.GroupNorm or
        InstanceNorm{1,2,3}d module (norm_args)."""
        if x.dim() != 2 + self.order:
            raise ValueError(f"expected a {2 + self.order}-D input (batch, channels, *grid)")
        geom = self._geom(tuple(x.shape[2:]), indices)
        bias = None if self.bias is None else self.bias[indices].reshape(-1)
        return Fn.spectral_block(x, self.corners(indices), geom, bias=bias, pw_weight=pw_weight, act=act,
                                 norm=None if norm is None else _norm_args_or_raise(norm, self.out_channels))

    def get_conv(self, indices):
        if self.n_layers == 1:
            raise ValueError("A single convolution is parametrized, directly use the main class.")
        return SubConv(self, indices)

    def __getitem__(self, indices):
        return self.get_conv(indices)


class SubConv(nn.Module):
    """spectral_convolution.py:364-379."""

    def __init__(self, main_conv, indices):
        super().__init__()
        self.main_conv = main_conv
        self.indices = indices

    def forward(self, x):
        return self.main_conv.forward(x, self.indices)


class SpectralConv1d(SpectralConv):
    pass


class SpectralConv2d(SpectralConv):
    pass


class SpectralConv3d(SpectralConv):
    pass


FactorizedSpectralConv = SpectralConv
FactorizedSpectralConv1d, FactorizedSpectralConv2d, FactorizedSpectralConv3d = SpectralConv1d, SpectralConv2d, SpectralConv3d


_ACT_NAMES = {F.gelu: "gelu", F.relu: "relu", torch.tanh: "tanh", F.tanh: "tanh", torch.sigmoid: "sigmoid",
              F.selu: "selu", F.sigmoid: "sigmoid"}


def _act_name(fn):
    if fn is None or isinstance(fn, str):
        return fn
    if fn in _ACT_NAMES:
        return _ACT_NAMES[fn]
    if isinstance(fn, nn.GELU):
        return "gelu"
    if isinstance(fn, nn.ReLU):
        return "relu"
    raise NotImplementedError(f"activation {fn} has no native kernel (gelu/relu/tanh/sigmoid/selu)")


class Lifting(nn.Module):
    """tfno.py:11-20."""

    def __init__(self, in_channels, out_channels, n_dim=2):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.fc = getattr(nn, f"Conv{n_dim}d")(in_channels, out_channels, 1)

    def forward(self, x):
        return Fn.pointwise_conv(x, self.fc.weight, self.fc.bias, None)


class Projection(nn.Module):
    """tfno.py:23-38: conv -> non-linearity -> conv."""

    def __init__(self, in_channels, out_channels, hidden_channels=None, n_dim=2, non_linearity=F.gelu):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.hidden_channels = in_channels if hidden_channels is None else hidden_channels
        self.non_linearity = non_linearity
        Conv = getattr(nn, f"Conv{n_dim}d")
        self.fc1 = Conv(in_channels, hidden_channels, 1)
        self.fc2 = Conv(hidden_channels, out_channels, 1)

    def forward(self, x):
        return Fn.mlp_head(x, self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias,
                           _act_name(self.non_linearity))


def norm_args(m, channels: int):
    """(groups, eps, weight, bias) of a norm module the spectral path implements, else None: nn.GroupNorm over `channels`
    channels, or InstanceNorm{1,2,3}d without running statistics (GroupNorm with one channel per group; the statistics are
    always the instance's own, in training and in eval).  weight / bias are None without affine parameters."""
    if isinstance(m, nn.GroupNorm):
        if m.num_channels != channels or channels % m.num_groups != 0:
            return None
        return m.num_groups, m.eps, m.weight, m.bias
    if isinstance(m, nn.modules.instancenorm._InstanceNorm) and not m.track_running_stats and m.num_features == channels:
        return channels, m.eps, m.weight, m.bias
    return None


def _norm_args_or_raise(m, channels):
    a = norm_args(m, channels)
    if a is None:
        raise NotImplementedError(f"{m} has no native kernel: GroupNorm, or InstanceNorm without running statistics")
    return a


class MLP(nn.Module):
    """mlp.py:10-54: n_layers 1x1 convs, the non-linearity after EVERY layer (quirk Q3: `i < n_layers` always holds).
    FNOBlocks runs its two-layer MLPs through Fn.channel_mlp; this forward is for standalone use."""

    def __init__(self, in_channels, out_channels=None, hidden_channels=None, n_layers=2, n_dim=2, non_linearity=F.gelu,
                 dropout=0.0, **kwargs):
        super().__init__()
        self.n_layers = n_layers
        self.in_channels = in_channels
        self.out_channels = in_channels if out_channels is None else out_channels
        self.hidden_channels = in_channels if hidden_channels is None else hidden_channels
        self.non_linearity = non_linearity
        self.dropout = nn.ModuleList([nn.Dropout(dropout) for _ in range(n_layers)]) if dropout > 0.0 else None
        Conv = getattr(nn, f"Conv{n_dim}d")
        self.fcs = nn.ModuleList()
        for i in range(n_layers):
            ci = self.in_channels if i == 0 else self.hidden_channels
            co = self.out_channels if i == n_layers - 1 else self.hidden_channels
            self.fcs.append(Conv(ci, co, 1))

    def forward(self, x):
        for i, fc in enumerate(self.fcs):
            x = Fn.pointwise_conv(x, fc.weight, fc.bias, _act_name(self.non_linearity))
            if self.dropout is not None:
                x = self.dropout[i](x)
        return x


class SoftGating(nn.Module):
    """skip_connections.py:37-74: x * weight (+ bias), weight (1, C, 1...) initialised to ones."""

    def __init__(self, in_features, out_features=None, n_dim=2, bias=False):
        super().__init__()
        if out_features is not None and in_features != out_features:
            raise ValueError(f"Got in_features={in_features} and out_features={out_features} "
                             "but these two must be the same for soft-gating")
        self.in_features, self.out_features, self.n_dim = in_features, out_features, n_dim
        self.weight = nn.Parameter(torch.ones(1, self.in_features, *(1,) * n_dim))
        self.bias = nn.Parameter(torch.ones(1, self.in_features, *(1,) * n_dim)) if bias else None

    def forward(self, x):
        # a diagonal 1x1 conv on the native pointwise kernel
        return Fn.pointwise_conv(x, torch.diag(self.weight.reshape(-1)),
                                 None if self.bias is None else self.bias.reshape(-1), None)


def mlp_supported(mlp, skip, channels: int) -> bool:
    """True for the channel MLP Fn.channel_mlp implements (fno_block.py:123-170 with use_mlp): two 1x1 convs with biases,
    C -> H -> C, GELU, no dropout, and a soft-gating skip without bias."""
    if not (hasattr(mlp, "fcs") and len(mlp.fcs) == 2 and getattr(mlp, "dropout", None) is None
            and isinstance(skip, nn.Module) and type(skip).__name__ == "SoftGating" and getattr(skip, "bias", None) is None):
        return False
    try:
        if _act_name(mlp.non_linearity) != "gelu":
            return False
    except NotImplementedError:
        return False
    fc1, fc2 = mlp.fcs
    return (fc1.weight.shape[1] == channels and fc2.weight.shape[0] == channels and fc2.weight.shape[1] == fc1.weight.shape[0]
            and fc1.bias is not None and fc2.bias is not None and tuple(skip.weight.shape[:2]) == (1, channels))


class FNOBlocks(nn.Module):
    """fno_block.py:10-191 restricted to what FNO1d/2d/3d can reach (quirk Q2): linear skips, no preactivation.  Per layer
    ONE fused pass: spectral conv + bias [-> instance / group norm] + 1x1 skip + (GELU iff index < n_layers - index,
    fno_block.py:149).  The norm is applied to the conv's kept-mode spectrum before the inverse transform
    (ops.spec_norm_fwd), so it adds no pass over the activation.  With use_mlp (fno_block.py:123-170) the activation is
    always applied, then the channel MLP C -> round(C mlp_expansion) -> C (GELU after both convs), its soft-gating skip of
    the block input and the activation for every layer but the last run as one more fused node (Fn.channel_mlp); use_mlp
    with a norm, MLP dropout and the 'linear' / 'identity' MLP skips raise."""

    def __init__(self, in_channels, out_channels, n_modes, output_scaling_factor=None, n_layers=1,
                 incremental_n_modes=None, use_mlp=False, mlp_dropout=0, mlp_expansion=0.5,
                 non_linearity=F.gelu, norm=None, ada_in_features=None, preactivation=False,
                 fno_skip="linear", mlp_skip="soft-gating", separable=False, factorization=None, rank=1.0,
                 SpectralConv=SpectralConv, joint_factorization=False, fixed_rank_modes=False,
                 implementation="factorized", decomposition_kwargs=dict(), fft_norm="forward", **kwargs):
        super().__init__()
        if isinstance(n_modes, int):
            n_modes = [n_modes]
        if preactivation:
            raise NotImplementedError("native FNOBlocks: preactivation is outside the hot path (no BASELINE config enables it)")
        if use_mlp and norm is not None:
            # the second norm would act on the MLP output, which is not band-limited: no spectral form
            raise NotImplementedError("native FNOBlocks: use_mlp together with a norm has no native kernel")
        if use_mlp and mlp_dropout > 0:
            raise NotImplementedError("native FNOBlocks: mlp_dropout > 0 has no native kernel")
        if use_mlp and mlp_skip != "soft-gating":
            raise NotImplementedError("native FNOBlocks: the MLP skip runs natively as 'soft-gating' only")
        if norm not in (None, "instance_norm", "group_norm"):
            if norm == "ada_in":
                raise NotImplementedError("native FNOBlocks: norm='ada_in' is outside the hot path")
            raise ValueError(f"Got norm={norm} but expected None or one of [instance_norm, group_norm, ada_in]")
        if fno_skip != "linear":
            raise NotImplementedError("native FNOBlocks implements the 'linear' skip (the only one FNO2d reaches)")
        if output_scaling_factor is not None:
            raise NotImplementedError("native FNOBlocks: output_scaling_factor (FNO2d forces None, tfno.py:444)")
        self.n_modes, self.n_dim = n_modes, len(n_modes)
        self.output_scaling_factor = None
        self._incremental_n_modes = incremental_n_modes
        self.in_channels, self.out_channels, self.n_layers = in_channels, out_channels, n_layers
        self.joint_factorization = joint_factorization
        self.non_linearity = non_linearity
        self.fno_skip, self.mlp_skip, self.fft_norm = fno_skip, mlp_skip, fft_norm
        self.mlp = None
        self.mlp_skips = None
        self.norm = None
        self.convs = SpectralConv(in_channels, out_channels, self.n_modes, output_scaling_factor=None,
                                  incremental_n_modes=incremental_n_modes, rank=rank, fft_norm=fft_norm,
                                  fixed_rank_modes=fixed_rank_modes, implementation=implementation,
                                  separable=separable, factorization=factorization,
                                  decomposition_kwargs=decomposition_kwargs,
                                  joint_factorization=joint_factorization, n_layers=n_layers)
        Conv = getattr(nn, f"Conv{self.n_dim}d")
        self.fno_skips = nn.ModuleList([Conv(in_channels, out_channels, kernel_size=1, bias=False)
                                        for _ in range(n_layers)])
        if use_mlp:     # fno_block.py:75-84, registered after the fno skips
            self.mlp = nn.ModuleList([MLP(in_channels=out_channels, hidden_channels=int(round(out_channels * mlp_expansion)),
                                          dropout=mlp_dropout, n_dim=self.n_dim) for _ in range(n_layers)])
            self.mlp_skips = nn.ModuleList([SoftGating(in_channels, out_channels, n_dim=self.n_dim) for _ in range(n_layers)])
        if norm == "instance_norm":     # fno_block.py:94-105 with n_norms = 1 (no MLP), registered after the skips
            self.norm = nn.ModuleList([getattr(nn, f"InstanceNorm{self.n_dim}d")(num_features=out_channels)
                                       for _ in range(n_layers)])
        elif norm == "group_norm":
            self.norm = nn.ModuleList([nn.GroupNorm(num_groups=1, num_channels=out_channels) for _ in range(n_layers)])

    def forward(self, x, index=0):
        if self.mlp is not None:
            return self._forward_mlp(x, index)
        act = _act_name(self.non_linearity) if index < (self.n_layers - index) else None
        norm = None if self.norm is None else self.norm[index]
        if hasattr(self.convs, "forward_fused"):
            return self.convs.forward_fused(x, index, pw_weight=self.fno_skips[index].weight, act=act, norm=norm)
        # a user-supplied SpectralConv class: keep the reference's composition
        y = self.convs(x, index)
        if norm is not None:
            y = norm(y)
        y = y + Fn.pointwise_conv(x, self.fno_skips[index].weight, None, None)
        return self.non_linearity(y) if act is not None else y

    def _forward_mlp(self, x, index):
        """fno_block.py:123-170 with an MLP: u = act(conv(x) + skip x) (the activation always on), then
        y = gelu(fc2 gelu(fc1 u)) + g x, followed by act for every layer but the last."""
        act = _act_name(self.non_linearity)
        if hasattr(self.convs, "forward_fused"):
            u = self.convs.forward_fused(x, index, pw_weight=self.fno_skips[index].weight, act=act)
        else:
            u = self.non_linearity(self.convs(x, index) + Fn.pointwise_conv(x, self.fno_skips[index].weight, None, None))
        fc1, fc2 = self.mlp[index].fcs
        return Fn.channel_mlp(u, x, fc1.weight, fc1.bias, fc2.weight, fc2.bias, self.mlp_skips[index].weight,
                              act if index < self.n_layers - 1 else None)

    @property
    def incremental_n_modes(self):
        return self._incremental_n_modes

    @incremental_n_modes.setter
    def incremental_n_modes(self, incremental_n_modes):
        self.convs.incremental_n_modes = incremental_n_modes

    def get_block(self, indices):
        if self.n_layers == 1:
            raise ValueError("A single layer is parametrized, directly use the main class.")
        return SubModule(self, indices)

    def __getitem__(self, indices):
        return self.get_block(indices)


class SubModule(nn.Module):
    """fno_block.py:194-209."""

    def __init__(self, main_module, indices):
        super().__init__()
        self.main_module = main_module
        self.indices = indices

    def forward(self, x):
        return self.main_module.forward(x, self.indices)


class FNO(nn.Module):
    """tfno.py:42-219 (dense weights; domain padding / output scaling are out of the hot path)."""

    def __init__(self, n_modes, hidden_channels, in_channels=3, out_channels=1, lifting_channels=256,
                 projection_channels=256, n_layers=4, output_scaling_factor=None, incremental_n_modes=None,
                 use_mlp=False, mlp_dropout=0, mlp_expansion=0.5, non_linearity=F.gelu, norm=None,
                 preactivation=False, fno_skip="linear", mlp_skip="soft-gating", separable=False,
                 factorization=None, rank=1.0, joint_factorization=False, fixed_rank_modes=False,
                 implementation="factorized", decomposition_kwargs=dict(), domain_padding=None,
                 domain_padding_mode="one-sided", fft_norm="forward", SpectralConv=SpectralConv, **kwargs):
        super().__init__()
        if domain_padding is not None and domain_padding > 0:
            raise NotImplementedError("native FNO: domain_padding is outside the hot path (no config enables it)")
        if use_mlp:
            # the mirrored model classes keep rejecting use_mlp; channel-MLP blocks run natively as FNOBlocks(use_mlp=True):
            # the blocks of a converted reference model (convert_), or blocks assigned to fno_blocks, run by forward() below
            raise NotImplementedError("native FNO: use_mlp is not built by FNO / FNO1d / FNO2d / FNO3d; build the model with "
                                      "the reference classes and convert_() it, or assign FNOBlocks(use_mlp=True) to fno_blocks")
        self.n_dim = len(n_modes)
        self.n_modes = n_modes
        self.hidden_channels = hidden_channels
        self.lifting_channels, self.projection_channels = lifting_channels, projection_channels
        self.in_channels, self.out_channels, self.n_layers = in_channels, out_channels, n_layers
        self.joint_factorization = joint_factorization
        self.non_linearity = non_linearity
        self.fno_skip, self.mlp_skip = (fno_skip,), (mlp_skip,)  # 1-tuples as in tfno.py:147-148
        self.fft_norm = fft_norm
        self.domain_padding = None
        self._incremental_n_modes = incremental_n_modes
        self.output_scaling_factor = output_scaling_factor
        self.fno_blocks = FNOBlocks(
            in_channels=hidden_channels, out_channels=hidden_channels, n_modes=self.n_modes,
            output_scaling_factor=output_scaling_factor, use_mlp=use_mlp, mlp_dropout=mlp_dropout,
            mlp_expansion=mlp_expansion, non_linearity=non_linearity, norm=norm, preactivation=preactivation,
            fno_skip=fno_skip, mlp_skip=mlp_skip, incremental_n_modes=incremental_n_modes, rank=rank,
            fft_norm=fft_norm, fixed_rank_modes=fixed_rank_modes, implementation=implementation,
            separable=separable, factorization=factorization, decomposition_kwargs=decomposition_kwargs,
            joint_factorization=joint_factorization, SpectralConv=SpectralConv, n_layers=n_layers)
        self.lifting = Lifting(in_channels=in_channels, out_channels=self.hidden_channels, n_dim=self.n_dim)
        self.projection = Projection(in_channels=self.hidden_channels, out_channels=out_channels,
                                     hidden_channels=projection_channels, non_linearity=non_linearity,
                                     n_dim=self.n_dim)

    def forward(self, x):
        x = self.lifting(x)
        blocks = self.fno_blocks
        norm_args_l = None
        if isinstance(blocks, FNOBlocks) and blocks.norm is not None and hasattr(blocks.convs, "forward_fused"):
            norm_args_l = [_norm_args_or_raise(blocks.norm[i], blocks.out_channels) for i in range(self.n_layers)]
        if (isinstance(blocks, FNOBlocks) and blocks.mlp is None and hasattr(blocks.convs, "forward_fused")
                and blocks.convs.bias is not None
                and blocks.convs.output_scaling_factor is None and x.dim() == 2 + blocks.convs.order
                and (norm_args_l is None or len({(a[0], a[1], a[2] is None) for a in norm_args_l}) == 1)):
            # the whole stack as one autograd node: the backward chains act'(z) into the dx epilogues
            convs = blocks.convs
            geom = convs._geom(tuple(x.shape[2:]), 0)
            acts = [(_act_name(blocks.non_linearity) if i < (blocks.n_layers - i) else None) for i in range(self.n_layers)]
            layers = [(blocks.fno_skips[i].weight, convs.corners(i)) for i in range(self.n_layers)]
            norm = None
            if norm_args_l is not None:    # one (groups, eps) for the stack, each layer's own weight / bias
                norm = (norm_args_l[0][0], norm_args_l[0][1], [a[2:] for a in norm_args_l])
            x = Fn.fno_stack(x, geom, convs.bias, layers, acts, norm=norm)
        else:
            for layer_idx in range(self.n_layers):
                x = self.fno_blocks(x, layer_idx)
        return self.projection(x)

    @property
    def incremental_n_modes(self):
        return self._incremental_n_modes

    @incremental_n_modes.setter
    def incremental_n_modes(self, incremental_n_modes):
        self.fno_blocks.incremental_n_modes = incremental_n_modes


def _fno_nd_kwargs(kw):
    # FNO1d/2d/3d pass `skip=` which FNO.__init__ swallows (quirk Q2) and force output_scaling_factor=None
    kw = dict(kw)
    kw.pop("skip", None)
    kw["output_scaling_factor"] = None
    return kw


class FNO1d(FNO):
    def __init__(self, n_modes_height, hidden_channels, **kw):
        super().__init__(n_modes=(n_modes_height,), hidden_channels=hidden_channels, **_fno_nd_kwargs(kw))
        self.n_modes_height = n_modes_height


class FNO2d(FNO):
    """tfno.py:342-463."""

    def __init__(self, n_modes_height, n_modes_width, hidden_channels, **kw):
        super().__init__(n_modes=(n_modes_height, n_modes_width), hidden_channels=hidden_channels,
                         **_fno_nd_kwargs(kw))
        self.n_modes_height, self.n_modes_width = n_modes_height, n_modes_width


class FNO3d(FNO):
    def __init__(self, n_modes_height, n_modes_width, n_modes_depth, hidden_channels, **kw):
        super().__init__(n_modes=(n_modes_height, n_modes_width, n_modes_depth), hidden_channels=hidden_channels,
                         **_fno_nd_kwargs(kw))
        self.n_modes_height, self.n_modes_width, self.n_modes_depth = n_modes_height, n_modes_width, n_modes_depth


class FNO2dObserver(nn.Module):
    """libs/models/fno_models.py:16-57."""

    def __init__(self, modes1, modes2, width, use_v_plane=False):
        super().__init__()
        self.modes1, self.modes2, self.width, self.use_v_plane = modes1, modes2, width, use_v_plane
        self.padding = 9
        self.input_channel_num = 4 if use_v_plane else 3
        self.fno2d = FNO2d(modes1, modes2, width, in_channels=self.input_channel_num, out_channels=1)
        self._grid_cache = {}

    def get_grid(self, shape, device):
        key = (tuple(shape[:3]), str(device))
        g = self._grid_cache.get(key)
        if g is None:
            b, sx, sy = shape[0], shape[1], shape[2]
            gx = torch.tensor(np.linspace(0, 1, sx), dtype=torch.float).reshape(1, sx, 1, 1).repeat([b, 1, sy, 1])
            gy = torch.tensor(np.linspace(0, 1, sy), dtype=torch.float).reshape(1, 1, sy, 1).repeat([b, sx, 1, 1])
            g = torch.cat((gx, gy), dim=-1).to(device)
            self._grid_cache = {key: g}
        return g

    def forward(self, p_plane, v_plane=None):
        # fno_models.py:41-57 concatenates channels-LAST and permutes; the lifting kernel wants channels-first, so the
        # concatenation writes that layout directly (one copy kernel instead of cat + permute copy; same values)
        grid = self.get_grid(p_plane.shape, p_plane.device)
        cf = self._grid_cache.get("cf")
        if cf is None or cf[0] is not grid:
            cf = (grid, grid.permute(0, 3, 1, 2).contiguous())     # the constant grid channels, channels-first, made once
            self._grid_cache["cf"] = cf
        parts = [p_plane, v_plane] if self.use_v_plane else [p_plane]
        # (B, H, W, 1) -> (B, 1, H, W) is a pure reshape
        cfirst = [t.reshape(t.shape[0], 1, t.shape[1], t.shape[2]) if t.shape[-1] == 1 else t.permute(0, 3, 1, 2) for t in parts]
        return self.fno2d(torch.cat(cfirst + [cf[1]], dim=1))


class LpLoss(object):
    """libs/utilities3.py:295-337 (p=2 relative loss on the native reduction kernel)."""

    def __init__(self, d=2, p=2, size_average=True, reduction=True):
        assert d > 0 and p > 0
        if p != 2:
            raise NotImplementedError("native LpLoss implements p=2")
        self.d, self.p, self.reduction, self.size_average = d, p, reduction, size_average

    def rel(self, x, y):
        if not self.reduction:
            raise NotImplementedError("native LpLoss implements the reduced form")
        return Fn.rel_l2_loss(x, y, self.size_average)

    def __call__(self, x, y):
        return self.rel(x, y)


# =============================================================================================
# RNO family (neuralop/models/rno.py)
# =============================================================================================
class RnoSpectralConv2d(nn.Module):
    """rno.py:34-77: real-pair weights, un-halved modes, norm='ortho', FFT size (n, n)."""

    def __init__(self, in_channels, out_channels, modes1, modes2, norm="ortho"):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.modes1, self.modes2 = modes1, modes2
        scale = 1 / (in_channels * out_channels)
        self.fourier_weight = nn.ParameterList([
            nn.Parameter(torch.empty(in_channels, out_channels, modes1, modes2, 2)) for _ in range(2)])
        for param in self.fourier_weight:
            nn.init.xavier_normal_(param, gain=scale * np.sqrt(in_channels + out_channels))
        self.norm = norm

    def geom(self, grid) -> SpecGeom:
        n = grid[-1]
        if self.modes2 > n // 2 + 1 or self.modes1 > n:
            raise ValueError("modes exceed the transform size")
        return SpecGeom(nin=tuple(grid), half=(self.modes1, self.modes2), norm=self.norm, nfft=(n, n), nout=(n, n))

    def forward(self, x):
        return self.forward_fused(x)

    def forward_fused(self, x, bias=None, pw_weight=None, act=None):
        return Fn.spectral_block(x, list(self.fourier_weight), self.geom(tuple(x.shape[2:])), bias=bias,
                                 pw_weight=pw_weight, act=act)


class FourierLayer2d(nn.Module):
    """rno.py:215-228: spec_conv(x) + Conv1d(k=1)(x), fused."""

    def __init__(self, modes1, modes2, width):
        super().__init__()
        self.modes1, self.modes2, self.width = modes1, modes2, width
        self.spec_conv = RnoSpectralConv2d(width, width, modes1, modes2, norm="ortho")
        self.norm_conv1d = nn.Conv1d(width, width, 1)

    def forward(self, x, act=None, extra_bias=None):
        bias = self.norm_conv1d.bias if extra_bias is None else self.norm_conv1d.bias + extra_bias
        if x.shape[-2] != x.shape[-1]:
            y = self.spec_conv(x)
            y = y + Fn.pointwise_conv(x, self.norm_conv1d.weight, bias, None)
            return y
        return self.spec_conv.forward_fused(x, bias=bias, pw_weight=self.norm_conv1d.weight, act=act)


class RNO_cell(nn.Module):
    """rno.py:231-260."""

    def __init__(self, in_dim, out_dim, modes1, modes2, width):
        super().__init__()
        self.modes1, self.modes2, self.width, self.in_dim, self.out_dim = modes1, modes2, width, in_dim, out_dim
        for k in range(1, 9):
            setattr(self, f"f{k}", FourierLayer2d(modes1, modes2, width))
        for k in range(1, 5):
            setattr(self, f"b{k}", nn.Parameter(torch.normal(torch.tensor(0.), torch.tensor(1.))))

    def _params(self):
        ps = []
        for k in range(1, 9):
            f = getattr(self, f"f{k}")
            ps += [f.spec_conv.fourier_weight[0], f.spec_conv.fourier_weight[1], f.norm_conv1d.weight, f.norm_conv1d.bias]
        return ps + [self.b1, self.b2, self.b3, self.b4]

    def forward_sequence(self, x_tm, h, return_sequences=False):
        """x_tm: (T', B, C, H, W) time-major.  All T' recurrent steps as ONE autograd node (functional.RnoLayerFn): the
        x-dependent halves f1, f3, f5, f7 hoisted over the frames, gates batched, activations in the epilogues."""
        Tn, B, C, H, W = x_tm.shape
        geom = self.f1.spec_conv.geom((H, W))
        return Fn.rno_layer(x_tm, h, geom, return_sequences, self._params())

    def forward(self, x, h):
        if Fn.rno_layer_supported(x, x.shape[1], x.shape[2], x.shape[3]) and x.shape == h.shape:
            return self.forward_sequence(x.unsqueeze(0), h)
        # shapes without the regrouped path (non-square grids, rno.py:66-67 crop / zero-pad): the reference's composition
        z = torch.sigmoid(self.f1(x) + self.f2(h, extra_bias=self.b1))
        z2 = torch.sigmoid(self.f7(x) + self.f8(h, extra_bias=self.b4))
        r = torch.sigmoid(self.f3(x) + self.f4(h, extra_bias=self.b2))
        h_hat = F.selu(self.f5(x) + self.f6(r * h, extra_bias=self.b3))
        return Fn.rno_gate(z, z2, h_hat, h)


class RNO_layer(nn.Module):
    """rno.py:263-290."""

    def __init__(self, in_dim, out_dim, modes1, modes2, width, return_sequences=False):
        super().__init__()
        self.modes1, self.modes2, self.width = modes1, modes2, width
        self.in_dim, self.out_dim, self.return_sequences = in_dim, out_dim, return_sequences
        self.cell = RNO_cell(in_dim, out_dim, modes1, modes2, width)
        self.bias_h = nn.Parameter(torch.normal(torch.tensor(0.), torch.tensor(1.)))

    def forward(self, x, h=None, time_major=False):
        """x: (B, T', C, H, W) as in the reference, or (T', B, C, H, W) with time_major (what RNO2d passes: the frames of
        one step are then contiguous, which is what the per-step kernels want)."""
        if time_major:
            timesteps, batch_size, dim, s1, s2 = x.shape
        else:
            batch_size, timesteps, dim, s1, s2 = x.shape
        if h is None:
            h = torch.zeros((batch_size, self.width, s1, s2), device=x.device) + self.bias_h
        if Fn.rno_layer_supported(x, dim, s1, s2) and dim == self.width:
            x_tm = x if time_major else x.transpose(0, 1)
            out = self.cell.forward_sequence(x_tm, h, self.return_sequences)
            if self.return_sequences and not time_major:
                out = out.transpose(0, 1)
            return out
        outputs = []
        for i in range(timesteps):
            h = self.cell(x[i] if time_major else x[:, i], h)
            if self.return_sequences:
                outputs.append(h)
        return torch.stack(outputs, dim=0 if time_major else 1) if self.return_sequences else h


class SpectralConvWithFC(nn.Module):
    """rno.py:80-106, expressed channels-first: act(spec_conv(dropout(x)) + linear(x))."""

    def __init__(self, in_channels, out_channels, modes1, modes2, n_grid=None, dropout=0.1, norm="ortho",
                 activation="silu", return_freq=False, debug=False):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.spec_conv = RnoSpectralConv2d(in_channels, out_channels, modes1, modes2, norm)
        self.linear = nn.Linear(in_channels, out_channels)
        if activation == "silu":
            raise NotImplementedError("native SpectralConvWithFC: silu has no kernel (RNO2d uses relu, rno.py:318)")
        self.activation = nn.ReLU()
        self.dropout = nn.Dropout(dropout)
        self.return_freq = return_freq

    def forward(self, x):
        """x: (B, X, Y, C) channels-last as in the reference; returns channels-last."""
        xcf = x.permute(0, 3, 1, 2)
        if self.training and self.dropout.p > 0 or xcf.shape[-2] != xcf.shape[-1]:
            res = Fn.pointwise_conv(xcf, self.linear.weight, self.linear.bias, None)
            y = torch.relu(self.spec_conv(self.dropout(xcf)) + res)
        else:
            y = self.spec_conv.forward_fused(xcf, bias=self.linear.bias, pw_weight=self.linear.weight, act="relu")
        if self.return_freq:
            raise RuntimeError("Not supported return freq")
        return y.permute(0, 2, 3, 1)


class SpectralRegressor(nn.Module):
    """rno.py:109-212 (2-D, the configuration RNO2d builds at rno.py:317-318)."""

    def __init__(self, in_dim, n_hidden, freq_dim, out_dim, modes: int, num_spectral_layers: int = 2, n_grid=None,
                 dim_feedforward=None, spacial_fc=False, spacial_dim=2, return_freq=False, return_latent=False,
                 normalizer=None, activation="silu", last_activation=True, dropout=0.1, debug=False):
        super().__init__()
        if spacial_dim != 2 or spacial_fc or return_freq or return_latent or not last_activation:
            raise NotImplementedError("native SpectralRegressor covers the configuration RNO2d builds")
        activation = "silu" if activation is None else activation
        if activation != "relu":
            raise NotImplementedError("native SpectralRegressor: relu only (rno.py:318)")
        self.activation = nn.ReLU()
        dropout = 0.1 if dropout is None else dropout
        self.spectral_conv = nn.ModuleList([SpectralConvWithFC(n_hidden, freq_dim, modes, modes, n_grid=n_grid,
                                                               dropout=dropout, activation=activation)])
        for _ in range(num_spectral_layers - 1):
            self.spectral_conv.append(SpectralConvWithFC(freq_dim, freq_dim, modes, modes, n_grid=n_grid,
                                                         dropout=dropout, activation=activation))
        self.dim_feedforward = 2 * spacial_dim * freq_dim if dim_feedforward is None else dim_feedforward
        self.regressor = nn.Sequential(nn.Linear(freq_dim, self.dim_feedforward), self.activation,
                                       nn.Linear(self.dim_feedforward, out_dim))
        self.normalizer = normalizer

    def forward(self, x, edge=None, pos=None, grid=None):
        for layer in self.spectral_conv:
            x = layer(x)
        xcf = x.permute(0, 3, 1, 2)
        y = Fn.mlp_head(xcf, self.regressor[0].weight, self.regressor[0].bias, self.regressor[2].weight,
                        self.regressor[2].bias, "relu")
        y = y.permute(0, 2, 3, 1)
        if self.normalizer:
            y = self.normalizer.inverse_transform(y)
        return y


class RNO2d(nn.Module):
    """rno.py:293-391."""

    def __init__(self, modes1, modes2, width, recurrent_index, layer_num=3, pad_amount=None, pad_dim="1"):
        super().__init__()
        self.modes1 = modes1
        self.modes1 = modes2  # quirk Q4 (rno.py:301-302)
        self.width, self.pad_amount, self.pad_dim = width, pad_amount, pad_dim
        self.recurrent_index = recurrent_index
        self.in_dim, self.out_dim, self.layer_num = 1, 1, layer_num
        self.input_projection_layer = nn.Linear(self.in_dim, self.width)
        torch.nn.init.normal_(self.input_projection_layer.weight, mean=0, std=1)
        mods = [RNO_layer(width, width, modes1, modes2, width, return_sequences=True) for _ in range(layer_num - 1)]
        mods.append(RNO_layer(width, width, modes1, modes2, width, return_sequences=False))
        self.layers = nn.ModuleList(mods)
        self.regressor = SpectralRegressor(in_dim=width, n_hidden=width, freq_dim=width, out_dim=self.out_dim,
                                           modes=modes2, activation="relu", dropout=0.3)

    def forward_one_step(self, x, v_plane=None, init_hidden_states=None):
        if init_hidden_states is None:
            init_hidden_states = [None] * self.layer_num
        B, T, s1, s2, dim = x.shape
        # Linear(in_dim -> width) on channels-last == 1x1 conv on (T*B, in_dim, s1, s2); the frames go time-major so that
        # every recurrent step reads one contiguous (B, C, s1, s2) block
        xt = x.transpose(0, 1)
        xin = xt.reshape(T * B, dim, s1, s2) if dim == 1 else xt.permute(0, 1, 4, 2, 3).reshape(T * B, dim, s1, s2)
        xc = Fn.pointwise_conv(xin, self.input_projection_layer.weight, self.input_projection_layer.bias, None)
        x = xc.reshape(T, B, self.width, s1, s2)
        if self.pad_amount:
            if self.pad_dim == "1":
                x = F.pad(x.permute(0, 1, 2, 4, 3), [0, self.pad_amount[0]]).permute(0, 1, 2, 4, 3)
            elif self.pad_dim == "2":
                x = F.pad(x, [0, self.pad_amount[1]])
            elif self.pad_dim == "both":
                x = F.pad(x.permute(0, 1, 2, 4, 3), [0, self.pad_amount[0]]).permute(0, 1, 2, 4, 3)
                x = F.pad(x, [0, self.pad_amount[1]])
        finals = []
        for i in range(self.layer_num):
            pred_x = self.layers[i](x, init_hidden_states[i], time_major=True)
            if i < self.layer_num - 1:
                x = x + pred_x
                finals.append(x[-1])
            else:
                x = pred_x
                finals.append(x)
        h = finals[-1]
        if self.pad_amount:
            if self.pad_dim == "1":
                h = h[:, :, :-self.pad_amount[0]]
            elif self.pad_dim == "2":
                h = h[..., :-self.pad_amount[1]]
            elif self.pad_dim == "both":
                h = h[:, :, :-self.pad_amount[0]]
                h = h[..., :-self.pad_amount[1]]
        pred = self.regressor(h.permute(0, 2, 3, 1))
        return pred, finals

    def forward(self, x, v_plane=None, timestep=2):
        result = self.predict(x, num_steps=x.shape[1])
        return result[:, self.recurrent_index, :, :, :]

    def predict(self, x, num_steps):
        output, states = [], [None] * self.layer_num
        for _ in range(num_steps):
            pred, states = self.forward_one_step(x, init_hidden_states=states)
            output.append(pred)
            x = pred.reshape((pred.shape[0], 1, pred.shape[1], pred.shape[2], pred.shape[3]))
        return torch.stack(output, dim=1)

    def count_params(self):
        return int(sum(np.prod(p.size()) for p in self.parameters() if p.requires_grad))


class RNO2dObserver(RNO2d):
    """libs/models/rno_models.py:12-15."""

    def __init__(self, modes1, modes2, width, recurrent_index, layer_num=3):
        super().__init__(modes1, modes2, width, recurrent_index, layer_num=layer_num)


# =============================================================================================
# PINO family (libs/models/pino_models)
# =============================================================================================
class PinoSpectralConv3d(nn.Module):
    """basics.py:99-143: cfloat weights1..4, corner order (lo,lo),(hi,lo),(lo,hi),(hi,hi), norm 'backward'."""

    def __init__(self, in_channels, out_channels, modes1, modes2, modes3):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.modes1, self.modes2, self.modes3 = modes1, modes2, modes3
        self.scale = 1 / (in_channels * out_channels)
        for k in range(1, 5):
            setattr(self, f"weights{k}", nn.Parameter(
                self.scale * torch.rand(in_channels, out_channels, modes1, modes2, modes3, dtype=torch.cfloat)))

    def corners(self):
        return [self.weights1, self.weights3, self.weights2, self.weights4]  # canonical order

    def geom(self, grid) -> SpecGeom:
        return SpecGeom(nin=tuple(grid), half=(self.modes1, self.modes2, self.modes3), norm="backward")

    def forward(self, x):
        return self.forward_fused(x)

    def forward_fused(self, x, bias=None, pw_weight=None, act=None):
        return Fn.spectral_block(x, self.corners(), self.geom(tuple(x.shape[2:])), bias=bias,
                                 pw_weight=pw_weight, act=act)


class MultiplicativeNet(nn.Module):
    """pinobserver.py:14-63 (affine: input1 @ B^T + input2 @ A^T + bias)."""

    def __init__(self, in1_features, in2_features, out_features, device=None, dtype=None):
        super().__init__()
        self.in1_features, self.in2_features, self.out_features = in1_features, in2_features, out_features
        self.A = nn.Parameter(torch.empty(out_features, in2_features))
        self.B = nn.Parameter(torch.empty(out_features, in1_features))
        self.bias = nn.Parameter(torch.empty(out_features))
        self.reset_parameters()

    def reset_parameters(self):
        bound = 1 / math.sqrt(self.in1_features)
        nn.init.kaiming_uniform_(self.A, a=math.sqrt(5))
        nn.init.kaiming_uniform_(self.B, a=math.sqrt(5))
        nn.init.uniform_(self.bias, -bound, bound)

    def forward(self, input1, input2):
        if input2.dim() < 2:
            input2 = input2.unsqueeze(-1)
        code = torch.einsum("bj,oj->bo", input2, self.A)[:, None, None, None, :]
        return torch.einsum("bthwi,oi->bthwo", input1, self.B) + code + self.bias


_PINO_ACTS = {"gelu": "gelu", "tanh": "tanh", "relu": "relu"}


def _pino_trunk_forward(x, re, fc0, mnet1, sp_convs, ws, mnet2, fc1, fc2, act_name, pad_ratio):
    """The PINO "FNO3d" trunk shared by PINObserver2d.forward (pinobserver.py:192-233), PlanePredHead.forward under
    PINObserverFullField / PolicyModel2D (:257-273, :337-368, :433-463).  x: (B, X, Y, T, in_dim) channels-last, re: (B,) or
    (B, 1) ALREADY scaled by the caller (the full-field / policy models divide by max_re, PINObserver2d does not).
    Returns (B, X, Y, T, out_dim).

    The pointwise head (fc0 + MultiplicativeNet1 + permute + pad) is folded into ONE 1x1 conv over the channels-first
    input [x (in_dim), re, valid-mask]; every Fourier layer is one fused pass (spectral conv + Conv1d(k=1) + bias + act);
    the tail (unpad + MultiplicativeNet2 + fc1 + act + fc2) runs on the padded grid with MultiplicativeNet2 folded into
    fc1 and the Reynolds term entering as a per-sample bias (fused head kernel) or a 1-channel map."""
    re = re.float()
    B, sx, sy, sz, _ = x.shape
    if max(pad_ratio) > 0:
        num_pad = [round(sz * i) for i in pad_ratio]
    else:
        num_pad = [0, 0]
    if re.dim() < 2:
        re = re.unsqueeze(-1)
    # ---- head: fold fc0 and MultiplicativeNet1 into one (C0 x (in_dim + 2)) 1x1 conv ----
    w_in = mnet1.B @ fc0.weight                                   # (C0, in_dim)
    b_in = mnet1.B @ fc0.bias + mnet1.bias                        # (C0,)
    w6 = torch.cat([w_in, mnet1.A, b_in[:, None]], dim=1)         # (C0, in_dim + 2)
    ones = torch.ones((B, sx, sy, sz, 1), dtype=x.dtype, device=x.device)
    x6 = torch.cat([x, re.reshape(B, 1, 1, 1, 1).expand(B, sx, sy, sz, 1), ones], dim=-1)
    x6 = x6.permute(0, 4, 1, 2, 3)
    if max(num_pad) > 0:
        x6 = F.pad(x6, (num_pad[0], num_pad[1]), "constant", 0)   # zero mask => padded output is exactly 0
    h = Fn.pointwise_conv(x6.contiguous(), w6, None, None)
    # ---- Fourier layers ----
    L = len(ws)
    same = all((c.in_channels, c.out_channels, c.modes1, c.modes2, c.modes3) ==
               (sp_convs[0].in_channels, sp_convs[0].out_channels, sp_convs[0].modes1, sp_convs[0].modes2, sp_convs[0].modes3)
               for c in sp_convs) and sp_convs[0].in_channels == sp_convs[0].out_channels
    if same and L > 1:
        # equal layers (the yaml configuration): the whole stack as ONE autograd node -- its backward chains act'(z) of the
        # layer below into each dx pass (no separate activation-backward pass over the activations)
        geom = sp_convs[0].geom(tuple(h.shape[2:]))
        bias_all = torch.stack([w.bias for w in ws], dim=0)
        layers = [(w.weight, conv.corners()) for conv, w in zip(sp_convs, ws)]
        acts = [act_name if i != L - 1 else None for i in range(L)]
        h = Fn.fno_stack(h, geom, bias_all, layers, acts)
    else:
        for i, (conv, w) in enumerate(zip(sp_convs, ws)):
            h = conv.forward_fused(h, bias=w.bias, pw_weight=w.weight, act=act_name if i != L - 1 else None)
    # ---- tail: fold MultiplicativeNet2 into fc1; run on the padded grid, slice the result ----
    w1 = fc1.weight @ mnet2.B                                     # (fc_dim, C)
    wre = fc1.weight @ mnet2.A                                    # (fc_dim, 1)
    b1 = fc1.weight @ mnet2.bias + fc1.bias                       # (fc_dim,)
    szp = sz + num_pad[0] + num_pad[1]
    needs_grad = torch.is_grad_enabled() and (h.requires_grad or w1.requires_grad)
    h = h if h.is_contiguous() else h.contiguous()
    if Fn.mlp_head_fused_available(h, w1, fc2.weight, None, needs_grad):
        # fused head (training and inference, out_dim 1..4 -- PINObserverFullField emits plane_num * out_dim): the
        # per-sample bias carries the Reynolds term, the fc_dim-wide hidden tensor is never materialised in the forward;
        # autograd reaches A / B / bias of MultiplicativeNet2 and fc1 through the folded w1 / per-sample b1
        out = Fn.mlp_head(h, w1, b1[None, :] + re @ wre.t(), fc2.weight, fc2.bias, act_name)
    else:
        re_map = re.reshape(B, 1, 1, 1, 1).expand(B, 1, sx, sy, szp).contiguous()
        t = Fn.pointwise_conv2(h, w1, b1, act_name, re_map, wre)
        out = Fn.pointwise_conv(t, fc2.weight, fc2.bias, None)    # (B, out_dim, sx, sy, szp)
    if max(num_pad) > 0:
        out = out[..., num_pad[0]: szp - num_pad[1]]
    return out.permute(0, 2, 3, 4, 1)


def _pad_pair(pad_ratio):
    if isinstance(pad_ratio, float):
        return [pad_ratio, pad_ratio]
    assert len(pad_ratio) == 2, "Cannot add padding in more than 2 directions."
    return pad_ratio


class PINObserver2d(nn.Module):
    """pinobserver.py:129-233 (see _pino_trunk_forward for how the pointwise head / tail are folded)."""

    def __init__(self, modes1, modes2, modes3, width=16, fc_dim=128, layers=None, in_dim=4, out_dim=1,
                 act="gelu", pad_ratio=[0., 0.], use_fourier_layer=False):
        super().__init__()
        pad_ratio = _pad_pair(pad_ratio)
        if use_fourier_layer:
            raise NotImplementedError("native PINObserver2d: use_fourier_layer is outside the hot path")
        if act not in _PINO_ACTS:
            raise NotImplementedError(f"native PINObserver2d: act={act!r} has no kernel")
        self.pad_ratio = pad_ratio
        self.modes1, self.modes2, self.modes3 = modes1, modes2, modes3
        self.in_dim = in_dim
        self.layers = [width] * 4 if layers is None else layers
        self.fc0 = nn.Linear(in_dim, self.layers[0])
        self.use_fourier_layer = False
        self.fourier_layer1 = None
        self.multiplicative_net1 = MultiplicativeNet(self.layers[0], 1, self.layers[0])
        self.sp_convs = nn.ModuleList([PinoSpectralConv3d(i, o, m1, m2, m3) for i, o, m1, m2, m3 in
                                       zip(self.layers, self.layers[1:], modes1, modes2, modes3)])
        self.ws = nn.ModuleList([nn.Conv1d(i, o, 1) for i, o in zip(self.layers, self.layers[1:])])
        self.multiplicative_net2 = MultiplicativeNet(self.layers[-1], 1, self.layers[-1])
        self.fc1 = nn.Linear(self.layers[-1], fc_dim)
        self.fc2 = nn.Linear(fc_dim, out_dim)
        self.act_name = _PINO_ACTS[act]

    def forward(self, x, re):
        return _pino_trunk_forward(x, re, self.fc0, self.multiplicative_net1, self.sp_convs, self.ws,
                                   self.multiplicative_net2, self.fc1, self.fc2, self.act_name, self.pad_ratio)


class PlanePredHead(nn.Module):
    """pinobserver.py:236-273: the Fourier layers + fc1 / fc2 of one prediction head (parameters only; the arithmetic is
    _pino_trunk_forward, driven by the owning PINObserverFullField / PolicyModel2D)."""

    def __init__(self, layers, modes1, modes2, modes3, fc_dim, out_dim, act):
        super().__init__()
        if act not in _PINO_ACTS:
            raise NotImplementedError(f"native PlanePredHead: act={act!r} has no kernel")
        self.layers, self.modes1, self.modes2, self.modes3 = layers, modes1, modes2, modes3
        self.sp_convs = nn.ModuleList([PinoSpectralConv3d(i, o, m1, m2, m3) for i, o, m1, m2, m3 in
                                       zip(self.layers, self.layers[1:], modes1, modes2, modes3)])
        self.ws = nn.ModuleList([nn.Conv1d(i, o, 1) for i, o in zip(self.layers, self.layers[1:])])
        self.fc1 = nn.Linear(layers[-1], fc_dim)
        self.fc2 = nn.Linear(fc_dim, out_dim)
        self.act_name = _PINO_ACTS[act]


class _PinoHeadedModel(nn.Module):
    """Shared constructor of PINObserverFullField / PolicyModel2D (pinobserver.py:276-331, 378-433)."""

    def _build(self, head_name, head_out_dim, modes1, modes2, modes3, width, fc_dim, layers, in_dim, act, pad_ratio,
               use_fourier_layer):
        if use_fourier_layer:
            raise NotImplementedError(f"native {type(self).__name__}: use_fourier_layer is outside the hot path")
        self.pad_ratio = _pad_pair(pad_ratio)
        self.modes1, self.modes2, self.modes3 = modes1, modes2, modes3
        self.max_re = 1000
        self.in_dim = in_dim
        self.layers = [width] * 4 if layers is None else layers
        self.fc0 = nn.Linear(in_dim, self.layers[0])
        self.use_fourier_layer = False
        self.fourier_layer1 = None
        self.multiplicative_net1 = MultiplicativeNet(self.layers[0], 1, self.layers[0])
        self.multiplicative_net2 = MultiplicativeNet(self.layers[-1], 1, self.layers[-1])
        setattr(self, head_name, PlanePredHead(self.layers, modes1, modes2, modes3, fc_dim, head_out_dim, act))

    def _trunk(self, head, x, re):
        return _pino_trunk_forward(x, re.float() / self.max_re, self.fc0, self.multiplicative_net1, head.sp_convs, head.ws,
                                   self.multiplicative_net2, head.fc1, head.fc2, head.act_name, self.pad_ratio)


class PINObserverFullField(_PinoHeadedModel):
    """pinobserver.py:276-375: the shared trunk with ONE head emitting plane_num * out_dim channels; re / max_re."""

    def __init__(self, plane_num, modes1, modes2, modes3, width=16, fc_dim=128, layers=None, in_dim=4, out_dim=1,
                 act="gelu", pad_ratio=[0., 0.], use_fourier_layer=False):
        super().__init__()
        self.plane_num = plane_num
        self._build("observer_head", out_dim * plane_num, modes1, modes2, modes3, width, fc_dim, layers, in_dim, act,
                    pad_ratio, use_fourier_layer)

    def forward(self, x, re):
        return self._trunk(self.observer_head, x, re).permute(0, 4, 1, 2, 3)      # (B, planes, X, Y, T)


class PolicyModel2D(_PinoHeadedModel):
    """pinobserver.py:378-463: the policy network of the gradient-through-observer control loop (run_control.py:162-185);
    every parameter starts at zero (:432-433)."""

    def __init__(self, modes1, modes2, modes3, width=16, fc_dim=128, layers=None, in_dim=4, out_dim=1, act="gelu",
                 pad_ratio=[0., 0.], use_fourier_layer=False):
        super().__init__()
        self._build("pred_net", out_dim, modes1, modes2, modes3, width, fc_dim, layers, in_dim, act, pad_ratio,
                    use_fourier_layer)
        for param in self.parameters():
            nn.init.zeros_(param)

    def forward(self, x, re):
        return self._trunk(self.pred_net, x, re)


# ---------------------------------------------------------------------------------------------
# libs/models/pino_models/{basics.SpectralConv2d, fourier2d.FNO2d}
# ---------------------------------------------------------------------------------------------
class PinoSpectralConv2d(nn.Module):
    """basics.py:64-96: cfloat weights1 (low rows) / weights2 (high rows), un-halved modes, norm 'backward'."""

    def __init__(self, in_channels, out_channels, modes1, modes2):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.modes1, self.modes2 = modes1, modes2
        self.scale = 1 / (in_channels * out_channels)
        for k in (1, 2):
            setattr(self, f"weights{k}", nn.Parameter(
                self.scale * torch.rand(in_channels, out_channels, modes1, modes2, dtype=torch.cfloat)))

    def corners(self):
        return [self.weights1, self.weights2]

    def geom(self, grid) -> SpecGeom:
        return SpecGeom(nin=tuple(grid), half=(self.modes1, self.modes2), norm="backward")

    def forward(self, x):
        return self.forward_fused(x)

    def forward_fused(self, x, bias=None, pw_weight=None, act=None):
        return Fn.spectral_block(x, self.corners(), self.geom(tuple(x.shape[2:])), bias=bias, pw_weight=pw_weight, act=act)


class PinoFNO2d(nn.Module):
    """libs/models/pino_models/fourier2d.py:6-87 (the class is called FNO2d there; exported here as PinoFNO2d because the
    neuralop FNO2d of tfno.py has that name in this package).  fc0 -> two-sided zero padding of both axes -> n x (spectral
    conv + Conv1d(k=1) + act, fused) -> unpad -> fc1, act, fc2, act, fc3."""

    def __init__(self, modes1, modes2, width=64, fc_dim=128, layers=None, in_dim=3, out_dim=1, act="gelu",
                 pad_ratio=[0., 0.]):
        super().__init__()
        if isinstance(pad_ratio, float):
            pad_ratio = [pad_ratio, pad_ratio]
        else:
            assert len(pad_ratio) == 2, "Cannot add padding in more than 2 directions"
        if act not in _PINO_ACTS:
            raise NotImplementedError(f"native PinoFNO2d: act={act!r} has no kernel")
        self.modes1, self.modes2, self.pad_ratio = modes1, modes2, pad_ratio
        self.layers = [width] * (len(modes1) + 1) if layers is None else layers
        self.fc0 = nn.Linear(in_dim, self.layers[0])
        self.sp_convs = nn.ModuleList([PinoSpectralConv2d(i, o, m1, m2) for i, o, m1, m2 in
                                       zip(self.layers, self.layers[1:], modes1, modes2)])
        self.ws = nn.ModuleList([nn.Conv1d(i, o, 1) for i, o in zip(self.layers, self.layers[1:])])
        self.fc1 = nn.Linear(self.layers[-1], fc_dim)
        self.fc2 = nn.Linear(fc_dim, self.layers[-1])
        self.fc3 = nn.Linear(self.layers[-1], out_dim)
        self.act_name = _PINO_ACTS[act]

    def forward(self, x):
        s1, s2 = x.shape[1], x.shape[2]
        if max(self.pad_ratio) > 0:
            p1 = [round(i * s1) for i in self.pad_ratio]
            p2 = [round(i * s2) for i in self.pad_ratio]
        else:
            p1 = p2 = [0, 0]
        h = Fn.pointwise_conv(x.permute(0, 3, 1, 2), self.fc0.weight, self.fc0.bias, None)
        padded = max(p1) > 0 or max(p2) > 0
        if padded:
            h = F.pad(h, (p2[0], p2[1], p1[0], p1[1]), "constant", 0.)
        L = len(self.ws)
        for i, (conv, w) in enumerate(zip(self.sp_convs, self.ws)):
            h = conv.forward_fused(h, bias=w.bias, pw_weight=w.weight, act=self.act_name if i != L - 1 else None)
        if padded:
            # remove_padding2 (utils.py:28-33) slices [p[0]:-p[1]]: with p[1] == 0 that is an EMPTY slice in the reference;
            # mirrored literally so that a mis-configured pad_ratio fails the same way
            h = h[..., p1[0]:-p1[1], p2[0]:-p2[1]]
        h = Fn.pointwise_conv(h, self.fc1.weight, self.fc1.bias, self.act_name)
        h = Fn.pointwise_conv(h, self.fc2.weight, self.fc2.bias, self.act_name)
        h = Fn.pointwise_conv(h, self.fc3.weight, self.fc3.bias, None)
        return h.permute(0, 2, 3, 1)
