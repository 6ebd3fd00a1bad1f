"""TEST INFRASTRUCTURE ONLY -- float64 closed-form oracle for the truncated spectral convolution.

This is the CPU restatement (SURVEY.md section 8a.0) of what the three reference spectral
convolutions compute:

  * neuralop/models/spectral_convolution.py:303-347   FactorizedSpectralConv.forward   (a1)
  * neuralop/models/rno.py:60-77                      SpectralConv2d.forward           (a4)
  * libs/models/pino_models/basics.py:114-143         SpectralConv3d.forward           (a6)

All three are  rfftn -> keep low modes -> per-mode channel mixing -> irfftn.  Here the same map is
written as explicit mode-restricted DFT matrices in complex128, together with the hand-derived
backward (dx, dW, dbias).  It is the *specification* the CUDA kernels are tested against; it is
pinned against the reference itself (tests/test_oracle_vs_reference.py, run where B2NO_REFERENCE_ROOT
names a checkout of it) and against the committed fixtures in tests/golden/ (generated from the reference by
tests/golden/make_golden.py).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this module; the
product path (pde_policylearning_b200) never does.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Sequence, Tuple

import torch

CD = torch.complex128
RD = torch.float64


@dataclass
class SpecGeom:
    """Geometry of one truncated spectral convolution.

    nin   : physical input grid (x.shape[2:])
    nfft  : forward transform lengths (== nin except rno.py:66-67 which forces (n, n))
    nout  : output grid (== nfft except FactorizedSpectralConv output_scaling_factor,
            spectral_convolution.py:339-342)
    half  : kept modes per dim.  Two-sided dims keep rows [0,h) U [N-h,N); the last dim keeps [0,h).
    norm  : 'forward' | 'backward' | 'ortho'
    """
    nin: Tuple[int, ...]
    half: Tuple[int, ...]
    norm: str = "backward"
    nfft: Tuple[int, ...] = None
    nout: Tuple[int, ...] = None

    def __post_init__(self):
        self.nin = tuple(int(v) for v in self.nin)
        self.half = tuple(int(v) for v in self.half)
        self.nfft = tuple(self.nin) if self.nfft is None else tuple(int(v) for v in self.nfft)
        self.nout = tuple(self.nfft) if self.nout is None else tuple(int(v) for v in self.nout)
        assert len(self.nin) == len(self.half) == len(self.nfft) == len(self.nout)
        for j in range(self.ndim - 1):
            assert self.half[j] <= self.nfft[j], "two-sided kept modes exceed the grid"

    @property
    def ndim(self):
        return len(self.nin)

    # ---- kept frequency rows -----------------------------------------------------------------
    def rows(self, j: int) -> List[Tuple[int, int, int]]:
        """For dim j: list of (frequency index f, corner bit, local weight index), in spectrum order.
        If 2h > N the high corner overwrites the low one on the overlap (assignment order
        spectral_convolution.py:412-416, rno.py:71-74, basics.py:127-139)."""
        N, h = self.nfft[j], self.half[j]
        if j == self.ndim - 1:
            return [(k, 0, k) for k in range(h)]
        out = []
        for f in sorted(set(range(0, h)) | set(range(N - h, N))):
            if f >= N - h:
                out.append((f, 1, f - (N - h)))
            else:
                out.append((f, 0, f))
        return out

    def kept(self) -> Tuple[int, ...]:
        return tuple(len(self.rows(j)) for j in range(self.ndim))

    # ---- scales -------------------------------------------------------------------------------
    def scales(self) -> Tuple[float, float]:
        n = math.prod(self.nfft)
        npr = math.prod(self.nout)
        if self.norm == "forward":
            return 1.0 / n, 1.0
        if self.norm == "backward":
            return 1.0, 1.0 / npr
        if self.norm == "ortho":
            return 1.0 / math.sqrt(n), 1.0 / math.sqrt(npr)
        raise ValueError(self.norm)

    # ---- DFT matrices -------------------------------------------------------------------------
    def fwd_matrix(self, j: int) -> torch.Tensor:
        """E[n, k] = exp(-2 pi i f_k n / N) for n < min(nin, nfft) (zero rows beyond the transform
        length = cropping; missing rows = zero padding), shape (nin_j, K_j).  For the last dim,
        modes >= N/2+1 do not exist in the rfft output and read as zero (basics.py:119,126)."""
        N, nin = self.nfft[j], self.nin[j]
        rows = self.rows(j)
        n = torch.arange(nin, dtype=RD).unsqueeze(1)
        f = torch.tensor([r[0] for r in rows], dtype=RD).unsqueeze(0)
        E = torch.exp(-2j * math.pi * (n * f / N).to(CD))
        E = E * (n < N).to(CD)
        if j == self.ndim - 1:
            E = E * (f < (N // 2 + 1)).to(CD)
        return E

    def inv_matrix(self, j: int) -> torch.Tensor:
        """G[k, n] = c(k) exp(+2 pi i f_k n / N') on the output grid N' (c == 1 except on the last dim),
        shape (K_j, nout_j).  irfftn(s=N') trims / zero-pads the spectrum at the END of each axis, so a
        kept row with f >= N' (two-sided) or f >= N'/2+1 (last dim) is dropped."""
        Np = self.nout[j]
        rows = self.rows(j)
        n = torch.arange(Np, dtype=RD).unsqueeze(0)
        f = torch.tensor([r[0] for r in rows], dtype=RD).unsqueeze(1)
        G = torch.exp(2j * math.pi * (f * n / Np).to(CD))
        if j == self.ndim - 1:
            c = torch.full_like(f, 2.0)
            c[f == 0] = 1.0
            if Np % 2 == 0:
                c[f == Np // 2] = 1.0
            c[f >= Np // 2 + 1] = 0.0
            # modes beyond the *input* rfft length never existed either
            c[f >= self.nfft[j] // 2 + 1] = 0.0
            G = G * c.to(CD)
        else:
            G = G * (f < Np).to(CD)
        return G


# ---------------------------------------------------------------------------------------------
# weights: corners -> effective tensor over the kept grid, and back
# ---------------------------------------------------------------------------------------------
def gather_weight(geom: SpecGeom, corners: Sequence[torch.Tensor]) -> torch.Tensor:
    """corners: 2^(d-1) complex tensors (Ci, Co, h_1..h_d) in canonical order -- corner index =
    sum_j bit_j * 2^(d-2-j) over the two-sided dims (== itertools.product order of
    spectral_convolution.py:330-337).  Returns W_eff (Ci, Co, K_1..K_d) complex128."""
    d = geom.ndim
    Ci, Co = corners[0].shape[:2]
    K = geom.kept()
    W = torch.zeros((Ci, Co) + K, dtype=CD)
    rows = [geom.rows(j) for j in range(d)]
    import itertools
    for idx in itertools.product(*[range(k) for k in K[:-1]]):
        cidx = 0
        loc = []
        for j, kk in enumerate(idx):
            _, bit, l = rows[j][kk]
            cidx = cidx * 2 + bit
            loc.append(l)
        src = corners[cidx].to(CD)
        W[(slice(None), slice(None)) + idx] = src[(slice(None), slice(None)) + tuple(loc)][..., : K[-1]]
    return W


def scatter_weight_grad(geom: SpecGeom, dW_eff: torch.Tensor, corner_shapes) -> List[torch.Tensor]:
    d = geom.ndim
    K = geom.kept()
    rows = [geom.rows(j) for j in range(d)]
    out = [torch.zeros(s, dtype=CD) for s in corner_shapes]
    import itertools
    for idx in itertools.product(*[range(k) for k in K[:-1]]):
        cidx = 0
        loc = []
        for j, kk in enumerate(idx):
            _, bit, l = rows[j][kk]
            cidx = cidx * 2 + bit
            loc.append(l)
        out[cidx][(slice(None), slice(None)) + tuple(loc)][..., : K[-1]] = dW_eff[(slice(None), slice(None)) + idx]
    return out


# ---------------------------------------------------------------------------------------------
# separable transforms
# ---------------------------------------------------------------------------------------------
def _apply_along(t: torch.Tensor, M: torch.Tensor, axis: int) -> torch.Tensor:
    """out[..., m, ...] = sum_j t[..., j, ...] * M[j, m] along `axis`."""
    t = t.movedim(axis, -1)
    out = t @ M
    return out.movedim(-1, axis)


def dft_trunc(geom: SpecGeom, x: torch.Tensor, scale: float, use_inv_conj: bool = False) -> torch.Tensor:
    """Truncated forward DFT  Xh[b,c,k] = scale * sum_n x[b,c,n] exp(-2 pi i k.n/N).
    use_inv_conj=True uses conj(inv_matrix)^T instead (the adjoint of the inverse: output grid N',
    includes the c(k) doubling) -- this is the gYh transform of the backward."""
    t = x.to(CD)
    d = geom.ndim
    for j in range(d - 1, -1, -1):
        M = geom.inv_matrix(j).conj().transpose(0, 1) if use_inv_conj else geom.fwd_matrix(j)
        t = _apply_along(t, M, 2 + j)
    return t * scale


def idft_trunc(geom: SpecGeom, Yh: torch.Tensor, scale: float, use_fwd_conj: bool = False) -> torch.Tensor:
    """y[b,o,n] = scale * Re( sum_k c(k_d) Yh[b,o,k] exp(+2 pi i k.n/N') ).
    use_fwd_conj=True uses conj(fwd_matrix)^T (adjoint of the forward: input grid, no c(k))."""
    t = Yh.to(CD)
    d = geom.ndim
    for j in range(d):
        M = geom.fwd_matrix(j).conj().transpose(0, 1) if use_fwd_conj else geom.inv_matrix(j)
        t = _apply_along(t, M, 2 + j)
    return t.real * scale


def spectral_conv_forward(geom: SpecGeom, x: torch.Tensor, corners: Sequence[torch.Tensor], bias=None):
    """Returns (y, Xh, Yh) in float64/complex128."""
    sf, si = geom.scales()
    W = gather_weight(geom, corners)
    Xh = dft_trunc(geom, x, sf)
    Yh = torch.einsum("bi...,io...->bo...", Xh, W)
    y = idft_trunc(geom, Yh, si)
    if bias is not None:
        y = y + bias.to(RD).reshape((1, -1) + (1,) * geom.ndim)
    return y, Xh, Yh


def spectral_conv_backward(geom: SpecGeom, x, corners, gy, has_bias=False):
    """Hand-derived backward (SURVEY.md 8a.0).  Returns dx, [dW corners] (complex, PyTorch
    conj-gradient convention: for real-pair storage dW_re = Re, dW_im = Im), dbias."""
    sf, si = geom.scales()
    W = gather_weight(geom, corners)
    Xh = dft_trunc(geom, x, sf)
    gYh = dft_trunc(geom, gy, si, use_inv_conj=True)
    gXh = torch.einsum("bo...,io...->bi...", gYh, W.conj())
    dx = idft_trunc(geom, gXh, sf, use_fwd_conj=True)
    dW_eff = torch.einsum("bi...,bo...->io...", Xh.conj(), gYh)
    dW = scatter_weight_grad(geom, dW_eff, [tuple(c.shape) for c in corners])
    db = gy.to(RD).sum(dim=[0] + list(range(2, gy.ndim))) if has_bias else None
    return dx, dW, db


# ---------------------------------------------------------------------------------------------
# geometry helpers mirroring the three reference classes
# ---------------------------------------------------------------------------------------------
def geom_neuralop(grid, n_modes, fft_norm="forward", output_scaling=None) -> SpecGeom:
    """FactorizedSpectralConv: half = n_modes // 2 for EVERY dim incl. the last
    (spectral_convolution.py:202,290,330)."""
    half = tuple(m // 2 for m in n_modes)
    nout = None
    if output_scaling is not None:
        nout = tuple(int(round(s * r)) for s, r in zip(grid, output_scaling))
    return SpecGeom(nin=tuple(grid), half=half, norm=fft_norm, nout=nout)


def geom_rno(grid, modes1, modes2) -> SpecGeom:
    """rno.SpectralConv2d: un-halved modes, norm='ortho', FFT size (n, n), n = x.shape[-1]
    (rno.py:35,66-67,76)."""
    n = grid[-1]
    return SpecGeom(nin=tuple(grid), half=(modes1, modes2), norm="ortho", nfft=(n, n), nout=(n, n))


def geom_pino3d(grid, m1, m2, m3) -> SpecGeom:
    """basics.SpectralConv3d: un-halved modes, default rfftn norm ('backward') (basics.py:117,142)."""
    return SpecGeom(nin=tuple(grid), half=(m1, m2, m3), norm="backward")


def pino_corners_to_canonical(w1, w2, w3, w4):
    """basics.py:125-139: weights1=(lo,lo) weights2=(hi,lo) weights3=(lo,hi) weights4=(hi,hi) on (x,y);
    canonical order is (lo,lo),(lo,hi),(hi,lo),(hi,hi)."""
    return [w1, w3, w2, w4]


def rno_pairs_to_complex(w: torch.Tensor) -> torch.Tensor:
    """rno.py:43-46 real pairs (Ci,Co,m1,m2,2) -> complex."""
    return torch.view_as_complex(w.detach().to(RD).contiguous())


def rel_l2(a: torch.Tensor, b: torch.Tensor) -> float:
    a = a.detach().to(RD if not a.is_complex() else CD).cpu()
    b = b.detach().to(RD if not b.is_complex() else CD).cpu()
    den = torch.linalg.vector_norm(b).item()
    num = torch.linalg.vector_norm(a - b).item()
    return num / den if den > 0 else num
