"""ctypes binding of libb2no.so (include/b2no.h).  No torch types cross this boundary: only raw device
pointers, sizes and a cudaStream_t.  There is no fallback: if the shared library is missing or a call
fails, we raise."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
# B2NO_LIB: load another build, e.g. the parent commit's, for A/B runs in one call
LIB_PATH = os.environ.get("B2NO_LIB") or os.path.join(_HERE, "libb2no.so")
CSRC = os.path.join(_HERE, "csrc")
SOURCES = ["plan.cu", "spectral.cu", "pointwise.cu", "tc_pointwise.cu", "tc_wgrad.cu", "tc_mlp.cu", "tc_head_bwd.cu", "tc_dft.cu", "tc_mix.cu", "tc_peak.cu", "pino_loss.cu", "optim.cu", "spec_norm.cu", "tc_channel_mlp.cu"]

MAX_DIM = 3
NORM = {"backward": 0, "forward": 1, "ortho": 2}
ACT = {None: 0, "none": 0, "identity": 0, "gelu": 1, "relu": 2, "sigmoid": 3, "selu": 4, "tanh": 5}


class Geom(C.Structure):
    _fields_ = [("ndim", C.c_int32), ("nin", C.c_int32 * MAX_DIM), ("nfft", C.c_int32 * MAX_DIM),
                ("nout", C.c_int32 * MAX_DIM), ("half", C.c_int32 * MAX_DIM), ("norm", C.c_int32),
                ("spec_layout", C.c_int32)]


class Weights(C.Structure):
    _fields_ = [("corner", C.c_void_p * 4), ("stride_i", C.c_int64), ("stride_o", C.c_int64),
                ("stride_k", C.c_int64 * MAX_DIM)]


class Epilogue(C.Structure):
    _fields_ = [("bias", C.c_void_p),
                ("pw_w", C.c_void_p), ("pw_x", C.c_void_p), ("pw_ci", C.c_int32), ("pw_transposed", C.c_int32),
                ("pw2_w", C.c_void_p), ("pw2_x", C.c_void_p), ("pw2_ci", C.c_int32), ("pw2_transposed", C.c_int32),
                ("add", C.c_void_p), ("mul", C.c_void_p), ("preact", C.c_void_p), ("act", C.c_int32),
                ("dact_z", C.c_void_p), ("dact", C.c_int32),
                ("gate_z", C.c_void_p), ("gate_h", C.c_void_p), ("mul_bstride", C.c_int64), ("gate_bstride", C.c_int64)]


NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "tc.cuh"), os.path.join(_HERE, "..", "include", "b2no.h")]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libb2no.so (in-tree, so it travels with the repo snapshot).  Each source becomes
    an object under csrc/_build/ (rebuilt only when it or a header changed; the compiles run in parallel), then one link."""
    from concurrent.futures import ThreadPoolExecutor
    hdr_time = max(os.path.getmtime(h) for h in HEADERS)
    if not force and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= max(
            [hdr_time] + [os.path.getmtime(os.path.join(CSRC, s)) for s in SOURCES]):
        return LIB_PATH                      # e.g. on the GPU box: the shipped .so is newer than every source
    bdir = os.path.join(CSRC, "_build")
    os.makedirs(bdir, exist_ok=True)
    jobs, objs = [], []
    for s in SOURCES:
        src, obj = os.path.join(CSRC, s), os.path.join(bdir, s[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_time):
            jobs.append(["nvcc"] + NVCC_FLAGS + ["-c", "-o", obj, src])
    if not jobs and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(o) for o in objs):
        return LIB_PATH

    def run(cmd):
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(run, jobs))
    run(["nvcc"] + NVCC_FLAGS + ["-shared", "-o", LIB_PATH] + objs)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU / PyTorch fallback for the spectral-conv hot path.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.b2no_version.restype = i32
    L.b2no_error_string.restype = C.c_char_p
    L.b2no_error_string.argtypes = [i32]
    L.b2no_device_info.argtypes = [C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i64)]
    L.b2no_plan_create.argtypes = [C.POINTER(Geom), C.POINTER(vp)]
    L.b2no_plan_destroy.argtypes = [vp]
    L.b2no_plan_kept.argtypes = [vp, C.POINTER(C.c_int32 * MAX_DIM)]
    L.b2no_plan_layout_supported.argtypes = [vp, i64, i64]
    L.b2no_plan_workspace_floats.restype = i64
    L.b2no_plan_workspace_floats.argtypes = [vp, i64, i64]
    L.b2no_set_tensor_core_mode.argtypes = [i32]
    L.b2no_set_precision.argtypes = [i32]
    L.b2no_tensor_core_launches.restype = i64
    L.b2no_kernel_launches.restype = i64
    L.b2no_dft_forward.argtypes = [vp, i32, vp, vp, vp, i64, vp]
    L.b2no_dft_inverse.argtypes = [vp, i32, vp, vp, vp, i32, i32, i64, C.POINTER(Epilogue), vp]
    L.b2no_mix.argtypes = [vp, i32, vp, C.POINTER(Weights), vp, i32, i32, i32, i32, vp]
    L.b2no_mix_dw.argtypes = [vp, vp, vp, C.POINTER(Weights), i32, i32, i32, i32, vp]
    L.b2no_act_bwd.argtypes = [vp, vp, vp, i64, i32, vp]
    L.b2no_spec_norm_fwd.argtypes = [vp, vp, vp, vp, vp, C.c_float, vp, vp, i32, i32, i32, vp]
    L.b2no_spec_norm_bwd_scratch_floats.restype = i64
    L.b2no_spec_norm_bwd_scratch_floats.argtypes = [i32, i32]
    L.b2no_spec_norm_bwd.argtypes = [vp] * 10 + [i32, i32, i32, vp]
    L.b2no_pw_wgrad_scratch_floats.restype = i64
    L.b2no_pw_wgrad_scratch_floats.argtypes = [i32, i32]
    L.b2no_pw_wgrad.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i64, vp]
    L.b2no_dft_inverse_wgrad.argtypes = [vp, i32, vp, vp, vp, i32, i32, i64, C.POINTER(Epilogue), vp, i32, vp, vp, vp, vp]
    L.b2no_mlp_head_fwd.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i64, i32, i32, vp]
    L.b2no_mlp_head_bwd_supported.argtypes = [i32, i32, i64]
    L.b2no_mlp_head_bwd_scratch_floats.restype = i64
    L.b2no_mlp_head_bwd_scratch_floats.argtypes = [i32]
    L.b2no_mlp_head_bwd.argtypes = [vp] * 9 + [i32, i32, i32, i64, i32, i32, vp, i32, vp]
    L.b2no_mlp_head_bwd_fused_supported.argtypes = [i32, i32, i64]
    L.b2no_mlp_head_bwd_fused_scratch_floats.restype = i64
    L.b2no_mlp_head_bwd_fused_scratch_floats.argtypes = [i32, i32]
    L.b2no_mlp_head_bwd_fused.argtypes = [vp] * 8 + [i32, i32, i32, i64, i32, vp, i32, vp]
    L.b2no_mlp_head_fwd_multi.argtypes = [vp] * 6 + [i32, i32, i32, i32, i64, i32, i32, vp]
    L.b2no_mlp_head_bwd_multi_supported.argtypes = [i32, i32, i32, i64]
    L.b2no_mlp_head_bwd_multi_scratch_floats.restype = i64
    L.b2no_mlp_head_bwd_multi_scratch_floats.argtypes = [i32, i32]
    L.b2no_mlp_head_bwd_multi.argtypes = [vp] * 9 + [i32, i32, i32, i32, i64, i32, i32, vp, i32, vp]
    L.b2no_channel_mlp_supported.argtypes = [i32, i32, i64]
    L.b2no_channel_mlp_fwd.argtypes = [vp] * 9 + [i32, i32, i32, i64, i32, vp]
    L.b2no_channel_mlp_scratch_floats.restype = i64
    L.b2no_channel_mlp_scratch_floats.argtypes = [i32]
    L.b2no_channel_mlp_bwd.argtypes = [vp] * 16 + [i32, i32, i32, i64, i32, vp]
    L.b2no_rno_gate_fwd.argtypes = [vp, vp, vp, vp, vp, i64, vp]
    L.b2no_rno_gate_bwd.argtypes = [vp] * 9 + [i64, vp]
    L.b2no_rno_cell_bwd.argtypes = [vp] * 7 + [i32, i32, i64, vp]
    L.b2no_rno_reset_bwd.argtypes = [vp] * 5 + [i64, vp]
    L.b2no_rel_l2_sums.argtypes = [vp, vp, vp, i32, i64, vp]
    L.b2no_rel_l2_bwd.argtypes = [vp, vp, vp, vp, i32, i64, vp]
    L.b2no_rel_l2_finish.argtypes = [vp, vp, vp, i32, i32, vp]
    L.b2no_rel_l2_bwd_g.argtypes = [vp, vp, vp, vp, vp, i32, i64, vp]
    L.b2no_gather_segments.argtypes = [vp, vp, vp, vp, i32, vp]
    f32 = C.c_float
    L.b2no_adam_step.argtypes = [vp, vp, vp, vp, i64, vp, f32, f32, f32, f32, f32, f32, vp]
    L.b2no_pino_residual_scratch_floats.restype = i64
    L.b2no_pino_residual_scratch_floats.argtypes = [i32, i32, i32, i32]
    L.b2no_pino_residual_fwd.argtypes = [vp, vp, vp, vp, f32, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    L.b2no_pino_residual_bwd.argtypes = [vp, vp, vp, vp, f32, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    L.b2no_tc_peak_probe.argtypes = [i32, i32, C.POINTER(C.c_double), vp]
    for name in EXPORTS:
        getattr(L, name)
    _lib = L
    return L


EXPORTS = [
    "b2no_version", "b2no_error_string", "b2no_device_info",
    "b2no_plan_create", "b2no_plan_destroy", "b2no_plan_kept", "b2no_plan_layout_supported", "b2no_plan_workspace_floats",
    "b2no_set_tensor_core_mode", "b2no_set_precision", "b2no_tensor_core_launches", "b2no_kernel_launches",
    "b2no_dft_forward", "b2no_dft_inverse", "b2no_mix", "b2no_mix_dw",
    "b2no_spec_norm_fwd", "b2no_spec_norm_bwd_scratch_floats", "b2no_spec_norm_bwd",
    "b2no_act_bwd", "b2no_pw_wgrad_scratch_floats", "b2no_pw_wgrad", "b2no_dft_inverse_wgrad", "b2no_mlp_head_fwd", "b2no_mlp_head_bwd_scratch_floats", "b2no_mlp_head_bwd_supported", "b2no_mlp_head_bwd",
    "b2no_mlp_head_bwd_fused_scratch_floats", "b2no_mlp_head_bwd_fused_supported", "b2no_mlp_head_bwd_fused",
    "b2no_mlp_head_fwd_multi", "b2no_mlp_head_bwd_multi_supported", "b2no_mlp_head_bwd_multi_scratch_floats",
    "b2no_mlp_head_bwd_multi",
    "b2no_channel_mlp_supported", "b2no_channel_mlp_fwd", "b2no_channel_mlp_scratch_floats", "b2no_channel_mlp_bwd",
    "b2no_rno_gate_fwd", "b2no_rno_gate_bwd", "b2no_rno_cell_bwd", "b2no_rno_reset_bwd", "b2no_rel_l2_sums", "b2no_rel_l2_bwd",
    "b2no_rel_l2_finish", "b2no_rel_l2_bwd_g", "b2no_adam_step", "b2no_gather_segments",
    "b2no_tc_peak_probe", "b2no_pino_residual_scratch_floats", "b2no_pino_residual_fwd", "b2no_pino_residual_bwd",
]


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib().b2no_error_string(int(code)).decode()
        raise RuntimeError(f"b2no {what} failed: {msg} (code {code})")
