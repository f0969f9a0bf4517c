"""ctypes binding of libb200forge.so — the C ABI declared in include/b200forge.h.

The library is the product: there is no Python/PyTorch fallback behind these calls.  `load()`
raises if the shared object is missing, and every wrapper raises `B200Error` on a non-zero
return code (with the library's own message).
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200FORGE_LIB") or os.path.join(_HERE, "libb200forge.so")  # override: instrumented builds
CSRC_DIR = os.path.join(_HERE, "csrc")

B200_F16, B200_BF16 = 0, 1
EPI_NONE, EPI_SILU, EPI_GEGLU, EPI_GELU, EPI_GELU_TANH = 0, 1, 2, 3, 4
STEP_EULER, STEP_DPMPP_2M, STEP_LINEAR = 0, 1, 2
E_UNSUPPORTED = -2


class B200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libb200forge error {code}: {msg}")
        self.code = code


class GemmDesc(C.Structure):
    _fields_ = [
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("lda", C.c_int), ("ldb", C.c_int), ("ldc", C.c_int),
        ("dtype", C.c_int), ("epilogue", C.c_int), ("block_n", C.c_int),
        ("bias", C.c_void_p), ("bias_along_m", C.c_int),
        ("residual", C.c_void_p), ("ldr", C.c_int),
        ("rowvec", C.c_void_p), ("ld_rowvec", C.c_int), ("rows_per_vec", C.c_int),
        ("A2", C.c_void_p), ("lda2", C.c_int), ("K1", C.c_int),
        ("ln_stats", C.c_void_p), ("ln_stats_parts", C.c_int), ("ln_c", C.c_void_p), ("ln_d", C.c_void_p), ("ln_eps", C.c_float),
        ("row_stats_out", C.c_void_p),
        ("B2", C.c_void_p), ("bias2", C.c_void_p), ("rowvec2", C.c_void_p),
        ("seg_period", C.c_int), ("seg_split", C.c_int), ("rowvec_mul", C.c_int), ("act_col0", C.c_int),
        ("alpha", C.c_float),
        ("workspace", C.c_void_p),
    ]


class Conv3x3Desc(C.Structure):
    _fields_ = [
        ("N", C.c_int), ("H", C.c_int), ("W", C.c_int),
        ("C1", C.c_int), ("C2", C.c_int), ("Cout", C.c_int),
        ("dtype", C.c_int), ("epilogue", C.c_int), ("block_n", C.c_int),
        ("bias", C.c_void_p), ("residual", C.c_void_p), ("ldr", C.c_int),
        ("temb", C.c_void_p), ("ld_temb", C.c_int),
        ("workspace", C.c_void_p),
    ]


class AttnDesc(C.Structure):
    _fields_ = [
        ("B", C.c_int), ("H", C.c_int), ("Lq", C.c_int), ("Lk", C.c_int), ("Dh", C.c_int),
        ("q_stride_b", C.c_longlong), ("q_stride_l", C.c_longlong),
        ("k_stride_b", C.c_longlong), ("k_stride_l", C.c_longlong),
        ("v_stride_b", C.c_longlong), ("v_stride_l", C.c_longlong),
        ("o_stride_b", C.c_longlong), ("o_stride_l", C.c_longlong),
        ("scale", C.c_float), ("dtype", C.c_int),
    ]


class GnDesc(C.Structure):
    _fields_ = [
        ("N", C.c_int), ("HW", C.c_int), ("C1", C.c_int), ("C2", C.c_int),
        ("groups", C.c_int), ("eps", C.c_float), ("silu", C.c_int), ("dtype", C.c_int),
    ]


class StepDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int), ("B", C.c_int), ("C", C.c_int), ("H", C.c_int), ("W", C.c_int),
        ("ld_eps", C.c_int), ("has_uncond", C.c_int), ("prediction", C.c_int),
        ("sigma", C.c_float), ("cfg_scale", C.c_float), ("dt", C.c_float), ("noise_scale", C.c_float),
        ("c_x", C.c_float), ("c_d", C.c_float), ("c_old", C.c_float), ("eps_dtype", C.c_int),
    ]


_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/b200forge.h one to one
SIGNATURES = {
    "b200_version": (_i, []),
    "b200_last_error": (C.c_char_p, []),
    "b200_device_ok": (_i, []),
    "b200_num_sms": (_i, []),
    "b200_gemm": (_i, [_vp, _vp, _vp, C.POINTER(GemmDesc), _vp]),
    "b200_gemm_workspace_bytes": (_sz, []),
    "b200_gemm_row_stats_parts": (_i, [_i, _i, _i]),
    "b200_conv3x3": (_i, [_vp, _vp, _vp, _vp, C.POINTER(Conv3x3Desc), _vp]),
    "b200_conv3x3_up2x": (_i, [_vp, _vp, _vp, _vp, C.POINTER(Conv3x3Desc), _vp]),
    "b200_attention": (_i, [_vp, _vp, _vp, _vp, C.POINTER(AttnDesc), _vp]),
    "b200_groupnorm_ws_bytes": (_sz, [C.POINTER(GnDesc)]),
    "b200_groupnorm_stats": (_i, [_vp, _vp, _vp, C.POINTER(GnDesc), _vp]),
    "b200_groupnorm_apply": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(GnDesc), _vp]),
    "b200_layernorm": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp]),
    "b200_fill_zero": (_i, [_vp, _sz, _vp]),
    "b200_upsample2x": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "b200_im2col3x3": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b200_nchw_to_nhwc": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _f, _i, _i, _vp]),
    "b200_nhwc_to_nchw": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b200_silu": (_i, [_vp, _vp, _sz, _i, _vp]),
    "b200_softmax_rows": (_i, [_vp, _i, _i, _i, _i, _f, _i, _vp]),
    "b200_softmax_rows_blockdiag": (_i, [_vp, _i, _i, _i, _f, _i, _i, _i, _i, _vp]),
    "b200_timestep_embedding": (_i, [_vp, _vp, _i, _i, _f, _i, _vp]),
    "b200_unet_input_im2col": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b200_sampler_step": (_i, [_vp, _vp, _vp, _vp, _vp, C.POINTER(StepDesc), _vp]),
    "b200_vae_postprocess": (_i, [_vp, _vp, _sz, _i, _i, _vp]),
    "b200_images_to_u8": (_i, [_vp, _vp, _sz, _vp]),
    "b200_tile_blend": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _f, _i, _i, _vp]),
    "b200_tile_resolve": (_i, [_vp, _vp, _sz, _i, _f, _i, _vp]),
    "b200_sampler_update": (_i, [_vp, _vp, _vp, _vp, C.POINTER(StepDesc), _vp]),
    "b200_eps_to_denoised": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b200_add_nchw": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "b200_add_control": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b200_vae_preprocess": (_i, [_vp, _vp, _sz, _i, _vp]),
    "b200_vae_posterior": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _vp]),
    "b200_adaln": (_i, [_vp, _vp, _i, _i, _f, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "b200_qk_norm_rope": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _vp]),
    "b200_rmsnorm_rows": (_i, [_vp, _vp, _vp, _i, _i, _f, _i, _vp]),
    "b200_flux_patchify": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "b200_flux_unpatchify": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
}

_lib = None
_lock = threading.Lock()


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libb200forge.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC_DIR, "-j8"]
    if shutil.which("nvcc") is None:  # a CUDA install that is not on PATH
        cmd.append("NVCC=" + os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc"))
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libb200forge.so failed")
    return LIB_PATH


def load() -> C.CDLL:
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise FileNotFoundError(
                    f"{LIB_PATH} is missing — run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(there is no non-CUDA fallback)")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().b200_last_error()
        raise B200Error(rc, msg.decode("utf-8", "replace") if msg else "")
