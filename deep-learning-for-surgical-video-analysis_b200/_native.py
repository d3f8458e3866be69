"""ctypes binding of libsurgvid.so (the C ABI declared in include/surgvid.h) and its in-tree build.

There is no CPU fallback anywhere in this package: if the shared library is missing or a CUDA call fails,
the caller gets a RuntimeError carrying `sv_last_error()`.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from ctypes import POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_size_t, c_uint16, c_void_p

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(_PKG_DIR, "csrc")
# SURGVID_LIB: load another build of the same native library (same-box A/B of two builds); never a non-native path
LIB_PATH = os.environ.get("SURGVID_LIB") or os.path.join(_PKG_DIR, "lib", "libsurgvid.so")
INCLUDE_DIR = os.path.join(os.path.dirname(_PKG_DIR), "include")
SOURCES = ["api.cu", "gemm_tcgen05.cu", "elementwise.cu", "attention.cu", "attention_tc.cu", "attention_probs.cu", "dwconv_tma.cu", "stem.cu", "mixffn.cu", "mstcn.cu", "trans_head.cu", "evp.cu", "preprocess.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]

SV_OK = 0
EXPORTED_SYMBOLS = [
    "sv_last_error", "sv_abi_version",
    "sv_evp_create", "sv_evp_destroy", "sv_evp_set_tensor", "sv_evp_pack_weights", "sv_evp_workspace_bytes",
    "sv_evp_forward", "sv_evp_classify", "sv_evp_read_tap", "sv_evp_last_launch_count", "sv_evp_set_profile", "sv_evp_get_profile", "sv_evp_dump_profile",
    "sv_mstcn_create", "sv_mstcn_destroy", "sv_mstcn_set_tensor", "sv_mstcn_pack_weights", "sv_mstcn_workspace_bytes",
    "sv_mstcn_forward", "sv_mstcn_last_launch_count", "sv_mstcn_forward_query", "sv_op_causal_windows",
    "sv_op_gemm_bf16", "sv_op_layernorm", "sv_op_im2col", "sv_op_dwconv3x3_gelu", "sv_op_attention", "sv_op_attention_kernel", "sv_op_gauss5x5",
    "sv_op_bilinear_tokens", "sv_op_token_mean", "sv_op_stem_conv", "sv_op_mixffn_fc2", "sv_op_gemm_bf16_cat",
    "sv_prep_create", "sv_prep_destroy", "sv_prep_workspace_bytes", "sv_prep_images", "sv_prep_flow",
    "sv_trans_create", "sv_trans_destroy", "sv_trans_set_tensor", "sv_trans_pack_weights", "sv_trans_forward",
    "sv_mstcn_stream_state_bytes", "sv_mstcn_stream_workspace_bytes", "sv_mstcn_stream_reset", "sv_mstcn_stream_step",
    "sv_trans_stream_state_bytes", "sv_trans_stream_reset", "sv_trans_stream_forward",
    "sv_evp_attention_maps_layout", "sv_evp_forward_attention", "sv_op_attention_probs", "sv_op_gemm_plan_info",
    "sv_op_conv_gemm_bf16", "sv_op_conv_gemm_plan_info",
    "sv_evp_stage_shapes", "sv_evp_forward_features", "sv_op_layernorm_nchw", "sv_op_dwconv_plan_info",
]

# entry points an earlier build of the library, loaded through SURGVID_LIB for a same-box A/B run, may not have (build() still requires
# every EXPORTED_SYMBOLS entry of the library it builds)
_ABSENT_IN_EARLIER_BUILDS = ("sv_op_conv_gemm_bf16", "sv_op_conv_gemm_plan_info", "sv_evp_stage_shapes", "sv_evp_forward_features",
                             "sv_op_layernorm_nchw", "sv_op_dwconv_plan_info")


class EvpCfg(Structure):
    _fields_ = [("embed_dims", c_int32 * 4), ("num_heads", c_int32 * 4), ("depths", c_int32 * 4), ("sr_ratios", c_int32 * 4),
                ("mlp_ratio", c_int32), ("embedding_dim", c_int32), ("fold_head", c_int32)]


class TransCfg(Structure):
    _fields_ = [("d_model", c_int32), ("d_ff", c_int32), ("d_k", c_int32), ("d_v", c_int32), ("n_layers", c_int32), ("n_heads", c_int32),
                ("len_q", c_int32)]


class MstcnCfg(Structure):
    _fields_ = [("stages", c_int32), ("layers", c_int32), ("f_maps", c_int32), ("f_dim", c_int32), ("out_features", c_int32),
                ("causal", c_int32)]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into lib/libsurgvid.so (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC_DIR, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC_DIR, f) for f in os.listdir(CSRC_DIR) if f.endswith(".cuh")] + [os.path.join(INCLUDE_DIR, "surgvid.h")]
    if not force and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(d) for d in deps):
        return LIB_PATH
    obj_dir = os.path.join(CSRC_DIR, "build")
    os.makedirs(obj_dir, exist_ok=True)
    os.makedirs(os.path.dirname(LIB_PATH), exist_ok=True)
    nvcc = _nvcc()
    procs = []
    objs = []
    for s in srcs:
        o = os.path.join(obj_dir, os.path.basename(s)[:-3] + ".o")
        objs.append(o)
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + (out or ""))
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed: " + " ".join(cmd) + "\n" + r.stdout)
    return LIB_PATH


_lib = None
_lock = threading.Lock()


def _declare(lib):
    f32p, u16p, i64p = POINTER(c_float), POINTER(c_uint16), POINTER(c_int64)
    lib.sv_last_error.restype = c_char_p
    lib.sv_last_error.argtypes = []
    lib.sv_abi_version.restype = c_int32
    lib.sv_evp_create.argtypes = [POINTER(EvpCfg), POINTER(c_void_p)]
    lib.sv_evp_destroy.argtypes = [c_void_p]
    lib.sv_evp_set_tensor.argtypes = [c_void_p, c_char_p, c_void_p, i64p, c_int32]
    lib.sv_evp_pack_weights.argtypes = [c_void_p]
    lib.sv_evp_workspace_bytes.argtypes = [c_void_p, c_int32, c_int32, c_int32]
    lib.sv_evp_workspace_bytes.restype = c_size_t
    lib.sv_evp_forward.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_size_t, c_void_p]
    lib.sv_evp_classify.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]
    lib.sv_evp_read_tap.argtypes = [c_void_p, c_char_p, c_void_p, c_int64, i64p, c_void_p]
    lib.sv_evp_last_launch_count.argtypes = [c_void_p]
    lib.sv_evp_last_launch_count.restype = c_int64
    lib.sv_evp_set_profile.argtypes = [c_void_p, c_int32]
    lib.sv_evp_get_profile.argtypes = [c_void_p, POINTER(ctypes.c_double), i64p, POINTER(ctypes.c_double), POINTER(ctypes.c_double)]
    lib.sv_evp_dump_profile.argtypes = [c_void_p, c_char_p]
    lib.sv_mstcn_create.argtypes = [POINTER(MstcnCfg), POINTER(c_void_p)]
    lib.sv_mstcn_destroy.argtypes = [c_void_p]
    lib.sv_mstcn_set_tensor.argtypes = [c_void_p, c_char_p, c_void_p, i64p, c_int32]
    lib.sv_mstcn_pack_weights.argtypes = [c_void_p]
    lib.sv_mstcn_workspace_bytes.argtypes = [c_void_p, c_int64]
    lib.sv_mstcn_workspace_bytes.restype = c_size_t
    lib.sv_mstcn_forward.argtypes = [c_void_p, c_void_p, i64p, c_int32, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.sv_mstcn_last_launch_count.argtypes = [c_void_p]
    lib.sv_mstcn_forward_query.argtypes = [c_void_p, c_void_p, i64p, c_int32, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.sv_op_causal_windows.argtypes = [c_void_p, c_int64, c_int32, i64p, c_int32, c_int32, c_void_p, c_void_p]
    lib.sv_mstcn_last_launch_count.restype = c_int64
    lib.sv_op_gemm_bf16.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_int64,
                                    c_void_p, c_int64, c_int32, c_void_p]
    lib.sv_op_gemm_bf16_cat.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p, c_int32,
                                        c_void_p, c_int64, c_void_p, c_int64, c_int32, c_void_p]
    lib.sv_op_gemm_plan_info.argtypes = [c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, POINTER(c_int32)]
    if hasattr(lib, "sv_op_conv_gemm_bf16"):   # see _ABSENT_IN_EARLIER_BUILDS
        lib.sv_op_conv_gemm_bf16.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64, c_int32,
                                             c_void_p, c_int32, c_void_p, c_int64, c_void_p, c_int64, c_int32, c_void_p]
        lib.sv_op_conv_gemm_plan_info.argtypes = [c_int32] * 12 + [POINTER(c_int32), POINTER(c_int32)]
    lib.sv_op_layernorm.argtypes = [c_void_p, c_void_p, c_void_p, c_float, c_int64, c_int32, c_void_p, c_void_p, c_void_p]
    if hasattr(lib, "sv_evp_forward_features"):   # see _ABSENT_IN_EARLIER_BUILDS
        lib.sv_op_layernorm_nchw.argtypes = [c_void_p, c_void_p, c_void_p, c_float, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]
        lib.sv_evp_stage_shapes.argtypes = [POINTER(EvpCfg), c_int32, c_int32, POINTER(c_int32)]
        lib.sv_evp_forward_features.argtypes = [c_void_p, c_void_p, c_void_p, POINTER(c_void_p), i64p, c_void_p, c_int64, c_int32, c_int32,
                                                c_int32, c_int32, c_void_p, c_size_t, c_void_p]
    lib.sv_op_im2col.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p]
    lib.sv_op_dwconv3x3_gelu.argtypes = [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p]
    if hasattr(lib, "sv_op_dwconv_plan_info"):   # see _ABSENT_IN_EARLIER_BUILDS
        lib.sv_op_dwconv_plan_info.argtypes = [c_int32, c_int32, c_int32, c_int32, c_int32, POINTER(c_int32)]
    lib.sv_op_attention.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int32, c_int32, c_int32,
                                    c_int32, c_int32, c_float, c_void_p]
    lib.sv_op_attention_kernel.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int32, c_int32]
    lib.sv_op_gauss5x5.argtypes = [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p]
    lib.sv_op_bilinear_tokens.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p]
    lib.sv_op_stem_conv.argtypes = [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_float, c_int32, c_int32, c_int32, c_int32, c_int32,
                                    c_int32, c_void_p, c_void_p, c_void_p]
    lib.sv_op_token_mean.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p]
    lib.sv_op_mixffn_fc2.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int32, c_int32,
                                     c_int32, c_int32, c_int32, c_void_p]
    lib.sv_trans_create.argtypes = [POINTER(TransCfg), POINTER(c_void_p)]
    lib.sv_trans_destroy.argtypes = [c_void_p]
    lib.sv_trans_set_tensor.argtypes = [c_void_p, c_char_p, c_void_p, i64p, c_int32]
    lib.sv_trans_pack_weights.argtypes = [c_void_p]
    lib.sv_trans_forward.argtypes = [c_void_p, c_void_p, c_int64, c_void_p, i64p, c_int32, c_void_p, c_void_p]
    i32p = POINTER(c_int32)
    lib.sv_mstcn_stream_state_bytes.argtypes = [c_void_p, c_int32]
    lib.sv_mstcn_stream_state_bytes.restype = c_size_t
    lib.sv_mstcn_stream_workspace_bytes.argtypes = [c_void_p, c_int64]
    lib.sv_mstcn_stream_workspace_bytes.restype = c_size_t
    lib.sv_mstcn_stream_reset.argtypes = [c_void_p, c_void_p, c_size_t, c_int32, i32p, c_int32, c_void_p]
    lib.sv_mstcn_stream_step.argtypes = [c_void_p, c_void_p, c_size_t, c_int32, c_void_p, i32p, i64p, c_int32, c_void_p, c_void_p, c_void_p,
                                         c_size_t, c_void_p]
    lib.sv_trans_stream_state_bytes.argtypes = [c_void_p, c_int32]
    lib.sv_trans_stream_state_bytes.restype = c_size_t
    lib.sv_trans_stream_reset.argtypes = [c_void_p, c_void_p, c_size_t, c_int32, i32p, c_int32, c_void_p]
    lib.sv_trans_stream_forward.argtypes = [c_void_p, c_void_p, c_size_t, c_int32, c_void_p, c_int64, c_void_p, i32p, i64p, c_int32, c_void_p,
                                            c_void_p]
    lib.sv_evp_attention_maps_layout.argtypes = [POINTER(EvpCfg), c_int32, c_int32, c_int32, i64p, i32p, c_int32, i32p]
    lib.sv_evp_forward_attention.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32,
                                             c_int32, c_void_p, c_size_t, c_void_p]
    lib.sv_op_attention_probs.argtypes = [c_void_p, c_int64, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, c_float, c_void_p,
                                          c_void_p]
    lib.sv_prep_create.argtypes = [c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, f32p, f32p, POINTER(c_void_p)]
    lib.sv_prep_destroy.argtypes = [c_void_p]
    lib.sv_prep_workspace_bytes.argtypes = [c_void_p, c_int32]
    lib.sv_prep_workspace_bytes.restype = c_size_t
    lib.sv_prep_images.argtypes = [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.sv_prep_flow.argtypes = [c_void_p, c_void_p, c_int32, c_void_p, c_void_p]
    for name in EXPORTED_SYMBOLS:
        if name in _ABSENT_IN_EARLIER_BUILDS and not hasattr(lib, name):
            continue
        fn = getattr(lib, name)
        if name not in ("sv_last_error", "sv_evp_workspace_bytes", "sv_mstcn_workspace_bytes", "sv_evp_last_launch_count",
                        "sv_mstcn_last_launch_count", "sv_prep_workspace_bytes", "sv_mstcn_stream_state_bytes",
                        "sv_mstcn_stream_workspace_bytes", "sv_trans_stream_state_bytes"):
            fn.restype = c_int32


def lib():
    """The loaded libsurgvid.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"libsurgvid.so not found at {LIB_PATH}: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(nvcc, sm_100a). surgvid_b200 has no CPU / PyTorch fallback.")
            handle = ctypes.CDLL(LIB_PATH)
            _declare(handle)
            _lib = handle
    return _lib


def last_error() -> str:
    return lib().sv_last_error().decode("utf-8", "replace")


def check(status: int, what: str = "libsurgvid"):
    if status != SV_OK:
        raise RuntimeError(f"{what} failed (status {status}): {last_error()}")


def set_tensors(set_tensor, handle, named_tensors, what: str):
    """Hand (name, tensor) pairs, e.g. `module.state_dict().items()`, to a handle's `sv_*_set_tensor` as contiguous fp32 host copies."""
    import numpy as np
    import torch

    for name, t in named_tensors:
        a = np.ascontiguousarray(t.detach().to("cpu", torch.float32).numpy())
        shape = (c_int64 * max(a.ndim, 1))(*a.shape)
        check(set_tensor(handle, name.encode(), a.ctypes.data_as(c_void_p), shape, a.ndim), what)
