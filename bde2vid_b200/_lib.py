"""ctypes binding of libbde2vid_sm100.so (the C ABI declared in include/bde2vid.h).

There is no CPU fallback anywhere in this package: if the shared library is missing or the
device is not a Blackwell-class GPU the ops raise.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# BDE2VID_LIB: another build of the same library (ablation builds of tools/attn64_probe.sh); the default is the in-tree one
LIB_PATH = os.environ.get("BDE2VID_LIB") or os.path.join(_HERE, "libbde2vid_sm100.so")

F32, BF16 = 0, 1
ABI_VERSION = 3
ACT_NONE, ACT_RELU, ACT_RELU6, ACT_GELU, ACT_SIGMOID = 0, 1, 2, 3, 4
EPI_STORE, EPI_LSTM, EPI_SCATTER, EPI_GRU_UR, EPI_GRU_OUT = 0, 1, 2, 3, 4
ENGINE_SIMT, ENGINE_TCGEN05 = 0, 1

TORCH_DTYPE = {F32: torch.float32, BF16: torch.bfloat16}
BDE_DTYPE = {torch.float32: F32, torch.bfloat16: BF16}


class GemmDesc(C.Structure):
    """Mirror of ``struct bde_gemm_desc``."""
    _fields_ = [
        ("engine", C.c_int), ("dtype", C.c_int),
        ("a0", C.c_void_p), ("a1", C.c_void_p),
        ("c0", C.c_int), ("c1", C.c_int),
        ("n_img", C.c_int), ("h_in", C.c_int), ("w_in", C.c_int), ("h_out", C.c_int), ("w_out", C.c_int),
        ("ksize", C.c_int), ("stride", C.c_int), ("pad", C.c_int),
        ("w", C.c_void_p), ("bias", C.c_void_p),
        ("n", C.c_int), ("w_ld", C.c_int), ("k_order", C.c_int),
        ("ln_mode", C.c_int), ("ln_D", C.c_int), ("ln_n_tok", C.c_int),
        ("ln_frames", C.c_void_p * 8), ("ln_tok_map", C.c_void_p),
        ("epi", C.c_int), ("act", C.c_int), ("out_f32", C.c_int),
        ("out", C.c_void_p), ("residual", C.c_void_p), ("c_prev", C.c_void_p), ("c_out", C.c_void_p),
        ("row_map", C.c_void_p), ("out2", C.c_void_p), ("res_mode", C.c_int),
        ("a0_ld", C.c_int), ("a1_ld", C.c_int),
    ]


EXPORTS = {
    "bde_last_error": (C.c_char_p, []),
    "bde_abi_version": (C.c_int, []),
    "bde_device_ok": (C.c_int, []),
    "bde_voxelize_seq": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 8 + [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "bde_voxelize_seq_strided": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 8 + [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int,
                                           C.c_int, C.c_void_p, C.c_void_p]),
    "bde_voxelize_raw_strided": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 8 + [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int,
                                           C.c_int, C.c_void_p, C.c_void_p]),
    "bde_voxel_normalize": (C.c_int, [C.c_void_p, C.c_size_t] + [C.c_int] * 9 + [C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    "bde_hot_pixel_mask": (C.c_int, [C.c_void_p] * 3 + [C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bde_frame_metrics": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 7 + [C.c_double, C.c_void_p, C.c_void_p]),
    "bde_head_conv": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 7 + [C.c_void_p]),
    "bde_pack_voxel_nhwc": (C.c_int, [C.c_void_p] + [C.c_int] * 5 + [C.c_void_p, C.c_int, C.c_void_p]),
    "bde_profile_begin": (C.c_int, [C.c_int]),
    "bde_profile_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "bde_profile_flops": (C.c_int, [C.POINTER(C.c_double)]),
    "bde_gemm": (C.c_int, [C.POINTER(GemmDesc), C.c_void_p]),
    "bde_add": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int,
                          C.c_void_p]),
    "bde_upsample2x_sum": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_float] + [C.c_int] * 4
                           + [C.c_void_p, C.c_int, C.c_void_p]),
    "bde_shuffle2x_sum": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 4 + [C.c_void_p, C.c_int, C.c_void_p]),
    "bde_pred_sigmoid": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "bde_window_reduce": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bde_ln_gather": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "bde_layernorm": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                C.c_void_p]),
    "bde_window_attention": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 5 + [C.c_void_p, C.c_int, C.c_void_p]),
    "bde_ln_gather_qkv": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
                          + [C.c_void_p] * 6 + [C.c_int, C.c_void_p]),
    "bde_window_attention_mma_bias_stride": (C.c_int, [C.c_int]),
    "bde_window_attention_mma": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 5 + [C.c_void_p, C.c_void_p]),
    "bde_window_attention_mma_qkv": (C.c_int, [C.c_void_p, C.c_void_p] + [C.c_int] * 6 + [C.c_void_p, C.c_void_p]),
    "bde_window_attention_fused_supported": (C.c_int, [C.c_int] * 4),
    "bde_window_attention_fused": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
                                   + [C.c_void_p] * 8),
    "bde_mlp_fused_supported": (C.c_int, [C.c_int, C.c_int]),
    "bde_mlp_fused": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int] + [C.c_void_p] * 5),
    "bde_mlp_fused_sum": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_int] + [C.c_void_p] * 7),
    "bde_cast": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p]),
}

_lib = None


def load():
    """Load the shared library (once) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libbde2vid_sm100.so is not built (%s). Run `python -m bde2vid_b200.build`; "
            "there is no CPU or PyTorch fallback for this path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.bde_abi_version() != ABI_VERSION:
        raise RuntimeError("libbde2vid_sm100.so ABI mismatch")
    _lib = lib
    return lib


def require_device():
    """Raise unless CUDA is available and the current device is compute capability 10.x."""
    if not torch.cuda.is_available():
        raise RuntimeError("bde2vid_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
    lib = load()
    ok = lib.bde_device_ok()
    if ok != 1:
        raise RuntimeError("bde2vid_b200 kernels are built for sm_100a only (device check returned %d: %s)"
                           % (ok, lib.bde_last_error().decode()))
    return lib


def check(rc, what=""):
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (what or "bde call", rc, load().bde_last_error().decode()))


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "bde2vid_b200 ops need contiguous CUDA tensors"
    return C.c_void_p(t.data_ptr())
