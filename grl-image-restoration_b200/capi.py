"""ctypes binding of libgrl_b200.so (include/grl_b200.h).  This is the only place the Python surface
touches native code; there is no CPU or eager-PyTorch fallback: a missing library or a non-CUDA tensor is an
error."""
import ctypes
import os
import re

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libgrl_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_PKG), "include", "grl_b200.h")

ABI_VERSION = 3
c_int, c_i64, c_f32, c_vp, c_sz = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t


class GrlGrid(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("H", "W", "wh", "ww", "sh", "sw")]

    def __repr__(self):
        return f"GrlGrid({self.H}x{self.W}, win {self.wh}x{self.ww}, shift {self.sh},{self.sw})"


def grid(H, W, wh, ww, sh=0, sw=0):
    return GrlGrid(int(H), int(W), int(wh), int(ww), int(sh), int(sw))


class GrlTcGemm(ctypes.Structure):
    _fields_ = [("fmt", ctypes.c_int32), ("x", c_vp), ("w", c_vp), ("bias", c_vp), ("M", c_i64), ("B", ctypes.c_int32), ("H", ctypes.c_int32),
                ("W", ctypes.c_int32), ("kpad", ctypes.c_int32), ("npad", ctypes.c_int32), ("taps", ctypes.c_int32),
                ("epi", ctypes.c_int32), ("n_store", ctypes.c_int32), ("n_real", ctypes.c_int32), ("out_bf16", c_vp),
                ("ldo_bf16", c_i64), ("out_f32", c_vp), ("ldo_f32", c_i64), ("res_f32", c_vp), ("ldr", c_i64),
                ("act", ctypes.c_int32), ("slope", c_f32), ("slot_scale", c_vp), ("C", ctypes.c_int32), ("gamma", c_vp),
                ("beta", c_vp), ("eps", c_f32), ("res_scale", c_f32), ("cab_y", c_vp), ("ld_caby", c_i64),
                ("cab_gate", c_vp), ("L", c_i64), ("ps_r", ctypes.c_int32), ("out_nchw", c_vp), ("nchw_r", ctypes.c_int32),
                ("Hc", ctypes.c_int32), ("Wc", ctypes.c_int32), ("post_scale", c_f32), ("post_shift", c_f32 * 4)]


class GrlTcMlp(ctypes.Structure):
    _fields_ = [("fmt", ctypes.c_int32), ("x", c_vp), ("w1", c_vp), ("b1", c_vp), ("w2", c_vp), ("b2", c_vp), ("M", c_i64),
                ("C", ctypes.c_int32), ("cpad", ctypes.c_int32), ("hpad", ctypes.c_int32), ("n_ln", ctypes.c_int32),
                ("gamma", c_vp), ("beta", c_vp), ("eps", c_f32), ("res_scale", c_f32), ("res_f32", c_vp), ("ldr", c_i64),
                ("out_f32", c_vp), ("ldo_f32", c_i64), ("out_bf16", c_vp), ("ldo_bf16", c_i64)]


class GrlTcAttn(ctypes.Structure):
    _fields_ = [("fmt", ctypes.c_int32), ("gq", GrlGrid), ("gk", GrlGrid), ("q", c_vp), ("ldq", c_i64), ("q_off", ctypes.c_int32), ("k", c_vp),
                ("ldk", c_i64), ("k_off", ctypes.c_int32), ("v", c_vp), ("ldv", c_i64), ("v_off", ctypes.c_int32),
                ("v_dense", ctypes.c_int32), ("out", c_vp), ("ldo", c_i64), ("o_off", ctypes.c_int32),
                ("o_dense", ctypes.c_int32), ("B", ctypes.c_int32), ("heads", ctypes.c_int32), ("bias", c_vp),
                ("rows", ctypes.c_int32), ("rows_pad", ctypes.c_int32), ("use_mask", ctypes.c_int32), ("ones_col", ctypes.c_int32)]


_SIGNATURES = {
    "grl_last_error": (ctypes.c_char_p, []),
    "grl_abi_version": (c_int, []),
    "grl_device_ok": (c_int, []),
    "grl_launch_count": (ctypes.c_uint64, []),
    "grl_rel_index_host": (c_int, [c_int, c_int, c_int, c_int, c_vp]),
    "grl_shift_mask_host": (c_int, [c_int] * 8 + [c_vp]),
    "grl_token_map_host": (c_int, [GrlGrid, c_vp]),
    "grl_tc_attn_box_tokens": (c_int, [GrlGrid]),
    "grl_coords_table_host": (c_int, [c_int, c_int, c_int, c_vp]),
    "grl_bias_table_f32": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp]),
    "grl_tc_bias_table4": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_f32, c_int, c_vp, c_vp]),
    "grl_tc_pack16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "grl_tc_unpack16": (c_int, [c_vp, c_i64, c_int, c_vp, c_i64, c_i64, c_int, c_int, c_vp]),
    "grl_tc_head_pack": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_f32), c_f32, c_vp, c_int, c_vp, c_int, c_vp]),
    "grl_tc_avgpool16": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "grl_tc_slot_scale": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp]),
    "grl_tc_channel_gate_workspace": (c_sz, [c_int, c_i64, c_int]),
    "grl_tc_channel_gate": (c_int, [c_vp, c_i64, c_int, c_int, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_sz, c_vp]),
    "grl_tc_gemm": (c_int, [ctypes.POINTER(GrlTcGemm), c_vp]),
    "grl_tc_mlp": (c_int, [ctypes.POINTER(GrlTcMlp), c_vp]),
    "grl_tc_attn": (c_int, [ctypes.POINTER(GrlTcAttn), c_vp]),
    "grl_tc_attn_variant": (c_int, [c_int]),
    "grl_tc_attn2_debug": (c_int, [ctypes.POINTER(c_int)]),
    "grl_psnr_f32": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_sz, c_vp, c_vp, c_vp]),
    "grl_affine_f32": (c_int, [c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_vp]),
    "grl_linear_f32": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_int, c_int, c_f32, c_vp]),
    "grl_conv3x3_f32": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_f32, c_vp]),
    "grl_avgpool_f32": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "grl_ln_residual_f32": (c_int, [c_vp, c_vp, c_vp, c_vp, c_f32, c_f32, c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_vp]),
    "grl_channel_gate_workspace": (c_sz, [c_int, c_i64, c_int]),
    "grl_channel_gate_f32": (c_int, [c_vp, c_int, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_sz, c_vp]),
    "grl_window_attn_f32": (c_int, [c_vp, c_i64, c_vp, c_i64, c_int, GrlGrid, c_int, c_int, c_vp, c_vp, c_int, c_vp]),
    "grl_stripe_attn_workspace": (c_sz, [c_int, GrlGrid, GrlGrid, c_int, c_int]),
    "grl_stripe_attn_f32": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, GrlGrid, GrlGrid, c_int, c_int,
                                    c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_sz, c_vp]),
}

_lib = None


def header_symbols():
    """Every function name declared in include/grl_b200.h."""
    with open(HEADER_PATH) as f:
        src = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(grl_[a-z0-9_]+)\s*\(", src)))


def lib():
    """Loads the library (never builds it implicitly on a GPU box: the .so ships with the snapshot)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU / eager fallback for the GRL hot path)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.grl_abi_version() != ABI_VERSION:
            raise RuntimeError("libgrl_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError(f"grl_b200 error {rc}: {lib().grl_last_error().decode()}")


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("grl_b200 operators need CUDA tensors (no CPU fallback)")
    return ctypes.c_void_p(t.data_ptr())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_device(t):
    """The C ABI launches on the CURRENT device's current stream (one process per GPU, as under DDP / torchrun).  A
    tensor living on another device of the same process would be launched with foreign pointers: refuse it with a
    clear message instead (wrap the call in `with torch.cuda.device(t.device):`)."""
    if not t.is_cuda:
        raise RuntimeError("grl_b200: input is not on a CUDA device; the B200 kernels have no CPU fallback")
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError(f"grl_b200: tensor on cuda:{t.device.index} but the current device is cuda:{torch.cuda.current_device()}; "
                           f"call torch.cuda.set_device / use `with torch.cuda.device(...)` (kernels launch on the current device)")
