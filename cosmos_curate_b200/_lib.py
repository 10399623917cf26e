"""ctypes binding of libcurate_b200.so (C ABI declared in include/curate_b200.h).

The library is the product: if it is missing (or fails to load) every entry point raises - there is
no Python / torch / CPU fallback on this path.
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libcurate_b200.so"

CB_OK = 0
CB_ERR = {-1: "CB_ERR_CUDA", -2: "CB_ERR_ARG", -3: "CB_ERR_UNSUPPORTED", -4: "CB_ERR_NVDEC", -5: "CB_ERR_DEMUX", -6: "CB_ERR_STATE"}
ROWDOT_UPPER, ROWDOT_CLIP = 1, 2
FMT_NV12, FMT_RGB24, FMT_NV12_SWS = 0, 1, 2
DT_F16, DT_BF16, DT_F32 = 0, 1, 2
LAYOUT_NCHW, LAYOUT_PATCH = 0, 1
ACT_QUICK_GELU, ACT_GELU_TANH = 0, 1
ARCH_CLIP, ARCH_SIGLIP = 0, 1
EPI_NONE, EPI_QUICK_GELU, EPI_GELU_TANH = 0, 1, 2
DECODE_SEEK_SYNC, DECODE_DISCARD_ALL = 1, 2
DECODE_BACKENDS = {0: "nvdec", 1: "libavcodec"}
CUBIC_OPENCV, CUBIC_IPP = 0, 1


class CurateB200Error(RuntimeError):
    def __init__(self, code: int, where: str, msg: str):
        super().__init__(f"{where}: {CB_ERR.get(code, code)}: {msg}")
        self.code = code


class SurfacePool(C.Structure):
    _fields_ = [
        ("base", C.c_void_p), ("slot_stride", C.c_size_t), ("width", C.c_int), ("height", C.c_int),
        ("pitch", C.c_int), ("luma_rows", C.c_int), ("format", C.c_int),
    ]  # fmt: skip


class VitCfg(C.Structure):
    _fields_ = [
        ("image_size", C.c_int), ("patch", C.c_int), ("hidden", C.c_int), ("layers", C.c_int), ("heads", C.c_int),
        ("mlp", C.c_int), ("proj_dim", C.c_int), ("act", C.c_int), ("arch", C.c_int), ("ln_eps", C.c_float),
    ]  # fmt: skip


class Mp4Info(C.Structure):
    _fields_ = [
        ("codec", C.c_int), ("width", C.c_int), ("height", C.c_int), ("timescale", C.c_uint32),
        ("n_samples", C.c_int), ("n_sync", C.c_int), ("has_ctts", C.c_int), ("duration", C.c_uint64), ("sample_bytes", C.c_uint64),
    ]  # fmt: skip


class DecodeStats(C.Structure):
    _fields_ = [
        ("frames_decoded", C.c_int), ("frames_emitted", C.c_int), ("coded_width", C.c_int), ("coded_height", C.c_int),
        ("width", C.c_int), ("height", C.c_int),
    ]  # fmt: skip


_vp, _i, _f = C.c_void_p, C.c_int, C.c_float
_pf, _pi32 = C.POINTER(C.c_float), C.POINTER(C.c_int32)

# name -> (restype, argtypes); must list every symbol include/curate_b200.h declares
SIGNATURES = {
    "cb_abi_version": (_i, []),
    "cb_init": (_i, [_i, C.POINTER(_vp)]),
    "cb_destroy": (None, [_vp]),
    "cb_last_error": (C.c_char_p, [_vp]),
    "cb_device_info": (_i, [_vp, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(C.c_size_t)]),
    "cb_device_pci_bus_id": (_i, [_vp, C.c_char_p, _i]),
    "cb_launch_count": (C.c_ulonglong, [_vp]),
    "cb_profile_begin": (_i, [_vp]),
    "cb_profile_end": (_i, [_vp, _vp, _pf, C.POINTER(_i), _i]),
    "cb_preprocess_clip": (_i, [_vp, C.POINTER(SurfacePool), _pi32, _i, _i, _i, _i, _i, _i, _pf, _pf, _vp, _vp]),
    "cb_preprocess_clip_u8": (_i, [_vp, C.POINTER(SurfacePool), _pi32, _i, _i, _vp, _vp]),
    "cb_preprocess_bilinear_u8": (_i, [_vp, C.POINTER(SurfacePool), _pi32, _i, _i, _i, _vp, _vp]),
    "cb_resize_cubic_u8": (_i, [_vp, C.POINTER(SurfacePool), _pi32, _i, _i, _i, _i, _vp, _vp]),
    "cb_video_tube": (_i, [_vp, C.POINTER(SurfacePool), _pi32, _i, _i, _i, _pf, _pf, _vp, _vp, _vp]),
    "cb_nv12_to_rgb": (_i, [_vp, C.POINTER(SurfacePool), _pi32, _i, _vp, _vp]),
    "cb_vit_create": (_i, [_vp, C.POINTER(VitCfg), C.POINTER(_vp)]),
    "cb_vit_destroy": (None, [_vp]),
    "cb_vit_set_tensor": (_i, [_vp, C.c_char_p, _pf, C.c_size_t]),
    "cb_vit_set_aesthetic": (_i, [_vp, _pf, C.c_size_t, _f]),
    "cb_vit_finalize": (_i, [_vp, _i]),
    "cb_vit_k_pad": (_i, [_vp]),
    "cb_vit_forward": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "cb_vit_embed_surfaces": (_i, [_vp, C.POINTER(SurfacePool), _pi32, _i, _pf, _pf, _vp, _vp, _vp, _vp]),
    "cb_affine_score": (_i, [_vp, _vp, _vp, _f, _vp, _i, _i, _vp]),
    "cb_mp4_index": (_i, [_vp, _vp, C.c_size_t, C.POINTER(Mp4Info), C.POINTER(C.c_int64), C.POINTER(C.c_uint8), _i]),
    "cb_mp4_cut": (_i, [_vp, _vp, C.c_size_t, _i, _i, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "cb_decode_backend": (_i, [_vp, C.POINTER(_i)]),
    "cb_decoder_create": (_i, [_vp, C.POINTER(_vp)]),
    "cb_decoder_destroy": (None, [_vp]),
    "cb_decoder_decode": (_i, [_vp, _vp, C.c_size_t, _pi32, _i, C.POINTER(SurfacePool), _pi32, C.POINTER(DecodeStats)]),
    "cb_decoder_decode_ex": (_i, [_vp, _vp, C.c_size_t, _pi32, _i, C.POINTER(SurfacePool), _pi32, _i, C.POINTER(DecodeStats)]),
    "cb_decoder_decode_thumbnails": (_i, [_vp, _vp, C.c_size_t, _i, _i, _vp, _i, C.POINTER(DecodeStats)]),
    "cb_transnet_create": (_i, [_vp, C.POINTER(_vp)]),
    "cb_transnet_destroy": (None, [_vp]),
    "cb_transnet_set_tensor": (_i, [_vp, C.c_char_p, _vp, C.c_size_t]),
    "cb_transnet_finalize": (_i, [_vp, _i]),
    "cb_transnet_forward": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "cb_transnet_predict": (_i, [_vp, _vp, _i, _vp, _vp]),
    "cb_rowdot_argmax": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _i, _f, _vp, _vp, _vp]),
    "cb_rows_l2_normalize": (_i, [_vp, _vp, _i, _i, _vp, _vp]),
    "cb_cluster_sums": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "cb_gemm_f16": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "cb_layernorm_f16": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "cb_attention_f16": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
}

_lib = None


def header_symbols() -> list[str]:
    """Function names declared in include/curate_b200.h (used by the CPU export test)."""
    import re

    text = (PKG.parent / "include" / "curate_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cb_[a-z0-9_]+)\s*\(", text)))


def load() -> C.CDLL:
    """Load the shared library (building is the job of __graft_entry__.build(), not of import)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise CurateB200Error(-1, "load", f"{LIB_PATH} is missing - run `python -c 'import __graft_entry__ as g; g.build()'`; there is no CPU fallback")
    lib = C.CDLL(os.fspath(LIB_PATH), mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol: fail loudly
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(rc: int, where: str, ctx=None) -> None:
    if rc != CB_OK:
        msg = load().cb_last_error(ctx)
        raise CurateB200Error(rc, where, msg.decode(errors="replace") if msg else "")
