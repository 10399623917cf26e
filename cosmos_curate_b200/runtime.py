"""Thin Python layer over the C ABI: torch tensors are only zero-copy containers (data_ptr()).

Nothing here computes on the data path; every operation is a call into libcurate_b200.so.
"""

from __future__ import annotations

import ctypes as C
import weakref

import numpy as np
import torch

from . import _lib
from ._lib import SurfacePool, VitCfg, check

CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)  # reference: cosmos_curate/models/clip.py:57-60
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)
IMAGENET_MEAN = (0.485, 0.456, 0.406)  # reference: cosmos_curate/models/internvideo2_mm.py:378-379
IMAGENET_STD = (0.229, 0.224, 0.225)

_TORCH_DT = {torch.float16: _lib.DT_F16, torch.bfloat16: _lib.DT_BF16, torch.float32: _lib.DT_F32}


def _f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


def _stream_ptr(stream=None) -> int:
    s = stream if stream is not None else torch.cuda.current_stream()
    return int(s.cuda_stream)


class Context:
    """One per process/GPU (cb_init).  Fails loudly when the library or a CUDA device is missing."""

    def __init__(self, device: int | None = None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.CurateB200Error(-1, "Context", "no CUDA device; this path has no CPU fallback")
        self.device = torch.cuda.current_device() if device is None else int(device)
        torch.cuda.set_device(self.device)
        torch.cuda.init()
        h = C.c_void_p()
        check(self.lib.cb_init(self.device, C.byref(h)), "cb_init")
        self.h = h
        self._children = weakref.WeakSet()  # towers / decoders created on this context: closed before it

    def close(self):
        if getattr(self, "h", None):
            for child in list(self._children):
                child.close()
            self.lib.cb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def decode_backend(self) -> str:
        """"nvdec", or "libavcodec" where the driver exposes no NVDEC engine to this process (cb_decode_backend)."""
        b = C.c_int()
        check(self.lib.cb_decode_backend(self.h, C.byref(b)), "cb_decode_backend", self.h)
        return _lib.DECODE_BACKENDS[b.value]

    def launch_count(self) -> int:
        return int(self.lib.cb_launch_count(self.h))

    PROF_CATEGORIES = ("preprocess", "gemm", "layernorm", "attention", "other", "conv")

    def profile_begin(self) -> None:
        check(self.lib.cb_profile_begin(self.h), "cb_profile_begin", self.h)

    def profile_end(self) -> dict:
        n = len(self.PROF_CATEGORIES)
        ms, cnt = (C.c_float * n)(), (C.c_int * n)()
        check(self.lib.cb_profile_end(self.h, _stream_ptr(), ms, cnt, n), "cb_profile_end", self.h)
        return {k: {"ms": float(ms[i]), "launches": int(cnt[i])} for i, k in enumerate(self.PROF_CATEGORIES)}

    def device_info(self) -> dict:
        sm, ma, mi, mem = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
        check(self.lib.cb_device_info(self.h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem)), "cb_device_info", self.h)
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "total_mem": mem.value}

    # ---- surfaces -----------------------------------------------------------------------------
    def nv12_pool(self, buf: torch.Tensor, width: int, height: int, luma_rows: int | None = None, colour: str = "opencv") -> "Pool":
        """buf: uint8 cuda [slots, rows, pitch] with rows >= luma_rows + height/2.  colour: "opencv" (CV-CUDA / cv2.cvtColor
        semantics, the reference's CUDA branch) or "swscale" (libswscale's yuv420p -> rgb24, the reference's CPU decode branch)."""
        assert buf.is_cuda and buf.dtype == torch.uint8 and buf.dim() == 3 and buf.is_contiguous()
        luma_rows = height if luma_rows is None else luma_rows
        assert buf.shape[1] >= luma_rows + height // 2
        fmt = {"opencv": _lib.FMT_NV12, "swscale": _lib.FMT_NV12_SWS}[colour]
        return Pool(buf, SurfacePool(buf.data_ptr(), buf.shape[1] * buf.shape[2], width, height, buf.shape[2], luma_rows, fmt))

    def rgb_pool(self, frames: torch.Tensor) -> "Pool":
        """frames: uint8 cuda [n, H, W, 3] (contiguous).  Rows are re-pitched to a 16-byte multiple if needed."""
        assert frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[-1] == 3
        n, h, w, _ = frames.shape
        row = 3 * w
        pitch = (row + 15) & ~15
        if pitch != row or not frames.is_contiguous():
            buf = torch.zeros((n, h, pitch), dtype=torch.uint8, device=frames.device)
            buf[:, :, :row] = frames.reshape(n, h, row)
        else:
            buf = frames.reshape(n, h, row)
        stride = h * pitch
        if stride % 16:
            pad = torch.zeros((n, (stride + 15) // 16 * 16), dtype=torch.uint8, device=frames.device)
            pad[:, :stride] = buf.reshape(n, stride)
            buf, stride = pad, pad.shape[1]
        return Pool(buf, SurfacePool(buf.data_ptr(), stride, w, h, pitch, h, _lib.FMT_RGB24))

    # ---- preprocess ---------------------------------------------------------------------------
    def _slots(self, pool: "Pool", slots):
        n_slots = pool.buf.shape[0]
        arr = np.arange(n_slots, dtype=np.int32) if slots is None else np.ascontiguousarray(slots, dtype=np.int32)
        return arr, arr.ctypes.data_as(C.POINTER(C.c_int32))

    def preprocess_clip(self, pool: "Pool", slots=None, res: int = 224, dtype=torch.float16, layout: str = "nchw", patch: int = 0,
                        k_pad: int = 0, mean=CLIP_MEAN, std=CLIP_STD, out: torch.Tensor | None = None) -> torch.Tensor:
        arr, ptr = self._slots(pool, slots)
        n = len(arr)
        if layout == "nchw":
            shape, lay = (n, 3, res, res), _lib.LAYOUT_NCHW
        else:
            g = res // patch
            shape, lay = (n, g * g, k_pad), _lib.LAYOUT_PATCH
        if out is None:
            out = torch.empty(shape, dtype=dtype, device=pool.buf.device)
        check(self.lib.cb_preprocess_clip(self.h, C.byref(pool.desc), ptr, n, res, lay, patch, k_pad, _TORCH_DT[dtype], _f3(mean), _f3(std),
                                          out.data_ptr(), _stream_ptr()), "cb_preprocess_clip", self.h)  # fmt: skip
        return out

    def preprocess_clip_u8(self, pool: "Pool", slots=None, res: int = 224) -> torch.Tensor:
        arr, ptr = self._slots(pool, slots)
        out = torch.empty((len(arr), 3, res, res), dtype=torch.uint8, device=pool.buf.device)
        check(self.lib.cb_preprocess_clip_u8(self.h, C.byref(pool.desc), ptr, len(arr), res, out.data_ptr(), _stream_ptr()),
              "cb_preprocess_clip_u8", self.h)  # fmt: skip
        return out

    def preprocess_bilinear_u8(self, pool: "Pool", out_w: int, out_h: int, slots=None) -> torch.Tensor:
        arr, ptr = self._slots(pool, slots)
        out = torch.empty((len(arr), out_h, out_w, 3), dtype=torch.uint8, device=pool.buf.device)
        check(self.lib.cb_preprocess_bilinear_u8(self.h, C.byref(pool.desc), ptr, len(arr), out_w, out_h, out.data_ptr(), _stream_ptr()),
              "cb_preprocess_bilinear_u8", self.h)  # fmt: skip
        return out

    def resize_cubic_u8(self, pool: "Pool", out_w: int, out_h: int, slots=None, mode: int = _lib.CUBIC_IPP) -> torch.Tensor:
        """cv2.resize(frame, (out_w, out_h), INTER_CUBIC) per frame of the pool -> uint8 cuda [n, out_h, out_w, 3]."""
        arr, ptr = self._slots(pool, slots)
        out = torch.empty((len(arr), out_h, out_w, 3), dtype=torch.uint8, device=pool.buf.device)
        check(self.lib.cb_resize_cubic_u8(self.h, C.byref(pool.desc), ptr, len(arr), out_w, out_h, mode, out.data_ptr(), _stream_ptr()),
              "cb_resize_cubic_u8", self.h)  # fmt: skip
        return out

    def video_tube(self, pool: "Pool", out_w: int, out_h: int, slots=None, mean=IMAGENET_MEAN, std=IMAGENET_STD, want_u8: bool = False):
        """cv2.resize(frame, (out_w, out_h)) + ((x / 255 - mean) / std) per frame -> float32 cuda [n, 3, out_h, out_w]
        (internvideo2_mm.py:385-405); with want_u8 also the resized uint8 [n, out_h, out_w, 3] frames."""
        arr, ptr = self._slots(pool, slots)
        out = torch.empty((len(arr), 3, out_h, out_w), dtype=torch.float32, device=pool.buf.device)
        u8 = torch.empty((len(arr), out_h, out_w, 3), dtype=torch.uint8, device=pool.buf.device) if want_u8 else None
        check(self.lib.cb_video_tube(self.h, C.byref(pool.desc), ptr, len(arr), out_w, out_h, _f3(mean), _f3(std), out.data_ptr(),
                                     u8.data_ptr() if want_u8 else None, _stream_ptr()), "cb_video_tube", self.h)  # fmt: skip
        return (out, u8) if want_u8 else out

    def nv12_to_rgb(self, pool: "Pool", slots=None) -> torch.Tensor:
        arr, ptr = self._slots(pool, slots)
        out = torch.empty((len(arr), pool.desc.height, pool.desc.width, 3), dtype=torch.uint8, device=pool.buf.device)
        check(self.lib.cb_nv12_to_rgb(self.h, C.byref(pool.desc), ptr, len(arr), out.data_ptr(), _stream_ptr()), "cb_nv12_to_rgb", self.h)
        return out

    # ---- building blocks (parity tests) -----------------------------------------------------------
    def gemm(self, a: torch.Tensor, w: torch.Tensor, bias=None, residual=None, epilogue: int = _lib.EPI_NONE, out_f32: bool = False):
        m, k = a.shape
        n = w.shape[0]
        assert a.dtype == torch.float16 and w.dtype == torch.float16 and w.shape[1] == k and a.is_contiguous() and w.is_contiguous()
        if out_f32:
            out = residual if residual is not None else torch.empty((m, n), dtype=torch.float32, device=a.device)
            o32, o16 = out.data_ptr(), None
        else:
            out = torch.empty((m, n), dtype=torch.float16, device=a.device)
            o32, o16 = None, out.data_ptr()
        check(self.lib.cb_gemm_f16(self.h, a.data_ptr(), w.data_ptr(), bias.data_ptr() if bias is not None else None,
                                   residual.data_ptr() if residual is not None else None, o32, o16, m, n, k, epilogue, _stream_ptr()),
              "cb_gemm_f16", self.h)  # fmt: skip
        return out

    def layernorm(self, x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float) -> torch.Tensor:
        rows, d = x.shape
        y = torch.empty((rows, d), dtype=torch.float16, device=x.device)
        check(self.lib.cb_layernorm_f16(self.h, x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), rows, d, eps, _stream_ptr()),
              "cb_layernorm_f16", self.h)  # fmt: skip
        return y

    def attention(self, qkv: torch.Tensor, heads: int) -> torch.Tensor:
        n, t, three_d = qkv.shape
        d = three_d // 3
        out = torch.empty((n, t, d), dtype=torch.float16, device=qkv.device)
        check(self.lib.cb_attention_f16(self.h, qkv.data_ptr(), out.data_ptr(), n, t, heads, d // heads, _stream_ptr()), "cb_attention_f16", self.h)
        return out


_CONTEXTS: dict[int, Context] = {}


def get_context(device: int | None = None) -> Context:
    """Process-wide context per device (stages and models of one actor process share it)."""
    dev = torch.cuda.current_device() if (device is None and torch.cuda.is_available()) else int(device or 0)
    c = _CONTEXTS.get(dev)
    if c is None or c.h is None:
        c = _CONTEXTS[dev] = Context(dev)
    return c


def affine_score(ctx: Context, emb: torch.Tensor, w: torch.Tensor, b: float) -> torch.Tensor:
    n, d = emb.shape
    out = torch.empty((n,), dtype=torch.float32, device=emb.device)
    check(ctx.lib.cb_affine_score(ctx.h, emb.data_ptr(), w.data_ptr(), float(b), out.data_ptr(), n, d, _stream_ptr()), "cb_affine_score", ctx.h)
    return out


class Pool:
    def __init__(self, buf: torch.Tensor, desc: SurfacePool):
        self.buf, self.desc = buf, desc  # keep the tensor alive while the descriptor is in use


class VitTower:
    """cb_vit_* wrapper: weights in (fp32 numpy, names of include/curate_b200.h cb_vit_set_tensor), embeddings / scores out."""

    def __init__(self, ctx: Context, cfg: dict, weights: dict, max_batch: int = 256, aesthetic: tuple | None = None):
        self.ctx, self.lib = ctx, ctx.lib
        self.cfg = dict(cfg)
        c = VitCfg(cfg["image_size"], cfg["patch"], cfg["hidden"], cfg["layers"], cfg["heads"], cfg["mlp"], cfg["proj_dim"],
                   _lib.ACT_QUICK_GELU if cfg["act"] == "quick_gelu" else _lib.ACT_GELU_TANH,
                   _lib.ARCH_CLIP if cfg["arch"] == "clip" else _lib.ARCH_SIGLIP, cfg["ln_eps"])  # fmt: skip
        h = C.c_void_p()
        check(self.lib.cb_vit_create(ctx.h, C.byref(c), C.byref(h)), "cb_vit_create", ctx.h)
        self.h = h
        ctx._children.add(self)
        for name, arr in weights.items():
            a = np.ascontiguousarray(arr, dtype=np.float32)
            check(self.lib.cb_vit_set_tensor(self.h, name.encode(), a.ctypes.data_as(C.POINTER(C.c_float)), a.size), f"cb_vit_set_tensor({name})", ctx.h)
        self.out_dim = cfg["proj_dim"] or cfg["hidden"]
        self.has_aesthetic = False
        if aesthetic is not None:
            w, b = aesthetic
            w = np.ascontiguousarray(w, dtype=np.float32)
            check(self.lib.cb_vit_set_aesthetic(self.h, w.ctypes.data_as(C.POINTER(C.c_float)), w.size, float(b)), "cb_vit_set_aesthetic", ctx.h)
            self.has_aesthetic = True
        check(self.lib.cb_vit_finalize(self.h, max_batch), "cb_vit_finalize", ctx.h)
        self.k_pad = int(self.lib.cb_vit_k_pad(self.h))
        self.max_batch = max_batch

    def close(self):
        if getattr(self, "h", None):
            self.lib.cb_vit_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def forward_patches(self, patches: torch.Tensor, want_features: bool = False):
        n = patches.shape[0]
        dev = patches.device
        emb = torch.empty((n, self.out_dim), dtype=torch.float32, device=dev)
        feat = torch.empty((n, self.out_dim), dtype=torch.float32, device=dev) if want_features else None
        score = torch.empty((n,), dtype=torch.float32, device=dev) if self.has_aesthetic else None
        check(self.lib.cb_vit_forward(self.h, patches.data_ptr(), n, emb.data_ptr(), feat.data_ptr() if feat is not None else None,
                                      score.data_ptr() if score is not None else None, _stream_ptr()), "cb_vit_forward", self.ctx.h)  # fmt: skip
        return emb, feat, score

    def embed_pool(self, pool: Pool, slots=None, mean=CLIP_MEAN, std=CLIP_STD, want_features: bool = False):
        arr, ptr = self.ctx._slots(pool, slots)
        n, dev = len(arr), pool.buf.device
        emb = torch.empty((n, self.out_dim), dtype=torch.float32, device=dev)
        feat = torch.empty((n, self.out_dim), dtype=torch.float32, device=dev) if want_features else None
        score = torch.empty((n,), dtype=torch.float32, device=dev) if self.has_aesthetic else None
        check(self.lib.cb_vit_embed_surfaces(self.h, C.byref(pool.desc), ptr, n, _f3(mean), _f3(std), emb.data_ptr(),
                                             feat.data_ptr() if feat is not None else None, score.data_ptr() if score is not None else None,
                                             _stream_ptr()), "cb_vit_embed_surfaces", self.ctx.h)  # fmt: skip
        return emb, feat, score


class ShotNet:
    """cb_transnet_* wrapper: the reference state_dict in (its own key names), per-frame transition probabilities out."""

    UNUSED_KEYS = ("cls_layer2.weight", "cls_layer2.bias")  # many-hot head: built by the reference, never used by forward()

    def __init__(self, ctx: Context, state_dict: dict, max_windows: int = 16):
        self.ctx, self.lib = ctx, ctx.lib
        h = C.c_void_p()
        check(self.lib.cb_transnet_create(ctx.h, C.byref(h)), "cb_transnet_create", ctx.h)
        self.h = h
        ctx._children.add(self)
        for name, arr in state_dict.items():
            if name in self.UNUSED_KEYS or name.endswith("num_batches_tracked"):
                continue
            a = np.ascontiguousarray(arr.detach().cpu().numpy() if isinstance(arr, torch.Tensor) else arr, dtype=np.float32)
            check(self.lib.cb_transnet_set_tensor(self.h, name.encode(), a.ctypes.data_as(C.c_void_p), a.size), f"cb_transnet_set_tensor({name})", ctx.h)
        check(self.lib.cb_transnet_finalize(self.h, max_windows), "cb_transnet_finalize", ctx.h)
        self.max_windows = max_windows

    def close(self):
        if getattr(self, "h", None):
            self.lib.cb_transnet_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def forward(self, windows: torch.Tensor) -> torch.Tensor:
        """uint8 cuda [B, T, 27, 48, 3] -> fp32 cuda [B, T, 1] (the reference model's call signature, transnetv2.py:569-580)."""
        assert windows.is_cuda and windows.dtype == torch.uint8 and windows.dim() == 5 and tuple(windows.shape[2:]) == (27, 48, 3), windows.shape
        windows = windows.contiguous()
        b, t = windows.shape[:2]
        out = torch.empty((b, t, 1), dtype=torch.float32, device=windows.device)
        check(self.lib.cb_transnet_forward(self.h, windows.data_ptr(), b, t, out.data_ptr(), _stream_ptr()), "cb_transnet_forward", self.ctx.h)
        return out

    def predict(self, frames: torch.Tensor) -> torch.Tensor:
        """uint8 cuda [n, 27, 48, 3] (a whole video) -> fp32 cuda [n] stitched probabilities."""
        assert frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and tuple(frames.shape[1:]) == (27, 48, 3), frames.shape
        frames = frames.contiguous()
        out = torch.empty((frames.shape[0],), dtype=torch.float32, device=frames.device)
        check(self.lib.cb_transnet_predict(self.h, frames.data_ptr(), frames.shape[0], out.data_ptr(), _stream_ptr()), "cb_transnet_predict", self.ctx.h)
        return out


# ---- demux + NVDEC ------------------------------------------------------------------------------------
def _as_u8(data) -> np.ndarray:
    if isinstance(data, np.ndarray):
        return np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
    return np.frombuffer(bytes(data) if not isinstance(data, (bytes, bytearray, memoryview)) else data, dtype=np.uint8)


def mp4_index(data, ctx: Context | None = None) -> dict:
    """cb_mp4_index: video-track facts + per-sample PTS ticks (decode order) + sync flags (host-only parse)."""
    buf = _as_u8(data)
    lib = ctx.lib if ctx is not None else _lib.load()
    h = ctx.h if ctx is not None else None
    info = _lib.Mp4Info()
    check(lib.cb_mp4_index(h, buf.ctypes.data, buf.size, C.byref(info), None, None, 0), "cb_mp4_index", h)
    n = info.n_samples
    pts = np.empty(n, dtype=np.int64)
    sync = np.empty(n, dtype=np.uint8)
    check(lib.cb_mp4_index(h, buf.ctypes.data, buf.size, C.byref(info), pts.ctypes.data_as(C.POINTER(C.c_int64)),
                           sync.ctypes.data_as(C.POINTER(C.c_uint8)), n), "cb_mp4_index", h)  # fmt: skip
    return {"codec": info.codec, "width": info.width, "height": info.height, "timescale": info.timescale, "n_samples": n,
            "n_sync": info.n_sync, "has_ctts": bool(info.has_ctts), "duration": info.duration, "sample_bytes": info.sample_bytes,
            "pts": pts, "sync": sync}  # fmt: skip


class Decoder:
    """One decode session (cb_decoder_*): NVDEC, or libavcodec on the host where the driver exposes no NVDEC engine
    (`backend`, cb_decode_backend).  Not thread-safe: use one per host thread."""

    def __init__(self, ctx: Context):
        self.ctx, self.lib = ctx, ctx.lib
        self.backend = ctx.decode_backend()
        if self.backend == "libavcodec":
            try:
                import cv2  # noqa: F401 - maps opencv-python's libavcodec (and its dependencies) for the host decoder to find
            except ImportError:
                pass  # $CURATE_B200_LIBAVCODEC or a system libavcodec, else cb_decoder_create says what is missing
        h = C.c_void_p()
        check(self.lib.cb_decoder_create(ctx.h, C.byref(h)), "cb_decoder_create", ctx.h)
        self.h = h
        ctx._children.add(self)

    def close(self):
        if getattr(self, "h", None):
            self.lib.cb_decoder_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def decode(self, data, frame_ids, pool: Pool, dst_slots, seek_keyframes: bool = False) -> dict:
        """Decode `data` (mp4 bytes) and copy display-order frames `frame_ids` (ascending, repeats allowed)
        into `pool` slots `dst_slots`.  `seek_keyframes` skips GOPs that hold no wanted frame (identical output).
        Raises CurateB200Error on demux / decode failure."""
        buf = _as_u8(data)
        ids = np.ascontiguousarray(frame_ids, dtype=np.int32)
        slots = np.ascontiguousarray(dst_slots, dtype=np.int32)
        assert len(ids) == len(slots)
        st = _lib.DecodeStats()
        flags = _lib.DECODE_SEEK_SYNC if seek_keyframes else 0
        check(self.lib.cb_decoder_decode_ex(self.h, buf.ctypes.data, buf.size, ids.ctypes.data_as(C.POINTER(C.c_int32)), len(ids),
                                            C.byref(pool.desc), slots.ctypes.data_as(C.POINTER(C.c_int32)), flags, C.byref(st)),
              "cb_decoder_decode", self.ctx.h)  # fmt: skip
        return {"frames_decoded": st.frames_decoded, "frames_emitted": st.frames_emitted, "backend": self.backend, "coded": (st.coded_width, st.coded_height),
                "size": (st.width, st.height)}  # fmt: skip


def decode_discard(dec: Decoder, data) -> int:
    """Decode every picture of the clip and deliver none; returns the number decoded (NVDEC ceiling measurement)."""
    buf = _as_u8(data)
    st = _lib.DecodeStats()
    check(dec.lib.cb_decoder_decode_ex(dec.h, buf.ctypes.data, buf.size, None, 0, None, None, _lib.DECODE_DISCARD_ALL, C.byref(st)),
          "cb_decoder_decode_ex", dec.ctx.h)
    return st.frames_decoded


def decode_thumbnails(dec: Decoder, data, out_w: int, out_h: int, n_frames: int) -> torch.Tensor:
    """Every frame of the clip as uint8 cuda [n, out_h, out_w, 3] (cb_decoder_decode_thumbnails)."""
    buf = _as_u8(data)
    out = torch.empty((n_frames, out_h, out_w, 3), dtype=torch.uint8, device=f"cuda:{dec.ctx.device}")
    st = _lib.DecodeStats()
    check(dec.lib.cb_decoder_decode_thumbnails(dec.h, buf.ctypes.data, buf.size, out_w, out_h, out.data_ptr(), n_frames, C.byref(st)),
          "cb_decoder_decode_thumbnails", dec.ctx.h)  # fmt: skip
    return out[: st.frames_emitted]


def alloc_nv12_pool(ctx: Context, slots: int, width: int, height: int, colour: str = "opencv") -> Pool:
    """Device NV12 surface pool for `slots` frames of width x height (pitch aligned to 256 bytes); `colour` as Context.nv12_pool."""
    w2, h2 = (width + 1) & ~1, (height + 1) & ~1
    pitch = (w2 + 255) // 256 * 256
    buf = torch.empty((slots, h2 + h2 // 2, pitch), dtype=torch.uint8, device=f"cuda:{ctx.device}")
    return ctx.nv12_pool(buf, w2, h2, h2, colour)


# ---- host placement + persistent NVDEC sessions ---------------------------------------------------------
def _parse_cpulist(text: str) -> set[int]:
    out: set[int] = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        out.update(range(int(lo), int(hi or lo) + 1))
    return out


def device_numa_cpus(ctx: Context) -> tuple[int | None, list[int]]:
    """(NUMA node of the context's GPU, host CPUs of that node this process may run on).  ([] when the topology is not
    visible - e.g. numa_node = -1 on single-socket hosts - in which case nothing is pinned.)"""
    import os

    buf = C.create_string_buffer(32)
    try:
        check(ctx.lib.cb_device_pci_bus_id(ctx.h, buf, 32), "cb_device_pci_bus_id", ctx.h)
        bus = buf.value.decode().lower()
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None, []
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = _parse_cpulist(f.read())
        return node, sorted(cpus & os.sched_getaffinity(0))
    except (OSError, ValueError, _lib.CurateB200Error):
        return None, []


class SessionTable:
    """One NVDEC session per stream shape for a single-threaded caller (the same rule DecoderPool applies per worker thread:
    a session that is fed another resolution is destroyed and re-created by the driver, ~0.4 s each time)."""

    MAX_SHAPES = 4

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self._decs: dict = {}

    def get(self, shape) -> Decoder:
        d = self._decs.pop(shape, None)
        if d is None or d.h is None:
            while len(self._decs) >= self.MAX_SHAPES:
                self._decs.pop(next(iter(self._decs))).close()  # least recently used
            d = Decoder(self.ctx)
        self._decs[shape] = d
        return d

    def close(self) -> None:
        for d in self._decs.values():
            d.close()
        self._decs.clear()


class DecoderPool:
    """Persistent NVDEC sessions behind a thread pool: one `Decoder` per worker thread, created on first use and kept across
    calls (session creation costs ~10 ms and a context-lock round trip), worker threads pinned to the host CPUs of the GPU's
    NUMA node (bitstream parsing + H2D staging are host work: on a two-socket 8-GPU box the far socket costs decode rate)."""

    def __init__(self, ctx: Context, sessions: int, pin: bool = True):
        import threading
        from concurrent.futures import ThreadPoolExecutor

        self.ctx, self.sessions = ctx, int(sessions)
        self.numa_node, cpus = device_numa_cpus(ctx) if pin else (None, [])
        self.cpus = cpus
        self._tls = threading.local()
        self._decoders: list[Decoder] = []
        self._lock = threading.Lock()
        self._tp = ThreadPoolExecutor(max_workers=self.sessions, thread_name_prefix="cb-nvdec", initializer=self._init_thread)

    def _init_thread(self) -> None:
        import os

        if self.cpus:
            try:
                os.sched_setaffinity(0, self.cpus)  # pid 0 = the calling thread
            except OSError:
                pass

    MAX_SHAPES = 4  # sessions a worker thread keeps, one per stream shape (least recently used closed beyond that)

    def decoder(self, shape=None) -> Decoder:
        """This thread's session for streams of `shape` (any hashable, normally (width, height)).  A cuvid decoder is bound to
        one coded size: feeding a session a clip of another resolution destroys and re-creates it (hundreds of ms, serialised
        in the driver - measured: a 720p / 1080p / 4K mix ran 4-12x below the NVDEC rate with one session per thread), so a
        thread keeps one session per shape instead."""
        decs = getattr(self._tls, "decs", None)
        if decs is None:
            decs = self._tls.decs = {}
        d = decs.pop(shape, None)
        if d is None or d.h is None:
            while len(decs) >= self.MAX_SHAPES:
                old = decs.pop(next(iter(decs)))
                with self._lock:
                    if old in self._decoders:
                        self._decoders.remove(old)
                old.close()
            d = Decoder(self.ctx)
            with self._lock:
                self._decoders.append(d)
        decs[shape] = d  # most recently used last
        return d

    def submit(self, fn, *args, shape=None, **kw):
        """fn(decoder, *args, **kw) on a pool thread with that thread's own session (for streams of `shape`, see decoder())."""
        return self._tp.submit(lambda: fn(self.decoder(shape), *args, **kw))

    def close(self) -> None:
        self._tp.shutdown(wait=True)
        with self._lock:
            for d in self._decoders:
                d.close()
            self._decoders.clear()
