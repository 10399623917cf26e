"""GPU: MP4 index + NVDEC decode of sampled frames vs libavcodec (cv2), through the C ABI."""

from __future__ import annotations

import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from gpu_helpers import ctx  # noqa: F401

pytestmark = pytest.mark.gpu
os.environ.setdefault("OPENCV_LOG_LEVEL", "ERROR")


def _cv2_luma_and_bgr(path, ids):
    import cv2

    cap = cv2.VideoCapture(str(path))
    cap.set(cv2.CAP_PROP_CONVERT_RGB, 0)  # yuv420p comes back as the Y plane only
    capc = cv2.VideoCapture(str(path))
    luma, bgr, want = {}, {}, set(int(i) for i in ids)
    i = 0
    while True:
        ok, y = cap.read()
        ok2, c = capc.read()
        if not ok or not ok2:
            break
        if i in want:
            luma[i], bgr[i] = y.copy(), c.copy()
        i += 1
    return luma, bgr, i


def test_nvdec_sampled_frames_match_libavcodec(ctx):
    if ctx.decode_backend() != "nvdec":
        pytest.skip("compares NVDEC with libavcodec: the driver exposes no NVDEC engine here, so the decoder is libavcodec itself")
    from cosmos_curate_b200 import sampling
    from cosmos_curate_b200.runtime import Decoder, alloc_nv12_pool, mp4_index

    path = GOLDEN / "sintel_clip_10s.mp4"
    data = np.fromfile(path, dtype=np.uint8)
    idx = mp4_index(data, ctx)
    ts = sampling.timestamps_from_index(idx["pts"], idx["timescale"])
    ids, counts = sampling.frame_ids(ts, sampling.FrameExtractionPolicy.sequence, 2.0)
    assert len(ids) == 21 and ids[-2:].tolist() == [228, 239]
    pool = alloc_nv12_pool(ctx, len(ids), idx["width"], idx["height"])
    dec = Decoder(ctx)
    st = dec.decode(data, ids, pool, np.arange(len(ids)))
    assert st["frames_emitted"] == len(ids) and st["size"] == (854, 480)
    assert st["frames_decoded"] == 240  # the last sampled frame is the last frame of the clip
    luma, bgr, n = _cv2_luma_and_bgr(path, ids)
    assert n == 240
    got = pool.buf.cpu().numpy()
    rgb = ctx.nv12_to_rgb(pool).cpu().numpy()
    h, w = idx["height"], idx["width"]
    for k, i in enumerate(ids):
        np.testing.assert_array_equal(got[k, :h, :w], luma[int(i)].reshape(h, w))  # H.264 decode is bit-exact by spec
        d = np.abs(rgb[k].astype(int) - bgr[int(i)][..., ::-1].astype(int))
        assert d.mean() < 1.5 and d.max() <= 32  # swscale (bilinear chroma, own rounding) vs OpenCV-style nearest-chroma conversion (DESIGN.md)
    # early stop: only the frames up to the last wanted id are decoded
    st = dec.decode(data, [0, 24, 48], pool, [0, 1, 2])
    assert st["frames_emitted"] == 3 and st["frames_decoded"] <= 48 + 1 + 4
    # repeated ids (supersampling counts) land in several slots
    st = dec.decode(data, [5, 5, 7], pool, [0, 1, 2])
    g2 = pool.buf.cpu().numpy()
    np.testing.assert_array_equal(g2[0], g2[1])
    assert (g2[0] != g2[2]).any()
    dec.close()


def test_nvdec_error_paths(ctx):
    from cosmos_curate_b200._lib import CurateB200Error
    from cosmos_curate_b200.runtime import Decoder, alloc_nv12_pool

    data = np.fromfile(GOLDEN / "sintel_clip_10s.mp4", dtype=np.uint8)
    dec = Decoder(ctx)
    pool = alloc_nv12_pool(ctx, 2, 854, 480)
    with pytest.raises(CurateB200Error) as e:
        dec.decode(np.zeros(1000, np.uint8), [0], pool, [0])
    assert e.value.code == -5
    with pytest.raises(CurateB200Error):
        dec.decode(data, [3, 1], pool, [0, 1])  # not ascending
    with pytest.raises(CurateB200Error):
        dec.decode(data, [500], pool, [0])  # beyond the clip
    wrong = alloc_nv12_pool(ctx, 1, 1920, 1080)
    with pytest.raises(CurateB200Error) as e:
        dec.decode(data, [0], wrong, [0])
    assert e.value.code == -4
    assert dec.decode(data, [0], pool, [0])["frames_emitted"] == 1  # the session survives errors
    assert dec.decode(data, [], pool, [])["frames_emitted"] == 0  # empty request
    dec.close()


def test_decode_to_embedding_end_to_end(ctx):
    """mp4 bytes -> NVDEC -> fused preprocess -> tower, against the oracle fed with libavcodec luma-exact frames."""
    from cosmos_curate_b200 import sampling
    from cosmos_curate_b200.runtime import Decoder, VitTower, alloc_nv12_pool, mp4_index
    from oracle import color, preprocess, vit

    data = np.fromfile(GOLDEN / "sintel_clip_10s.mp4", dtype=np.uint8)
    idx = mp4_index(data, ctx)
    ts = sampling.timestamps_from_index(idx["pts"], idx["timescale"])
    ids, _ = sampling.frame_ids(ts, sampling.FrameExtractionPolicy.sequence, 1.0)
    pool = alloc_nv12_pool(ctx, len(ids), idx["width"], idx["height"])
    Decoder(ctx).decode(data, ids, pool, np.arange(len(ids)))
    cfg = vit.CLIP_TINY
    w = vit.random_weights(cfg, seed=3)
    tower = VitTower(ctx, cfg.to_dict(), w, max_batch=16)
    emb, _, _ = tower.embed_pool(pool)
    nv12 = pool.buf.cpu().numpy()
    h, wd = idx["height"], idx["width"]
    rgb = np.stack([color.nv12_to_rgb(np.ascontiguousarray(f[:, :wd]), h, wd) for f in nv12])
    ref = vit.forward(cfg, w, preprocess.clip_preprocess(rgb))["embedding"]
    rel = np.linalg.norm(emb.cpu().numpy() - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert rel.max() < 2e-3


def test_keyframe_seek_is_bit_identical_and_lossless_vs_source(ctx):
    """Multi-GOP synthetic clip: CB_DECODE_SEEK_SYNC decodes fewer pictures but delivers the same surfaces; the IDR
    pictures are I_PCM, so NVDEC output must equal the encoder's source samples exactly."""
    from cosmos_curate_b200.runtime import Decoder, alloc_nv12_pool, decode_discard, mp4_index
    from tools import synth_h264

    w, h, fps = 640, 368, 30
    mp4, src = synth_h264.make_clip(w, h, fps, 4.0, seed=11, gop=30, pan=(2, 1), return_sources=True)
    data = np.frombuffer(mp4, dtype=np.uint8)
    idx = mp4_index(data, ctx)
    assert idx["n_samples"] == 120 and idx["n_sync"] == 4 and (idx["width"], idx["height"]) == (w, h)
    ids = np.array([0, 30, 60, 75, 75, 90, 119], dtype=np.int32)  # IDRs, a mid-GOP frame twice, the last frame
    dec = Decoder(ctx)
    full, sparse = alloc_nv12_pool(ctx, len(ids), w, h), alloc_nv12_pool(ctx, len(ids), w, h)
    sparse.buf.fill_(7)
    st_full = dec.decode(data, ids, full, np.arange(len(ids)))
    st_seek = dec.decode(data, ids, sparse, np.arange(len(ids)), seek_keyframes=True)
    assert st_full["frames_decoded"] == 120
    assert st_seek["frames_decoded"] == 1 + 1 + 16 + 30  # GOP0: 1, GOP1: 1, GOP2: frames 60..75, GOP3: 90..119
    a, b = full.buf.cpu().numpy(), sparse.buf.cpu().numpy()
    np.testing.assert_array_equal(a[:, : h + h // 2, :w], b[:, : h + h // 2, :w])
    for k, i in enumerate(ids):
        if int(i) in src:  # IDR pictures: lossless
            y, u, v = src[int(i)]
            np.testing.assert_array_equal(a[k, :h, :w], y)
            np.testing.assert_array_equal(a[k, h : h + h // 2, 0:w:2], u)
            np.testing.assert_array_equal(a[k, h : h + h // 2, 1:w:2], v)
    # frame 75 = frame 60 panned by 15 * (2, 1) pixels (interior)
    k60, k75 = 2, 3
    np.testing.assert_array_equal(a[k75, 40 : h - 40, 40 : w - 80], a[k60, 40 + 15 : h - 40 + 15, 40 + 30 : w - 80 + 30])
    assert decode_discard(dec, data) == 120
    dec.close()


def test_nvdec_matches_libavcodec_on_residual_coded_clip(ctx, tmp_path):
    """The 4 Mb/s-class residual-coded synthetic stream (CAVLC coefficients, Intra16x16 IDRs, P_Skip runs, quarter-pel motion,
    in-loop deblocking): NVDEC luma == libavcodec luma on every sampled frame, sequential and keyframe-seek alike, and the
    I_PCM sentinel that ends every picture is intact (no entropy-decoding slip anywhere in the slice)."""
    if ctx.decode_backend() != "nvdec":
        pytest.skip("compares NVDEC with libavcodec: the driver exposes no NVDEC engine here, so the decoder is libavcodec itself")
    import cv2

    from cosmos_curate_b200.runtime import Decoder, alloc_nv12_pool, mp4_index
    from tools import synth_h264

    w, h, fps = 1280, 720, 30
    mp4, info = synth_h264.make_coded_clip(w, h, fps, 4.0, seed=21, bitrate=2.0e6, return_info=True)
    path = tmp_path / "coded.mp4"
    path.write_bytes(mp4)
    data = np.frombuffer(mp4, dtype=np.uint8)
    idx = mp4_index(data, ctx)
    assert idx["n_samples"] == 120 and idx["n_sync"] == 4 and not idx["has_ctts"]
    assert abs(8 * idx["sample_bytes"] / 4.0 - 2.0e6) / 2.0e6 < 0.15
    ids = np.array([0, 1, 29, 30, 45, 75, 90, 119], dtype=np.int32)
    cap = cv2.VideoCapture(str(path))
    cap.set(cv2.CAP_PROP_CONVERT_RGB, 0)
    luma, i = {}, 0
    while True:
        ok, y = cap.read()
        if not ok:
            break
        if i in set(ids.tolist()):
            luma[i] = y.copy()
        i += 1
    assert i == 120
    dec = Decoder(ctx)
    full, sparse = alloc_nv12_pool(ctx, len(ids), w, h), alloc_nv12_pool(ctx, len(ids), w, h)
    st = dec.decode(data, ids, full, np.arange(len(ids)))
    st2 = dec.decode(data, ids, sparse, np.arange(len(ids)), seek_keyframes=True)
    assert st["frames_decoded"] == 120 and st2["frames_decoded"] < 120
    a, b = full.buf.cpu().numpy(), sparse.buf.cpu().numpy()
    np.testing.assert_array_equal(a[:, : h + h // 2, :w], b[:, : h + h // 2, :w])
    pcm = info["pcm"]
    for k, f in enumerate(ids):
        np.testing.assert_array_equal(a[k, :h, :w], luma[int(f)].reshape(h, w))
        np.testing.assert_array_equal(a[k, h - 12 : h, w - 12 : w], pcm[:256].reshape(16, 16)[4:, 4:])  # sentinel interior, luma
        uv = a[k, h + h // 2 - 6 : h + h // 2, w - 12 : w]
        np.testing.assert_array_equal(uv[:, 0::2], pcm[256:320].reshape(8, 8)[2:, 2:])  # Cb
        np.testing.assert_array_equal(uv[:, 1::2], pcm[320:384].reshape(8, 8)[2:, 2:])  # Cr
    dec.close()


def test_decoder_pool_keeps_one_session_per_stream_shape(ctx):
    """runtime.DecoderPool: a worker thread owns one NVDEC session per stream shape (re-creating a session at a resolution
    switch costs ~0.4 s, tools/mixed_decode_probe.py), at most MAX_SHAPES of them (least recently used closed), and the frames
    do not depend on which session decoded them."""
    from cosmos_curate_b200.runtime import Decoder, DecoderPool, alloc_nv12_pool
    from tools import synth_h264

    shapes = [(320, 192), (640, 360), (352, 288), (480, 272), (256, 144)]
    clips = {s: synth_h264.make_clip(s[0], s[1], 30, 0.2, seed=i, gop=30) for i, s in enumerate(shapes)}
    pools = {s: alloc_nv12_pool(ctx, 2, s[0], s[1]) for s in shapes}
    ids, slots = np.array([0, 5], dtype=np.int32), np.arange(2, dtype=np.int32)
    ref = {}
    one = Decoder(ctx)
    for s in shapes:
        one.decode(clips[s], ids, pools[s], slots)
        ref[s] = pools[s].buf.cpu().numpy().copy()
        pools[s].buf.zero_()
    one.close()
    dp = DecoderPool(ctx, 1)  # one worker thread: every job meets the same thread-local session table
    seen = []

    def job(dec, s):
        seen.append(id(dec))
        return dec.decode(clips[s], ids, pools[s], slots)["frames_emitted"]

    for s in shapes[:2] * 3:
        assert dp.submit(job, s, shape=s).result() == 2
    assert len(set(seen)) == 2 and seen[0] == seen[2] == seen[4] and seen[1] == seen[3] == seen[5]
    for s in shapes:  # five shapes through a table of MAX_SHAPES = 4
        assert dp.submit(job, s, shape=s).result() == 2
        np.testing.assert_array_equal(pools[s].buf.cpu().numpy()[:, :, : s[0]], ref[s][:, :, : s[0]])  # the pitch padding is not written
    assert len(dp._decoders) == DecoderPool.MAX_SHAPES
    assert dp.submit(job, shapes[0], shape=None).result() == 2  # shape-less callers keep working (one shared session)
    dp.close()
    assert not dp._decoders
