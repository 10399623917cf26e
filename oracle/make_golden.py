"""Generate tests/golden/* by executing the REFERENCE's own code (build container only).

    python -m oracle.make_golden            # writes tests/golden/*.npz

The reference is Python, so its hot-path modules are imported from /root/reference
(oracle/ref_import.py installs the two stubs SURVEY.md 8c documents).  The vectors are what
travels to the GPU box; /root/reference itself does not.

Files written (all small):
  sampling_ref.npz        reference decoder_utils.sample_closest / find_closest_indices on a
                          spread of PTS tracks (CFR 24/30/29.97, VFR, dropped frames, offsets)
  clip_preprocess_ref.npz reference _CLIPImageEmbeddings.transforms (clip.py:48-62) on u8 frames
  clip_tiny_ref.npz       reference _CLIPImageEmbeddings.__call__ (clip.py:64-74), unmodified class,
                          on a tiny seeded CLIPModel saved with save_pretrained (weights included)
  aesthetic_ref.npz       reference aesthetics.MLP (aesthetics.py:30-66) seeded state_dict + outputs
  transnetv2_ref.npz      reference _TransNetV2 on seeded weights (oracle.transnetv2.random_state_dict) + the reference's
                          _get_predictions / _get_scenes / _get_filtered_scenes outputs
  resize_cubic_ref.npz    cv2.resize(INTER_CUBIC) exactly as extract_frames calls it (decoder_utils.py:666-670), once with Intel IPP
                          (x86 opencv-python default) and once with cv2.ipp.setUseIPP(False) (OpenCV's own code = aarch64 wheels)
  dedup_ref.npz           the array section of SemanticDedupActor.dedup (dedup_actor.py:404-466) executed from the reference's source
                          with numpy standing in for cupy (oracle/ref_import.dedup_core) on clusters with planted duplicates
  siglip_tiny_hf.npz      transformers SiglipVisionModel tiny seeded (stand-in; not in the reference)
  reference_cases.json    the reference's answers on the seeded cases of oracle/reference_cases.py (sampling, spans, chunking,
                          stage-output comparator, shot logic, InternVideo2 tubes)

Test infrastructure only (see oracle/__init__.py).
"""

from __future__ import annotations

import json
from fractions import Fraction
import tempfile
from pathlib import Path

import numpy as np
import torch

from oracle import ref_import, vit

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"


def pts_tracks() -> dict[str, np.ndarray]:
    """PTS tracks as the reference builds them: float(pts) * float(time_base) -> float32, sorted
    (decoder_utils.py:268-278)."""
    rng = np.random.default_rng(7)
    tracks = {}

    def from_ticks(ticks, timescale):
        tb = float(Fraction(1, timescale))  # PyAV time_base is a Fraction
        return np.sort(np.array([float(t) * tb for t in ticks], dtype=np.float32))

    tracks["cfr24_240_ts12288"] = from_ticks(np.arange(240) * 512, 12288)  # the Sintel fixture's timing
    tracks["cfr24_720_ts12288"] = from_ticks(np.arange(720) * 512, 12288)
    tracks["cfr30_300_ts15360"] = from_ticks(np.arange(300) * 512, 15360)
    tracks["cfr30_300_ts90000"] = from_ticks(np.arange(300) * 3000, 90000)
    tracks["ntsc_2997_300"] = from_ticks(np.arange(300) * 1001, 30000)
    tracks["cfr60_600_ts60"] = from_ticks(np.arange(600), 60)
    tracks["cfr24_120_5s"] = from_ticks(np.arange(120) * 512, 12288)  # config C1: 5 s
    tracks["offset_start_30"] = from_ticks(3003 + np.arange(150) * 3000, 90000)  # non-zero first PTS
    jitter = np.cumsum(rng.integers(2000, 4000, size=200))
    tracks["vfr_200"] = from_ticks(jitter, 90000)
    keep = np.ones(300, dtype=bool)
    keep[rng.choice(300, size=40, replace=False)] = False
    keep[0] = keep[-1] = True
    tracks["dropped_30"] = from_ticks((np.arange(300) * 3000)[keep], 90000)
    tracks["single_frame"] = np.array([0.0], dtype=np.float32)
    tracks["two_frames"] = np.array([0.0, 1.0 / 30], dtype=np.float32)
    tracks["lowfps_5_50"] = from_ticks(np.arange(50) * 18000, 90000)  # 5 fps source: supersampling
    return tracks


def gen_sampling() -> None:
    du = ref_import.decoder_utils()
    out, meta = {}, []
    case = 0
    for name, ts in pts_tracks().items():
        for rate in (0.5, 1.0, 2.0, 4.0, 8.0, 30.0):
            for endpoint in (True, False):
                if len(ts) < 2 and not endpoint:
                    continue
                try:
                    ids, counts, samples = du.sample_closest(ts, rate, start=ts[0], stop=ts[-1], endpoint=endpoint, dedup=True)
                except Exception as e:  # noqa: BLE001 - record reference failures too
                    meta.append({"case": case, "track": name, "rate": rate, "endpoint": endpoint, "raises": type(e).__name__})
                    case += 1
                    continue
                out[f"c{case}_ts"], out[f"c{case}_ids"], out[f"c{case}_counts"] = ts, ids, counts
                meta.append({"case": case, "track": name, "rate": rate, "endpoint": endpoint, "n": int(len(ids))})
                case += 1
    # find_closest_indices on random monotone arrays incl. exact ties and out-of-range queries
    rng = np.random.default_rng(11)
    for k in range(8):
        src = np.sort(rng.uniform(0, 10, size=rng.integers(2, 60))).astype(np.float32)
        dst = np.sort(np.concatenate([rng.uniform(-1, 12, size=40), (src[:-1] + src[1:]) / 2, src])).astype(np.float32)
        out[f"f{k}_src"], out[f"f{k}_dst"] = src, dst
        out[f"f{k}_idx"] = du.find_closest_indices(src, dst)
    # extract_frames policy path: `middle` quirk (one timestamp -> id 0)
    for name in ("cfr24_240_ts12288", "cfr30_300_ts90000", "single_frame"):
        ts = pts_tracks()[name]
        n = len(ts)
        mid = ts[(n // 2 - 1 if n % 2 == 0 else n // 2) :][:1]
        ids, counts, _ = du.sample_closest(mid, 1.0, start=mid[0], stop=mid[-1], endpoint=True, dedup=True)
        out[f"m_{name}_ts"], out[f"m_{name}_ids"], out[f"m_{name}_counts"] = ts, ids, counts
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(OUT / "sampling_ref.npz", **out)
    print("sampling_ref.npz:", case, "cases")


def test_frames() -> dict[str, np.ndarray]:
    rng = np.random.default_rng(3)
    frames = {}

    def scene(h, w, seed):
        yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
        base = np.stack(
            [128 + 100 * np.sin(xx / (7 + seed) + yy / 13), 128 + 90 * np.cos(xx / 11 - yy / (5 + seed)), (xx * 255 / w + yy * 3) % 256],
            axis=-1,
        )
        noise = rng.integers(-40, 41, size=(h, w, 3))
        img = np.clip(base + noise, 0, 255).astype(np.uint8)
        img[h // 4 : h // 4 + 9, :, :] = 255  # hard edges: overshoot/clamp exercise
        img[:, w // 3 : w // 3 + 5, :] = 0
        return img

    frames["land_270x480"] = np.stack([scene(270, 480, s) for s in range(2)])
    frames["port_480x270"] = scene(480, 270, 5)[None]
    frames["square_224"] = scene(224, 224, 6)[None]  # resize is the identity
    frames["small_100x160"] = scene(100, 160, 7)[None]  # upscale (scale < 1)
    frames["odd_301x225"] = scene(301, 225, 8)[None]  # odd crop offset (banker's rounding)
    frames["rand_360x640"] = rng.integers(0, 256, size=(1, 360, 640, 3), dtype=np.uint8)
    return frames


def _tiny_clip_dir(tmp: Path):
    from transformers import CLIPConfig, CLIPModel

    torch.manual_seed(0)
    cfg = CLIPConfig(
        text_config={"hidden_size": 32, "intermediate_size": 64, "num_hidden_layers": 1, "num_attention_heads": 2,
                     "vocab_size": 64, "max_position_embeddings": 8, "projection_dim": 64},
        vision_config={"hidden_size": 128, "intermediate_size": 256, "num_hidden_layers": 2, "num_attention_heads": 2,
                       "image_size": 224, "patch_size": 32, "projection_dim": 64},
        projection_dim=64,
    )  # fmt: skip
    model = CLIPModel(cfg).eval()
    with torch.no_grad():  # HF init leaves LN at (1,0) and biases at 0: perturb so every term is exercised
        g = torch.Generator().manual_seed(1)
        for n, p in model.named_parameters():
            if n.endswith("bias") or "layer_norm" in n or "layrnorm" in n or "layernorm" in n:
                p.add_(torch.randn(p.shape, generator=g) * 0.05)
    model.save_pretrained(tmp)
    return model


def gen_clip() -> None:
    cm = ref_import.clip_module()
    with tempfile.TemporaryDirectory() as td:
        hf = _tiny_clip_dir(Path(td))
        ref_import.register_weights_dir("tiny-clip", Path(td))
        ref = cm._CLIPImageEmbeddings("tiny-clip")  # the reference class, unmodified
        # transformers >= 5 returns an output object from get_image_features (SURVEY.md V11);
        # adapt the return type only, the reference's __call__ body runs as written.
        orig = ref.clip.get_image_features

        def _tensor_get_image_features(*a, **k):
            o = orig(*a, **k)
            return o if isinstance(o, torch.Tensor) else o.pooler_output

        ref.clip.get_image_features = _tensor_get_image_features
        pre, emb = {}, {}
        for name, fr in test_frames().items():
            x = torch.from_numpy(fr).permute(0, 3, 1, 2)
            pre[f"{name}_in"] = fr
            pre[f"{name}_out"] = ref.transforms(x).numpy()
            emb[f"{name}_in"] = fr
            emb[f"{name}_emb"] = ref(fr).cpu().numpy()
        np.savez_compressed(OUT / "clip_preprocess_ref.npz", **pre)
        cfg, w = vit.weights_from_hf_clip(hf)
        emb["cfg"] = np.frombuffer(json.dumps(cfg.to_dict()).encode(), dtype=np.uint8)
        for k, v in w.items():
            emb["w_" + k] = v
        np.savez_compressed(OUT / "clip_tiny_ref.npz", **emb)
    print("clip_preprocess_ref.npz, clip_tiny_ref.npz")


def gen_aesthetic() -> None:
    am = ref_import.aesthetics_module()
    torch.manual_seed(5)
    mlp = am.MLP().eval()
    sd = {k: v.detach().numpy() for k, v in mlp.state_dict().items()}
    rng = np.random.default_rng(9)
    e = rng.standard_normal((16, 768)).astype(np.float32)
    e /= np.linalg.norm(e, axis=1, keepdims=True)
    with torch.no_grad():
        y = mlp(torch.from_numpy(e)).squeeze(1).numpy()
    np.savez_compressed(OUT / "aesthetic_ref.npz", emb=e, score=y, **{"sd_" + k: v for k, v in sd.items()})
    print("aesthetic_ref.npz")


def gen_siglip() -> None:
    from transformers import SiglipVisionConfig, SiglipVisionModel

    torch.manual_seed(2)
    cfg = SiglipVisionConfig(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=4, image_size=64, patch_size=16)
    m = SiglipVisionModel(cfg).eval()
    with torch.no_grad():
        g = torch.Generator().manual_seed(3)
        for n, p in m.named_parameters():
            if n.endswith("bias") or "norm" in n or "probe" in n:
                p.add_(torch.randn(p.shape, generator=g) * 0.05)
    x = torch.randn(3, 3, 64, 64, generator=torch.Generator().manual_seed(4))
    with torch.no_grad():
        y = m(pixel_values=x).pooler_output.numpy()
    c, w = vit.weights_from_hf_siglip(m)
    out = {"x": x.numpy(), "pooled": y, "cfg": np.frombuffer(json.dumps(c.to_dict()).encode(), dtype=np.uint8)}
    out.update({"w_" + k: v for k, v in w.items()})
    np.savez_compressed(OUT / "siglip_tiny_hf.npz", **out)
    print("siglip_tiny_hf.npz")


def gen_transnet() -> None:
    """Reference _TransNetV2 (transnetv2.py:39-148) with the seeded state_dict + the reference's shot-logic functions."""
    from oracle import transnetv2 as tn

    mod = ref_import.transnetv2_module()
    fns = ref_import.transnetv2_stage_functions()
    sd = tn.random_state_dict(seed=3)
    model = mod._TransNetV2()
    missing = model.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()}, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    model.eval()
    out: dict[str, np.ndarray] = {"seed": np.array(3)}
    video = tn.synthetic_frames(170, seed=11, cuts=(40, 97, 131))
    out["video"] = video
    with torch.no_grad():
        for name, w in (("full", tn.windows(video)[1]), ("short95", tn.windows(video)[2]), ("short45", tn.windows(video)[3] if len(tn.windows(video)) > 3 else video[:45]),
                        ("tiny7", video[:7])):  # fmt: skip
            out[f"win_{name}"] = w
            out[f"prob_{name}"] = model(torch.from_numpy(w)[None]).numpy()[0, :, 0]
    # _get_predictions moves each window with .cuda(); on this CPU-only box that call is made a no-op for the run
    orig = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self  # type: ignore[method-assign]
    try:
        with torch.no_grad():
            for n in (170, 120, 100, 51, 10):
                probs = []

                def spy(x, probs=probs):
                    y = model(x)
                    probs.append(y[0, 25:75, 0].numpy())
                    return y

                thr = 0.5
                pred = fns["_get_predictions"](spy, video[:n], thr)
                out[f"pred_{n}"] = pred
                out[f"probs_{n}"] = np.concatenate(probs)[:n]
    finally:
        torch.Tensor.cuda = orig  # type: ignore[method-assign]
    out["pred_threshold"] = np.array(0.5)
    # shot logic on seeded 0/1 tracks
    rng = np.random.default_rng(5)
    cases = []
    tracks = [np.zeros(300, np.uint8), np.ones(50, np.uint8)]
    for n in (60, 300, 1000, 4000):
        for density in (0.002, 0.01, 0.05):
            t = (rng.random(n) < density).astype(np.uint8)
            tracks.append(t)
            t2 = t.copy()
            t2[0] = 1
            t2[-1] = 1
            tracks.append(t2)
    for ti, t in enumerate(tracks):
        out[f"track_{ti}"] = t
        for entire in (True, False):
            sc = fns["_get_scenes"](t.reshape(-1, 1), entire_scene_as_clip=entire)
            key = f"scenes_{ti}_{int(entire)}"
            out[key] = sc
            for ci, (mn, mx, mode, crop) in enumerate([(48, 1440, "stride", 12), (60, 1800, "truncate", 15), (None, 100, "stride", None), (48, None, "truncate", 0),
                                                        (10, 50, "stride", 3), (None, None, "truncate", None)]):  # fmt: skip
                fs = fns["_get_filtered_scenes"](sc.copy(), min_length=mn, max_length=mx, max_length_mode=mode, crop_length=crop)
                out[f"{key}_f{ci}"] = np.asarray(fs, dtype=np.int32).reshape(-1, 2)
                cases.append([ti, int(entire), ci])
    out["filter_cfgs"] = np.array([[48, 1440, 1, 12], [60, 1800, 0, 15], [-1, 100, 1, -1], [48, -1, 0, 0], [10, 50, 1, 3], [-1, -1, 0, -1]], dtype=np.int32)
    out["n_tracks"] = np.array(len(tracks))
    np.savez_compressed(OUT / "transnetv2_ref.npz", **out)
    print("transnetv2_ref.npz", {k: v.shape for k, v in out.items() if k.startswith("prob")})


def gen_resize_cubic() -> None:
    """target_res resize of extract_frames: frames = np.array([cv2.resize(frame, (target_res[1], target_res[0]), INTER_CUBIC) ...])."""
    import cv2

    rng = np.random.default_rng(20250923)
    cases = {"sq224_from_270x480": ((270, 480), (224, 224)), "up_odd": ((37, 53), (77, 51)), "sq224_from_64": ((64, 64), (224, 224)),
             "thumb_27x48": ((180, 320), (27, 48))}  # name: ((src_h, src_w), target_res = (h, w))
    out = {}
    for name, ((h, w), (th, tw)) in cases.items():
        smooth = cv2.GaussianBlur(rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8), (0, 0), 1.5)
        img = np.where(rng.random((h, w, 1)) < 0.5, smooth, rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)).astype(np.uint8)
        out[name + "_in"] = img
        out[name + "_res"] = np.array([th, tw])
        cv2.ipp.setUseIPP(True)
        out[name + "_ipp"] = cv2.resize(img, (tw, th), interpolation=cv2.INTER_CUBIC)
        cv2.ipp.setUseIPP(False)
        out[name + "_opencv"] = cv2.resize(img, (tw, th), interpolation=cv2.INTER_CUBIC)
        cv2.ipp.setUseIPP(True)
    out["cv2_version"] = np.frombuffer(cv2.__version__.encode(), dtype=np.uint8)
    out["ipp_version"] = np.frombuffer(str(cv2.ipp.getIppVersion()).encode(), dtype=np.uint8)
    np.savez_compressed(OUT / "resize_cubic_ref.npz", **out)
    print("resize_cubic_ref.npz", {k: v.shape for k, v in out.items() if k.endswith("_ipp")})


def gen_video_tube() -> None:
    """InternVideo2 input tubes from the reference's own `_construct_frames` / `_construct_image` (internvideo2_mm.py:390-415).
    Small target sizes keep the fixture small; the 224 x 224 cases store a sha256 of the float32 tube, the frames being
    regenerated from the seed by the test."""
    import hashlib

    import cv2

    iv2 = ref_import.internvideo2_formulator()
    rng = np.random.default_rng(20250924)

    def frames(n, h, w):
        out = []
        for _ in range(n):
            smooth = cv2.GaussianBlur(rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8), (0, 0), 1.2)
            out.append(np.where(rng.random((h, w, 1)) < 0.5, smooth, rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)).astype(np.uint8))
        return out

    out = {}
    # name: (n_frames, (src_h, src_w), target_size = (w, h))
    cases = {"down_21f": (21, (90, 122), (56, 40)), "decimate2x_8f": (8, (80, 112), (56, 40)), "up_9f": (9, (20, 30), (56, 40)),
             "same_17f": (17, (40, 56), (56, 40)), "tall_16f": (16, (131, 37), (40, 56))}
    for name, (n, (h, w), tsize) in cases.items():
        fr = frames(n, h, w)
        out[name + "_in"] = np.stack(fr)
        out[name + "_size"] = np.array(tsize)
        out[name + "_tube"] = iv2._construct_frames(fr, fnum=8, target_size=tsize)
        out[name + "_image"] = iv2._construct_image(fr[-1], target_size=tsize)
    out["short_tube"] = iv2._construct_frames(frames(5, 16, 16), fnum=8, target_size=(8, 8))  # too few frames: empty array
    for name, (n, (h, w)) in {"hd": (11, (1080, 1920)), "sd": (21, (480, 854)), "uhd": (8, (2160, 3840))}.items():
        big_rng = np.random.default_rng([20250924, h])
        fr = [big_rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for _ in range(n)]
        tube = iv2._construct_frames(fr, fnum=8, target_size=(224, 224))
        out[name + "_sha256"] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(tube).tobytes()).digest(), dtype=np.uint8)
        out[name + "_shape"] = np.array([n, h, w])
    out["cv2_version"] = np.frombuffer(cv2.__version__.encode(), dtype=np.uint8)
    np.savez_compressed(OUT / "video_tube_ref.npz", **out)
    print("video_tube_ref.npz", {k: v.shape for k, v in out.items() if k.endswith("_tube")})


def gen_fixed_stride() -> None:
    """Spans / clip uuids / populated clips from the reference's own fixed-stride helpers (clip_extraction_stages.py:444-660).
    Floats are stored as float.hex() strings: the window start accumulates by repeated addition, the comparison is bit for bit."""
    import types

    f = ref_import.fixed_stride_functions()
    out: dict = {"spans": [], "populate": []}
    for end_s in (30.0, 12.0, 9.99, 100.0 / 3.0, 0.0, 7.25):
        for clip_len, stride, min_len in ((10.0, 10.0, 10.0), (10.0, 5.0, 5.0), (10.0, 10.0, 2.0), (3.3, 0.1 * 7, 1.0), (1.0 / 3.0, 0.1, 0.2), (5.0, 12.5, 0.0)):
            spans = f["_make_spans_fixed_stride"](0.0, end_s, clip_len, stride, min_len)
            uuids = f["_make_clip_uuids"]("s3://bucket/session-7", spans)
            out["spans"].append({"args": [float.hex(0.0), float.hex(end_s), float.hex(clip_len), float.hex(stride), float.hex(min_len)],
                                 "spans": [[float.hex(a), float.hex(b)] for a, b in spans], "uuids": [str(u) for u in uuids]})

    def video(name, n_frames, fps, t0):
        ts = (t0 + np.arange(n_frames) / fps).astype(np.float32)
        return types.SimpleNamespace(input_video=name, timestamps=ts, errors={}, clips=[], metadata=types.SimpleNamespace(num_frames=n_frames, framerate=fps))

    cases = {"single_30s": ([("a.mp4", 900, 30.0, 0.0)], (10.0, 10.0, 10.0, 0)), "single_limit2": ([("a.mp4", 900, 30.0, 0.0)], (10.0, 5.0, 5.0, 2)),
             "multicam_offsets": ([("cam0.mp4", 900, 30.0, 0.0), ("cam1.mp4", 700, 24.0, 0.5), ("cam2.mp4", 1000, 29.97, 0.25)], (4.0, 2.5, 1.5, 0)),
             "ntsc": ([("n.mp4", 1799, 30000 / 1001, 0.0)], (10.0, 10.0, 5.0, 0))}
    for name, (vids, (clip_len, stride, min_len, limit)) in cases.items():
        vs = [video(*v) for v in vids]
        f["_populate_clips_fixed_stride"](vs, "session/" + name, clip_len, stride, min_len, limit_clips=limit)
        out["populate"].append({"name": name, "videos": [[v[0], v[1], float.hex(float(v[2])), float.hex(float(v[3]))] for v in vids],
                                "args": [float.hex(clip_len), float.hex(stride), float.hex(min_len), limit],
                                "clips": [[[str(c.uuid), c.source_video, float.hex(c.span[0]), float.hex(c.span[1])] for c in v.clips] for v in vs]})
    # chunk sizes of chunk_tasks (clip_extraction_stages.py:131-139): the reference's split_by_chunk_size over clip spans with its size function
    grouping = ref_import.grouping_module()
    out["chunks"] = []
    rng = np.random.default_rng(7)
    for n_clips, per_chunk in ((100, 32), (7, 1), (33, 4), (0, 32), (50, 2)):
        starts = np.cumsum(rng.uniform(0.3, 14.0, size=n_clips))
        spans = [(float(a), float(a + d)) for a, d in zip(starts, rng.uniform(0.2, 12.0, size=n_clips))]
        sizes = [len(c) for c in grouping.split_by_chunk_size(spans, per_chunk * 8, lambda x: int(x[1] - x[0]))]
        out["chunks"].append({"spans": [[float.hex(a), float.hex(b)] for a, b in spans], "num_clips_per_chunk": per_chunk, "chunk_sizes": sizes})
    (OUT / "fixed_stride_ref.json").write_text(json.dumps(out, indent=1))
    print("fixed_stride_ref.json", len(out["spans"]), "span cases,", len(out["populate"]), "populate cases")


def gen_dedup() -> None:
    core = ref_import.dedup_core()
    out = {}
    for name, (m, d, tile, seed) in {"multi_tile": (700, 64, 256, 1), "default_tile": (4500, 16, 4096, 2), "tiny": (3, 16, 4096, 3)}.items():
        rng = np.random.default_rng(seed)
        e = rng.standard_normal((m, d)).astype(np.float32)
        dup = rng.choice(m, size=max(1, m // 10), replace=False)
        src = rng.choice(m, size=len(dup))
        e[dup] = e[src] * rng.choice(np.array([1.0, 2.0, 0.5], dtype=np.float32), size=len(dup))[:, None]  # exact and scaled duplicates
        near = rng.choice(m, size=max(1, m // 10), replace=False)
        e[near] = e[rng.choice(m, size=len(near))] + np.float32(0.05) * rng.standard_normal((len(near), d)).astype(np.float32)
        dist = rng.random(m).astype(np.float32)
        dist[rng.choice(m, size=m // 5)] = np.float32(0.25)  # ties in the sort key: stable order matters
        order = np.argsort(-dist, kind="stable")  # cudf sort_values(ascending=False) on ties: pinned separately (not in this section)
        maxv, argi = core(e[order], tile)
        out[name + "_emb"], out[name + "_dist"], out[name + "_tile"] = e, dist, np.array(tile)
        out[name + "_maxv"], out[name + "_argi"] = maxv.astype(np.float32), argi.astype(np.int32)
    np.savez_compressed(OUT / "dedup_ref.npz", **out)
    print("dedup_ref.npz", {k: v.shape for k, v in out.items() if k.endswith("_maxv")})


def gen_reference_cases() -> None:
    """The reference's answers on the seeded cases of oracle/reference_cases.py: frame-index math, fixed-stride spans and uuids,
    chunk sizes, the stage-output comparator, shot logic and the InternVideo2 tube formulation (tubes as sha256)."""
    from oracle import reference_cases as R

    meta: dict = {"digest": {}, "sample_closest": [], "shots": []}
    du = ref_import.decoder_utils()
    cases = R.timestamp_cases()
    meta["digest"]["timestamps"] = R.digest(cases)
    for i, c in enumerate(cases):
        ts = c["ts"]
        res = du.sample_closest(ts, sample_rate=c["rate"], start=ts[0], stop=ts[-1], endpoint=c["endpoint"], dedup=c["dedup"])
        meta["sample_closest"].append({"outputs": [R.values_sha256(v) for v in res],
                                       "find_closest": R.values_sha256(du.find_closest_indices(ts, R.closest_targets(ts)))})  # fmt: skip

    f = ref_import.fixed_stride_functions()
    cases = R.fixed_stride_cases()
    meta["digest"]["fixed_stride"] = R.digest(cases)
    meta["fixed_stride"] = []
    for c in cases:
        spans = f["_make_spans_fixed_stride"](0.0, c["end"], c["clip_len"], c["stride"], c["min_len"])
        meta["fixed_stride"].append({"n_spans": len(spans), "spans_sha256": R.spans_sha256(spans),
                                     "uuids_sha256": R.uuids_sha256(f["_make_clip_uuids"](c["session"], spans[:50]))})  # fmt: skip

    grouping = ref_import.grouping_module()
    cases = R.chunk_cases()
    meta["digest"]["chunks"] = R.digest(cases)
    meta["chunks"] = [[len(ch) for ch in grouping.split_by_chunk_size(c["spans"], c["per_chunk"] * 8, R.chunk_size)] for c in cases]

    compare = ref_import.stage_compare_functions()["_compare_values"]
    cases = R.compare_cases()
    meta["digest"]["compare"] = R.digest(cases)
    meta["compare"] = [[repr([R.diff_key(d) for d in compare("t", c["golden"], other, atol=c["atol"])]) for other in (c["candidate"], c["golden"])]
                       for c in cases]  # fmt: skip
    table = R.comparator_table()
    meta["digest"]["comparator_table"] = R.digest(table)
    meta["comparator_table"] = {name: repr([R.diff_key(d) for d in compare("root", g, c, atol=atol)]) for name, g, c, atol in table}

    shots = ref_import.transnetv2_stage_functions()
    cases = R.shot_cases()
    meta["digest"]["shots"] = R.digest(cases)
    for c in cases:
        scenes = shots["_get_scenes"](c["track"].reshape(-1, 1), entire_scene_as_clip=c["entire"])
        filtered = shots["_get_filtered_scenes"](scenes.copy(), min_length=c["min_len"], max_length=c["max_len"], max_length_mode=c["mode"],
                                                 crop_length=c["crop"]) if len(scenes) else None  # fmt: skip
        meta["shots"].append({"scenes": R.values_sha256(scenes), "dtype": scenes.dtype.str, "n_scenes": len(scenes),
                              "filtered": None if filtered is None else R.values_sha256(filtered)})  # fmt: skip

    iv2 = ref_import.internvideo2_formulator()
    cases = R.tube_cases()
    meta["digest"]["tubes"] = R.digest(cases)
    meta["tubes"] = []
    for c in cases:
        tube = iv2._construct_frames(R.tube_frames(c), fnum=8, target_size=(c["tw"], c["th"]))
        meta["tubes"].append({"shape": list(tube.shape), "dtype": tube.dtype.str, "sha256": R.tube_sha256(tube)})
    (OUT / "reference_cases.json").write_text(json.dumps(meta, indent=0))
    print("reference_cases.json")


def main() -> None:
    assert ref_import.available(), "needs /root/reference (build container)"
    OUT.mkdir(parents=True, exist_ok=True)
    gen_sampling()
    gen_clip()
    gen_aesthetic()
    gen_siglip()
    gen_transnet()
    gen_resize_cubic()
    gen_dedup()
    gen_video_tube()
    gen_fixed_stride()
    gen_reference_cases()


if __name__ == "__main__":
    main()
