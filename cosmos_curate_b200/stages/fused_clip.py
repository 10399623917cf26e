"""NvdecClipAestheticStage: clip mp4 bytes -> NVDEC -> sampled NV12 surfaces -> fused preprocess -> tower -> scores.

Replaces the pair ClipFrameExtractionStage (CPU PyAV decode of every frame + RGB frames pickled to the next actor,
clip_frame_extraction_stages.py:102-165) -> AestheticFilterStage (aesthetic_filter_stages.py:120-221) with one GPU
stage that never materialises RGB frames.  Task mutations and the error convention are the reference's:

    clip.aesthetic_score, video.filtered_clips, video.clip_stats.num_filtered_by_aesthetic, task.stage_perf,
    no encoded_data            -> clip.errors["encoded_data"] = "empty", score -1.0
    demux / decode failure     -> clip.errors["frame_extraction"] = "video_decode_failed", encoded_data dropped, score -1.0
    task.stage_perf follows the reference's StageTimer call pattern (reinit BEFORE the work, aesthetic_filter_stages.py:161).
    (optional) clip.openai_embedding = L2-normalised mean of the per-frame embeddings (SURVEY.md 8b: the reference has
    no pooling rule for frame embeddings; this documented choice fills the existing generic clip-embedding slot).

Inside one `process_data` call the work is pipelined (this IS the product path bench.py times as `e2e`): the clips of
tower batches k+1 and k+2 are being decoded by the persistent NVDEC sessions (DecoderPool: one session per worker thread,
kept across calls, pinned to the GPU's NUMA node) while the SMs run preprocess + tower on batch k out of a three-deep ring
of surface pools; scores / embeddings come back through pinned host buffers with one async copy per batch.
"""

from __future__ import annotations

from typing import Literal

import numpy as np
import torch

from .. import sampling
from .._lib import CurateB200Error
from ..data_model import StageTimer
from ..interfaces import CuratorStage, CuratorStageResource, ModelInterface
from ..models.clip_aesthetics import CLIPAestheticScorer
from ..runtime import DecoderPool, alloc_nv12_pool, get_context, mp4_index

try:
    from loguru import logger
except Exception:  # noqa: BLE001
    import logging

    logger = logging.getLogger(__name__)


class NvdecClipAestheticStage(CuratorStage):
    def __init__(  # noqa: PLR0913
        self,
        score_threshold: float | None,
        reduction: Literal["mean", "min"] = "min",
        target_fps: float = 1.0,
        num_gpus_per_worker: float = 1.0,
        *,
        write_embedding: bool = False,
        max_batch: int = 256,
        num_decoders: int = 20,
        stage_batch_size: int = 8,
        seek_keyframes: bool = False,
        source: Literal["clip", "video_span"] = "clip",
        target_res: tuple[int, int] | None = None,
        cubic_mode: str | None = None,
        colour: str = "swscale",
        verbose: bool = False,
        log_stats: bool = False,
        model: CLIPAestheticScorer | None = None,
    ) -> None:
        self._timer = StageTimer(self)
        self._score_threshold, self._reduction, self._target_fps = score_threshold, reduction, target_fps
        self._num_gpus_per_worker = num_gpus_per_worker
        self._write_embedding, self._max_batch, self._num_decoders = write_embedding, max_batch, num_decoders
        self._stage_batch_size, self._verbose, self._log_stats = stage_batch_size, verbose, log_stats
        # False (default): every frame up to the last sampled one is decoded, the reference's decode work (decoder_utils.py:439-455) and
        # what bench.py's headline `e2e` times.  True: only the GOPs that hold sampled frames are decoded - bit-identical frames
        # (tested), 5x the clips/s on 1 fps sampling of GOP-30 clips; recommended in INTEGRATION.md, reported as `e2e_keyframe_seek`.
        self._seek = seek_keyframes
        if source not in ("clip", "video_span"):
            error_msg = f"source={source!r} not in ('clip', 'video_span')"
            raise ValueError(error_msg)
        # "video_span": analysis without the transcode (SURVEY.md 8f N2) - the clip's frames are decoded straight out of the SOURCE
        # video (video.encoded_data) at clip.span, so ClipTranscodingStage's re-encode + this stage's re-decode disappear for runs
        # that only need scores / embeddings.  Pixels are the source's, not the 4 Mb/s re-encode's: not bit-comparable with "clip".
        self._source = source
        # colour conversion of the decoded NV12 surfaces inside the fused kernel: "swscale" = bit-identical to the RGB frames the
        # reference's CPU decode hands to CLIP (libswscale yuv420p -> rgb24, decoder_utils.py:439-451), "opencv" = CV-CUDA semantics
        if colour not in ("swscale", "opencv"):
            error_msg = f"colour={colour!r} not in ('swscale', 'opencv')"
            raise ValueError(error_msg)
        self._colour = colour
        # clip_extraction_target_res of the reference pipeline (splitting_pipeline -> ClipFrameExtractionStage(target_res=(r, r))):
        # frames are squashed to (h, w) with cv2 INTER_CUBIC before the CLIP transforms (decoder_utils.py:666-670).  None / (-1, -1)
        # = native resolution into the antialiased short-side resize (the reference default).
        from .frame_extraction import CUBIC_MODES, default_cubic_mode

        self._target_res = None if target_res is None or target_res[0] <= 0 or target_res[1] <= 0 else (int(target_res[0]), int(target_res[1]))
        self._cubic_mode = CUBIC_MODES[cubic_mode or default_cubic_mode()]
        self._video_index: dict[int, tuple] = {}
        # Any ModelInterface with a `.tower` works: CLIPAestheticScorer (score + embedding) or an embedding-only tower such as
        # SigLIPImageEmbeddings (score_threshold=None: nothing is filtered, clip.openai_embedding is the output).
        self._model = model if model is not None else CLIPAestheticScorer(max_batch=max_batch)
        self._reduce_fn = np.min
        self._pools: dict[tuple[int, int], list] = {}
        self.last_call_stats: dict = {}

    @property
    def resources(self) -> CuratorStageResource:
        return CuratorStageResource(gpus=self._num_gpus_per_worker)

    @property
    def model(self) -> ModelInterface:
        return self._model

    @property
    def stage_batch_size(self) -> int:
        return self._stage_batch_size

    def stage_setup(self) -> None:
        if self._reduction not in ("mean", "min"):
            error_msg = f"Reduction `{self._reduction}` not implemented."
            raise NotImplementedError(error_msg)
        self._reduce_fn = np.mean if self._reduction == "mean" else np.min
        self._model.setup()
        self._ctx = get_context()
        self._norm = (getattr(self._model, "mean", None), getattr(self._model, "std", None))
        if self._score_threshold is not None and not self._model.tower.has_aesthetic:
            error_msg = "score_threshold given but the model has no aesthetic head (pass score_threshold=None for embedding-only towers)"
            raise ValueError(error_msg)
        if self._score_threshold is None and not self._write_embedding:
            error_msg = "embedding-only mode (score_threshold=None) needs write_embedding=True"
            raise ValueError(error_msg)
        self._decode_pool = DecoderPool(self._ctx, self._num_decoders)  # 7 NVDEC engines need ~20 sessions in flight (DESIGN.md 5)
        self._host: list[tuple[torch.Tensor, torch.Tensor | None]] = []

    def destroy(self) -> None:
        if getattr(self, "_decode_pool", None):
            self._decode_pool.close()
            self._decode_pool = None
        self._pools.clear()

    # ---- helpers ---------------------------------------------------------------------------------
    def _plan_span(self, clip, video):
        """Frames of the source video inside clip.span, re-timed from the clip start and sampled like a clip of its own."""
        data = video.encoded_data.resolve() if video.encoded_data else None
        if data is None:
            logger.warning(f"Clip {clip.uuid}: source video has no encoded_data.")
            clip.errors["encoded_data"] = "empty"
            clip.aesthetic_score = -1.0
            return None
        try:
            cached = self._video_index.get(id(video))
            if cached is None or cached[0] is not data:
                idx = mp4_index(data)
                cached = self._video_index[id(video)] = (data, idx, sampling.timestamps_from_index(idx["pts"], idx["timescale"]))
            _, idx, ts = cached
            ids = sampling.span_frame_ids(ts, clip.span, self._target_fps)
            return data, ids, ((idx["width"] + 1) & ~1, (idx["height"] + 1) & ~1)
        except (CurateB200Error, ValueError) as e:
            logger.error(f"Error extracting frames from clip {clip.uuid}: {e}")
            clip.errors["frame_extraction"] = "video_decode_failed"
            clip.aesthetic_score = -1.0
            return None

    def _plan(self, clip, video=None):
        """-> (data u8 array, frame ids expanded, (w, h)) or None (errors recorded on the clip)."""
        if self._source == "video_span":
            return self._plan_span(clip, video)
        data = clip.encoded_data.resolve() if clip.encoded_data else None
        if data is None:
            logger.warning(f"Clip {clip.uuid} has no encoded_data.")
            clip.errors["encoded_data"] = "empty"
            clip.aesthetic_score = -1.0
            return None
        try:
            idx = mp4_index(data)
            ts = sampling.timestamps_from_index(idx["pts"], idx["timescale"])
            ids, counts = sampling.frame_ids(ts, sampling.FrameExtractionPolicy.sequence, self._target_fps)
            return data, np.repeat(ids, counts).astype(np.int32), ((idx["width"] + 1) & ~1, (idx["height"] + 1) & ~1)
        except (CurateB200Error, ValueError) as e:
            self._decode_failed(clip, e)
            return None

    def _decode_failed(self, clip, e) -> None:
        logger.error(f"Error extracting frames from clip {clip.uuid}: {e}")
        clip.errors["frame_extraction"] = "video_decode_failed"
        if self._source == "clip":
            clip.encoded_data.drop()
        clip.aesthetic_score = -1.0

    RING = 3  # surface pools per resolution: tower on batch k, NVDEC filling k+1 and k+2

    def _pool(self, size, r: int):
        ring = self._pools.get(size)
        if ring is None:
            if len(self._pools) >= 4:  # mixed-resolution runs: keep the four most recent resolutions (LRU), free the rest
                self._pools.pop(next(iter(self._pools)))
            ring = [None] * self.RING
        else:
            self._pools.pop(size)
        self._pools[size] = ring  # most recently used last
        if ring[r] is None:
            ring[r] = alloc_nv12_pool(self._ctx, self._max_batch, size[0], size[1], self._colour)
        return ring[r]

    def _host_buffers(self, r: int):
        while len(self._host) <= r:
            tower = self._model.tower
            score = torch.empty((self._max_batch,), dtype=torch.float32).pin_memory() if tower.has_aesthetic else None
            emb = torch.empty((self._max_batch, tower.out_dim), dtype=torch.float32).pin_memory() if self._write_embedding else None
            self._host.append((score, emb))
        return self._host[r]

    def _make_batches(self, by_size):
        """[(size, [(clip, data, ids, first_slot)])]: whole clips, at most max_batch frames, one resolution per batch."""
        batches = []
        for size, clips in by_size.items():
            batch, used = [], 0
            for clip, data, ids in clips:
                if len(ids) > self._max_batch:
                    self._decode_failed(clip, ValueError(f"{len(ids)} sampled frames exceed max_batch={self._max_batch}"))
                    continue
                if used + len(ids) > self._max_batch:
                    batches.append((size, batch))
                    batch, used = [], 0
                batch.append((clip, data, ids, used))
                used += len(ids)
            if batch:
                batches.append((size, batch))
        return batches

    def _run_batches(self, batches) -> None:
        """Decode of batches k+1, k+2 (NVDEC + host parsing threads) overlaps preprocess + tower of batch k (SMs)."""
        seek, tower, stream = self._seek, self._model.tower, torch.cuda.current_stream()
        ring_pos: dict[tuple[int, int], int] = {}
        slots_of, futs, inflight = {}, {}, {}
        decoded = 0

        def decode_one(dec, data, ids, pool, first):
            return dec.decode(data, ids, pool, np.arange(first, first + len(ids), dtype=np.int32), seek_keyframes=seek)["frames_decoded"]

        def submit(k):
            size, items = batches[k]
            r = ring_pos.get(size, 0)
            ring_pos[size] = (r + 1) % self.RING
            pool = self._pool(size, r)
            slots_of[k] = (pool, k % self.RING)
            futs[k] = [self._decode_pool.submit(decode_one, data, ids, pool, first, shape=size) for _, data, ids, first in items]

        def finalize(k):
            """Batch k's results are on the host once its event has fired: write them onto the clips."""
            ev, errs, n = inflight.pop(k)
            ev.synchronize()
            score_h, emb_h = self._host_buffers(k % self.RING)
            score_h = score_h[:n].numpy() if score_h is not None else None
            for (clip, _, ids, first), err in zip(batches[k][1], errs):
                if err is not None:
                    self._decode_failed(clip, err)
                    continue
                if score_h is not None:
                    clip.aesthetic_score = float(self._reduce_fn(score_h[first : first + len(ids)]))
                if emb_h is not None:
                    m = emb_h[first : first + len(ids)].numpy().mean(axis=0)
                    clip.openai_embedding = (m / np.linalg.norm(m)).astype(np.float32)

        for k in range(min(2, len(batches))):
            submit(k)
        for k in range(len(batches)):
            errs = []
            for f in futs.pop(k):
                try:
                    decoded += f.result()
                    errs.append(None)
                except CurateB200Error as e:
                    errs.append(e)
            pool, r = slots_of.pop(k)
            n = sum(len(ids) for _, _, ids, _ in batches[k][1])
            norm = {} if self._norm[0] is None else {"mean": self._norm[0], "std": self._norm[1]}
            if self._target_res is not None:
                th, tw = self._target_res
                small = self._ctx.resize_cubic_u8(pool, tw, th, slots=np.arange(n, dtype=np.int32), mode=self._cubic_mode)
                emb, _, score = tower.embed_pool(self._ctx.rgb_pool(small), **norm)
            else:
                emb, _, score = tower.embed_pool(pool, slots=np.arange(n, dtype=np.int32), **norm)
            score_h, emb_h = self._host_buffers(r)
            if score_h is not None:
                score_h[:n].copy_(score, non_blocking=True)
            if emb_h is not None:
                emb_h[:n].copy_(emb, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
            inflight[k] = (ev, errs, n)
            if k >= 1:
                finalize(k - 1)  # also frees the surface pool and host buffers batch k+2 is about to reuse
            if k + 2 < len(batches):
                submit(k + 2)
        if batches:
            finalize(len(batches) - 1)
        self.last_call_stats = {"frames_decoded": decoded, "batches": len(batches), "nvdec_sessions": self._num_decoders,
                                "decode_backend": self._decode_pool.ctx.decode_backend(),
                                "numa_node": self._decode_pool.numa_node, "pinned_cpus": len(self._decode_pool.cpus)}  # fmt: skip

    # ---- stage entry -----------------------------------------------------------------------------
    def process_data(self, tasks):
        self._timer.reinit(self, sum(task.get_major_size() for task in tasks))
        n_clips = sum(len(video.clips) for task in tasks for video in task.videos)
        with self._timer.time_process(num_samples=max(1, n_clips)):
            by_size: dict[tuple[int, int], list] = {}
            for task in tasks:
                for video in task.videos:
                    for clip in video.clips:
                        plan = self._plan(clip, video)
                        if plan is not None:
                            data, ids, size = plan
                            by_size.setdefault(size, []).append((clip, data, ids))
            self._run_batches(self._make_batches(by_size))

            for task in tasks:
                for video in task.videos:
                    passed = []
                    if self._score_threshold is None:  # embedding-only tower: nothing to filter on
                        continue
                    for clip in video.clips:
                        if clip.aesthetic_score is None:
                            clip.aesthetic_score = -1.0
                        if clip.aesthetic_score < self._score_threshold:
                            video.filtered_clips.append(clip)
                            video.clip_stats.num_filtered_by_aesthetic += 1
                        else:
                            passed.append(clip)
                    video.clips = passed
        if self._log_stats:
            stage_name, stats = self._timer.log_stats()  # one batched call -> the same window on every task of the call
            for task in tasks:
                task.stage_perf[stage_name] = stats
        self._video_index.clear()
        return tasks
