"""Frame-extraction stages with NVDEC decode, same names / outputs as the reference stages.

ClipFrameExtractionStage  (clip_frame_extraction_stages.py:43-192): fills `clip.extracted_frames` with host RGB frames
    keyed by FrameExtractionSignature strings, so UNMODIFIED downstream stages keep working.  Only the sampled frames
    are colour-converted (cb_nv12_to_rgb) and copied to the host.  The fused NvdecClipAestheticStage avoids even that.
VideoFrameExtractionStage (frame_extraction_stages.py:71-204): whole video -> uint8 [n,27,48,3] in `video.frame_array`
    (the TransNetV2 input) through cb_decoder (NVDEC; libavcodec where the driver exposes no NVDEC engine, cb_decode_backend) + the
    fused NV12->RGB+bilinear kernel; no temp file
    (decode failure -> video.errors["frame_extraction"], like the reference's "null" result).
"""

from __future__ import annotations

import numpy as np
import torch

from .. import sampling
from .. import _lib
from .._lib import CurateB200Error
from ..data_model import LazyData, StageTimer
from ..interfaces import CuratorStage, CuratorStageResource
from ..runtime import SessionTable, alloc_nv12_pool, decode_thumbnails, get_context, mp4_index
from ..sampling import FrameExtractionPolicy

try:
    from loguru import logger
except Exception:  # noqa: BLE001
    import logging

    logger = logging.getLogger(__name__)


CUBIC_MODES = {"opencv": _lib.CUBIC_OPENCV, "ipp": _lib.CUBIC_IPP}


def default_cubic_mode() -> str:
    import os
    import platform

    return os.environ.get("CURATE_B200_CUBIC_MODE") or ("ipp" if platform.machine() in ("x86_64", "AMD64") else "opencv")


class ClipFrameExtractionStage(CuratorStage):
    def __init__(  # noqa: PLR0913
        self,
        extraction_policies: tuple[FrameExtractionPolicy, ...] = (FrameExtractionPolicy.sequence,),
        target_fps: list[float | int] | None = None,
        target_res: tuple[int, int] | None = None,
        *,
        num_gpus_per_worker: float = 0.25,
        verbose: bool = False,
        log_stats: bool = False,
        cubic_mode: str | None = None,
        colour: str = "swscale",
    ) -> None:
        self._timer = StageTimer(self)
        # "swscale": RGB frames bit-identical to the reference stage's (PyAV frame.to_ndarray("rgb24") = libswscale's yuv420p
        # -> rgb24, decoder_utils.py:439-451); "opencv": CV-CUDA / cv2.cvtColor semantics (the reference's nvcodec_utils branch)
        if colour not in ("swscale", "opencv"):
            msg = f"colour={colour!r} not in ('swscale', 'opencv')"
            raise ValueError(msg)
        self._colour = colour
        self._extraction_policies = extraction_policies
        self._target_fps = [2] if target_fps is None else target_fps
        self._target_res = (-1, -1) if target_res is None else target_res
        # target_res = (height, width): cv2.resize(frame, (target_res[1], target_res[0]), INTER_CUBIC), aspect ratio not preserved
        # (decoder_utils.py:666-670).  opencv-python-headless computes it with Intel IPP on x86-64 and with its own fixed-point
        # code on aarch64; `cubic_mode` picks the matching arithmetic (default: this host's architecture, like the wheel would).
        self._cubic_mode = cubic_mode or default_cubic_mode()
        if self._cubic_mode not in ("ipp", "opencv"):
            msg = f"cubic_mode={cubic_mode!r} not in ('ipp', 'opencv')"
            raise ValueError(msg)
        self._num_gpus = num_gpus_per_worker
        self._verbose, self._log_stats = verbose, log_stats

    @property
    def resources(self) -> CuratorStageResource:
        return CuratorStageResource(gpus=self._num_gpus)

    def stage_setup(self) -> None:
        self._ctx = get_context()
        self._sessions = SessionTable(self._ctx)  # one NVDEC session per clip resolution (a mixed stream would re-create a single one per clip)
        self._pools: dict[tuple, object] = {}

    def destroy(self) -> None:
        if getattr(self, "_sessions", None):
            self._sessions.close()

    MAX_POOLS = 4  # resolutions kept resident (LRU); a 64-slot 1080p pool is 0.2 GB and the actor may own only 0.25 GPU

    def _surface_pool(self, width: int, height: int, n_frames: int):
        """One pool per resolution, capacity a power of two >= 64 (grown by replacement), least recently used evicted."""
        key = (width, height)
        pool = self._pools.pop(key, None)
        cap = 64
        while cap < n_frames:
            cap *= 2
        if pool is None or pool.buf.shape[0] < cap:
            pool = None  # drop the smaller pool before allocating its replacement
            while len(self._pools) >= self.MAX_POOLS:
                self._pools.pop(next(iter(self._pools)))
            pool = alloc_nv12_pool(self._ctx, cap, width, height, self._colour)
        self._pools[key] = pool  # most recently used last
        return pool

    def _extract(self, data) -> dict[str, np.ndarray]:
        idx = mp4_index(data)
        ts = sampling.timestamps_from_index(idx["pts"], idx["timescale"])
        plan = sampling.plan_extraction(ts, self._extraction_policies, self._target_fps)
        all_ids = np.unique(np.concatenate(list(plan.values()))).astype(np.int32)
        pool = self._surface_pool(idx["width"], idx["height"], len(all_ids))
        self._sessions.get((idx["width"], idx["height"])).decode(data, all_ids, pool, np.arange(len(all_ids), dtype=np.int32))
        slots = np.arange(len(all_ids), dtype=np.int32)
        if self._target_res[0] > 0 and self._target_res[1] > 0:  # only 3 * th * tw bytes per frame cross PCIe (150 KB instead of 6 MB)
            th, tw = self._target_res
            rgb = self._ctx.resize_cubic_u8(pool, tw, th, slots=slots, mode=CUBIC_MODES[self._cubic_mode]).cpu().numpy()
        else:
            rgb = self._ctx.nv12_to_rgb(pool, slots=slots)[:, : idx["height"], : idx["width"]].cpu().numpy()
        pos = {int(f): i for i, f in enumerate(all_ids)}
        return {sig: rgb[[pos[int(f)] for f in ids]] for sig, ids in plan.items()}

    def process_data(self, tasks):
        for task in tasks:
            self._timer.reinit(self, task.get_major_size())
            for video in task.videos:
                with self._timer.time_process():
                    for clip in video.clips:
                        data = clip.encoded_data.resolve() if clip.encoded_data else None
                        if data is None:
                            logger.warning(f"Clip {clip.uuid} has no encoded_data.")
                            clip.errors["encoded_data"] = "empty"
                            continue
                        try:
                            frames = self._extract(data)
                            clip.extracted_frames = LazyData(value=frames, nbytes=sum(a.nbytes for a in frames.values()))
                        except (CurateB200Error, ValueError) as e:
                            logger.error(f"Error extracting frames from clip {clip.uuid}: {e}")
                            clip.errors["frame_extraction"] = "video_decode_failed"
                            clip.encoded_data.drop()
            if self._log_stats:
                stage_name, stats = self._timer.log_stats()
                task.stage_perf[stage_name] = stats
        return tasks


class VideoFrameExtractionStage(CuratorStage):
    def __init__(self, output_hw: tuple[int, int] = (27, 48), decoder_mode: str = "nvdec", *, num_gpus_per_worker: float = 0.1,
                 batch_size: int = 64, verbose: bool = False, log_stats: bool = False) -> None:  # fmt: skip
        super().__init__()
        if decoder_mode not in ("nvdec", "pynvc"):
            msg = f"decoder_mode={decoder_mode!r}: this stage decodes through cb_decoder only (NVDEC, or libavcodec where the driver exposes no NVDEC engine)"
            raise ValueError(msg)
        self.output_hw, self.decoder_mode = output_hw, decoder_mode
        self._num_gpus, self._batch, self._verbose, self._log_stats = num_gpus_per_worker, batch_size, verbose, log_stats
        self._timer = StageTimer(self)

    @property
    def conda_env_name(self) -> str:
        return "unified"

    @property
    def resources(self) -> CuratorStageResource:
        return CuratorStageResource(gpus=self._num_gpus)

    def stage_setup(self) -> None:
        self._ctx = get_context()
        self._sessions = SessionTable(self._ctx)

    def destroy(self) -> None:
        if getattr(self, "_sessions", None):
            self._sessions.close()

    def _frames(self, data) -> np.ndarray:
        idx = mp4_index(data)
        h, w = self.output_hw
        if h == -1 or w == -1:  # the reference's "pick a size for me" rule (nvcodec_utils.py:129-136)
            w, h = sampling.pynvc_target_size(idx["width"], idx["height"], w, h)
        return decode_thumbnails(self._sessions.get((idx["width"], idx["height"])), data, w, h, idx["n_samples"]).cpu().numpy()

    def process_data(self, tasks):
        self._timer.reinit(self, sum(x.get_major_size() for x in tasks))
        for task in tasks:
            video = task.video
            data = video.encoded_data.resolve()
            if data is None:
                error_msg = "Please load video bytes!"
                raise ValueError(error_msg)
            with self._timer.time_process():
                try:
                    video.frame_array = self._frames(data)
                except CurateB200Error as e:
                    logger.error(f"Video frame extraction failed on {video.input_video}: {e}")
                    video.errors["frame_extraction"] = "null"
                    continue
        if self._log_stats and tasks:
            stage_name, stats = self._timer.log_stats()
            tasks[-1].stage_perf[stage_name] = stats
        return tasks
