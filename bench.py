#!/usr/bin/env python
"""bench.py - throughput of the decode -> sample -> preprocess -> embed/classify hot path on B200.

    python bench.py --gpus 1 --steps K --warmup W                 # this repo's CUDA path
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # ... and what its last timed step returned, as DIR/*.npy
    python bench.py --impl reference --gpus 1 --steps K --warmup W # the reference's CPU path (oracle) on host cores
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1]): synthetic 1920x1080 30 fps 10 s H.264 clips at ~4 Mb/s (tools/synth_h264.make_coded_clip:
residual-coded Intra16x16 IDRs + P pictures, CAVLC, deblocking on - no encoder exists in this image), 64 distinct clips per
rank, sampled at 1 fps like AestheticFilterStage (11 frames per clip), CLIP ViT-L/14 image tower (seeded random weights) +
aesthetic affine head.  One STEP = `--clips-per-step` clips (default 24 -> 264 frames, the closest whole-clip count to the
256-frame batch BASELINE.json names).

--dump-outputs writes what the last timed step returned (rank 0) in float32, one row per sampled frame in slot order (clip j's
frames_per_clip frames at rows j * frames_per_clip ...): embedding.npy [frames_per_step, 768] and aesthetic_score.npy
[frames_per_step].  The inputs are seeded (clips, weights), so two builds run with the same arguments can be compared output for
output.

Printed JSON line (rank 0):
  value   clips/s, whole job, decoded NV12 surfaces of the step already resident in HBM (preprocess + tower + head),
          timed with CUDA events, max over ranks.
  e2e     clips/s through the PRODUCT stage: NvdecClipAestheticStage.process_data(tasks) on host SplitPipeTasks holding mp4 bytes
          (one call = `--tasks-per-call` = 20 tasks x clips-per-step clips = 480 clips, a few source videos' worth); MP4 index + NVDEC decode of every frame up to the last
          sampled one (the reference's decode semantics) + fused preprocess + tower + pinned D2H of scores/embeddings, the decode /
          tower overlap happening inside the stage; wall clock between device synchronisations, max over ranks.
  e2e_keyframe_seek  the same call with seek_keyframes=True (opt-in: identical frames, only GOPs with sampled frames are decoded).
  roofline      the dominant kernel (tcgen05 GEMM): algorithmic FLOPs per launch / CUDA-event time per launch vs the
                measured sustained bf16 peak (MEASURED_PEAKS.json); roofline_other has preprocess / LayerNorm (HBM).
  cpu_baseline  the oracle's CPU restatement of the reference path timed on the host cores (N=1, rank 0), bounded sample.
  gpu_library_baseline  the reference's GPU *library* path restated without Ray (torch-CUDA torchvision transforms + HF CLIPModel
                fp32, one call per clip, clip.py:36-74 / aesthetic_filter_stages.py:181-183), N=1 rank 0, bounded sample.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
os.environ.setdefault("OPENCV_LOG_LEVEL", "ERROR")

import numpy as np  # noqa: E402

FRAME_W, FRAME_H, FPS, SECONDS = 1920, 1080, 30, 10.0
SAMPLE_FPS = 1.0
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DUMP_LIMIT_BYTES = 64 << 20


def peaks() -> tuple[dict, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured"
    return dict(FALLBACK_PEAKS), "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)  # fmt: skip
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        busy = sorted(sm)[len(sm) // 2 :] if sm else []  # upper half = samples under load
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


BITRATE = 4.0e6  # the reference's transcode default (decoder_utils.py:43)


def _gen_clip(args) -> str:
    seed, path = args[:2]
    w, h, bitrate = args[2:] if len(args) > 2 else (FRAME_W, FRAME_H, BITRATE)
    from tools import synth_h264

    if not os.path.exists(path):
        data = synth_h264.make_coded_clip(w, h, FPS, SECONDS, seed=seed, gop=FPS, bitrate=bitrate)
        tmp = f"{path}.{os.getpid()}.tmp"
        with open(tmp, "wb") as f:
            f.write(data)
        os.replace(tmp, path)
    return path


def make_clips(n_distinct: int, rank: int, workers: int | None = None, size: tuple[int, int] = (FRAME_W, FRAME_H), bitrate: float = BITRATE) -> list[bytes]:
    """`n_distinct` residual-coded clips (seed = 1000 * rank + i), generated by a fork pool BEFORE CUDA is initialised and
    cached in the temporary directory (both arms on one machine reuse them)."""
    import multiprocessing as mp

    root = os.path.join(os.environ.get("CB_CLIP_CACHE", tempfile.gettempdir()), f"cb_clips_{size[0]}x{size[1]}_{FPS}_{int(SECONDS)}s_{int(bitrate)}")
    os.makedirs(root, exist_ok=True)
    jobs = [(1000 * rank + i, os.path.join(root, f"clip_{1000 * rank + i}.mp4"), size[0], size[1], bitrate) for i in range(n_distinct)]
    todo = [j for j in jobs if not os.path.exists(j[1])]
    if todo:
        world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
        workers = workers or max(1, min(32, len(os.sched_getaffinity(0)) // max(1, world)))
        if workers > 1 and len(todo) > 1:
            with mp.get_context("fork").Pool(min(workers, len(todo))) as pool:
                pool.map(_gen_clip, todo)
        else:
            for j in todo:
                _gen_clip(j)
    out = []
    for job in jobs:
        with open(job[1], "rb") as f:
            out.append(f.read())
    return out


def host_cpu_info() -> dict:
    """Logical CPUs, the CPUs this process may run on, and the cgroup CPU quota (what `cores` really means on this box)."""
    info = {"logical_cpus": os.cpu_count(), "affinity_cpus": len(os.sched_getaffinity(0)), "cgroup_quota_cpus": None}
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
        info["cgroup_quota_cpus"] = None if q == "max" else float(q) / float(per)
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                q, per = int(f.read()), int(g.read())
            info["cgroup_quota_cpus"] = None if q < 0 else q / per
        except (OSError, ValueError):
            pass
    return info


def effective_cores() -> int:
    h = host_cpu_info()
    n = h["affinity_cpus"] or h["logical_cpus"] or 1
    if h["cgroup_quota_cpus"]:
        n = min(n, max(1, int(h["cgroup_quota_cpus"])))
    return n


# ================================================================================================ reference arm
def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # under torchrun only rank 0 measures the CPU path
    from oracle import cpu_path, vit

    cores = effective_cores()
    procs, threads = cpu_layout(cores)
    clips = make_clips(8, 0)
    pool = cpu_path.CpuReferencePool(vit.CLIP_VIT_L14, seed=0, procs=procs, threads=threads)
    sample = max(procs, args.ref_clips)  # at least one clip per worker so every host core is busy
    batch = [clips[i % len(clips)] for i in range(sample)]
    pool.run(batch[:procs], SAMPLE_FPS)  # one warm-up pass (a CPU step takes ~25 s; more warm-up would only burn minutes)
    t, frames, phases = 0.0, 0, {"decode_s": 0.0, "preprocess_s": 0.0, "model_s": 0.0}
    for _ in range(args.steps):
        r = pool.run(batch, SAMPLE_FPS)
        t += r["seconds"]
        frames += r["frames"]
        for k in phases:
            phases[k] += r[k]
    pool.close()
    value = sample * args.steps / t
    line = {
        "impl": "reference", "metric": "clips_per_sec", "value": value, "unit": "clips/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "frames_per_sec": frames / t,
        "config": {"workload": WORKLOAD, "implementation": "reference CPU path (oracle port): libavcodec decode, torchvision transforms, torch-fp32 tower", "clips_per_step": sample,
                   "frames_per_clip": frames // (sample * args.steps), "network": "clip-vit-large-patch14 (seeded random weights), fp32", "sharding": "host worker processes"},
        "cpu_baseline": {"value": value, "unit": "clips/s", "cores": procs * threads, "kind": "port",
                         "sample": f"{sample} clip(s) per step x {args.steps} steps over {procs} worker processes x {threads} threads; cv2/libavcodec decode "
                                   "(PyAV stand-in) + torchvision transforms + oracle torch-fp32 tower, one model call per clip",
                         "worker_seconds": phases},
        "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cores": cores, "host": host_cpu_info(),
    }  # fmt: skip
    print(json.dumps(line))


# ================================================================================================ this repo's arm
def run_b200(args) -> None:
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    clips = make_clips(args.distinct_clips, rank)  # fork pool: before torch / CUDA are touched
    clips_4k = make_clips(4, 0, size=(3840, 2160), bitrate=16.0e6) if (rank == 0 and world == 1 and not args.no_secondary) else None
    clips_720 = make_clips(8, 0, size=(1280, 720), bitrate=2.0e6) if (rank == 0 and world == 1 and not args.no_secondary) else None

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):  # both print the version banner to stdout: keep stdout to the one JSON line
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import uuid

    from cosmos_curate_b200 import sampling
    from cosmos_curate_b200.data_model import Clip, SplitPipeTask, Video
    from cosmos_curate_b200.models import weights as W
    from cosmos_curate_b200.models.clip_aesthetics import CLIPAestheticScorer
    from cosmos_curate_b200.runtime import alloc_nv12_pool, decode_discard, get_context, mp4_index
    from cosmos_curate_b200.stages import NvdecClipAestheticStage

    cfg = W.CLIP_VIT_L14
    cps = args.clips_per_step
    plans = []
    for c in clips:
        idx = mp4_index(c)
        ts = sampling.timestamps_from_index(idx["pts"], idx["timescale"])
        ids, counts = sampling.frame_ids(ts, sampling.FrameExtractionPolicy.sequence, SAMPLE_FPS)
        plans.append(np.repeat(ids, counts).astype(np.int32))
    fpc = len(plans[0])
    frames_per_step = cps * fpc
    clip_arrays = [np.frombuffer(c, dtype=np.uint8) for c in clips]  # host buffers the tasks point at (LazyData holds a view)

    # ---- the product stage (what a cosmos-curate actor would run): set up once, process_data per call
    model = CLIPAestheticScorer(seed=0, max_batch=frames_per_step, config=cfg)

    def make_stage(seek: bool):
        st = NvdecClipAestheticStage(score_threshold=5.0, reduction="min", target_fps=SAMPLE_FPS, write_embedding=True, max_batch=frames_per_step,
                                     num_decoders=args.decoders, stage_batch_size=args.tasks_per_call, seek_keyframes=seek, log_stats=True, model=model)  # fmt: skip
        st.stage_setup()
        return st

    stage = make_stage(seek=False)
    ctx = get_context()
    backend = ctx.decode_backend()  # "libavcodec" (host) where the driver exposes no NVDEC engine: every decode figure below is then host decode
    decoder = "NVDEC" if backend == "nvdec" else "libavcodec host decode (no NVDEC engine exposed)"
    tower = model.tower

    def make_tasks(call: int) -> list:
        """`tasks_per_call` SplitPipeTasks x `cps` clips, walking the distinct clips round-robin; host mp4 bytes in."""
        tasks = []
        for t in range(args.tasks_per_call):
            base = (call * args.tasks_per_call + t) * cps
            cl = [Clip(uuid=uuid.UUID(int=base + j + 1), source_video="v.mp4", span=(0.0, SECONDS), encoded_data=clip_arrays[(base + j) % len(clips)]) for j in range(cps)]
            tasks.append(SplitPipeTask(session_id=f"s{call}-{t}", video=Video(input_video="v.mp4", clips=cl)))
        return tasks

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- resident-input measurement (value): decoded surfaces of one step already in HBM
    pool0 = alloc_nv12_pool(ctx, frames_per_step, FRAME_W, FRAME_H, colour="swscale")  # the conversion the product stage uses
    dp = stage._decode_pool
    futs = [dp.submit(lambda dec, j=j: dec.decode(clips[j % len(clips)], plans[j % len(clips)], pool0, np.arange(j * fpc, (j + 1) * fpc, dtype=np.int32))) for j in range(cps)]
    for f in futs:
        f.result()
    barrier()
    for _ in range(max(args.warmup, 3)):
        tower.embed_pool(pool0)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.profile_begin()
    ev0.record()
    for _ in range(args.steps):
        emb, _, score = tower.embed_pool(pool0)
    ev1.record()
    prof = ctx.profile_end()
    barrier()
    dev_s = max_over_ranks(ev0.elapsed_time(ev1) / 1e3)
    launches = ctx.launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"embedding": emb, "aesthetic_score": score})
    value = world * cps * args.steps / dev_s
    del pool0

    # ---- end-to-end measurement (e2e): the product stage on host tasks
    cpu_t = lambda: sum(os.times()[:2])  # noqa: E731 - user + system CPU seconds of this process (decode threads included)

    def e2e_measure(st, n_calls: int) -> dict:
        st.process_data(make_tasks(0))  # warm-up call: sessions created, pools + pinned buffers allocated
        barrier()
        c0, t0 = cpu_t(), time.perf_counter()
        decoded = scored = 0
        perf_s = 0.0
        for k in range(n_calls):
            tasks = st.process_data(make_tasks(k + 1))
            decoded += st.last_call_stats["frames_decoded"]
            for t in tasks:
                v = t.video
                scored += sum(1 for c in v.clips + v.filtered_clips if c.aesthetic_score is not None and c.aesthetic_score > -1.0 and c.openai_embedding is not None)
            perf_s += tasks[0].stage_perf["NvdecClipAestheticStage"].process_time
        barrier()
        wall_local = time.perf_counter() - t0
        sec = max_over_ranks(wall_local)
        cpu_used = cpu_t() - c0
        n_clips = cps * args.tasks_per_call * n_calls
        assert scored == n_clips, f"{scored} of {n_clips} clips scored"
        h2d = sum(len(clips[(args.tasks_per_call * cps + j) % len(clips)]) for j in range(cps * args.tasks_per_call))
        decoded_all = sum_over_ranks(decoded)
        return {"value": world * n_clips / sec, "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": cps * args.tasks_per_call * fpc * (cfg.proj_dim + 1) * 4,
                "api": "NvdecClipAestheticStage.process_data(list[SplitPipeTask]) on a set-up stage (the call xenna's StageWorker makes)",
                "clips_per_call": cps * args.tasks_per_call, "calls": n_calls, "ms_per_call": 1e3 * sec / n_calls,
                "frames_per_sec": world * n_clips * fpc / sec, "decoded_frames_per_sec": decoded_all / sec,
                "decoded_frames_per_clip": decoded / max(1, n_clips), "decode_backend": backend, "decode_sessions": args.decoders,
                "stage_perf_process_time_s": perf_s, "wall_s_this_rank": wall_local,
                "host_cpu_cores_busy_this_rank": cpu_used / wall_local, "numa_node": st.last_call_stats.get("numa_node"),
                "pinned_cpus": st.last_call_stats.get("pinned_cpus"), "seek_keyframes": bool(st._seek)}  # fmt: skip

    def gather_per_rank(x: float) -> list:
        if world == 1:
            return [x]
        t = torch.zeros(world, dtype=torch.float64, device="cuda")
        t[rank] = x
        dist.all_reduce(t)
        return [float(v) for v in t.tolist()]

    def decode_only(dpool, data_list, seconds: float) -> float:
        """Every session decoding whole clips back to back for `seconds`, surfaces discarded: frames/s of this GPU."""
        deadline = [0.0]

        def loop(dec, k):
            n, i = 0, k
            while time.perf_counter() < deadline[0]:
                n += decode_discard(dec, data_list[i % len(data_list)])
                i += dpool.sessions
            return n

        list(f.result() for f in [dpool.submit(lambda dec, k=k: decode_discard(dec, data_list[k % len(data_list)])) for k in range(dpool.sessions)])  # sessions up
        t0 = time.perf_counter()
        deadline[0] = t0 + seconds
        n = sum(f.result() for f in [dpool.submit(loop, k) for k in range(dpool.sessions)])
        return n / (time.perf_counter() - t0)

    e2e = e2e_sparse = ceiling = exchange = None
    e2e_error = None
    if not args.no_e2e:
        try:
            e2e = e2e_measure(stage, args.e2e_steps)
            e2e["per_rank_decoded_fps"] = gather_per_rank(e2e["decoded_frames_per_clip"] * cps * args.tasks_per_call * args.e2e_steps / e2e["wall_s_this_rank"])
            e2e["note"] = ("every frame up to the last sampled one is decoded (reference semantics, decoder_utils.py:439-455); residual-coded ~4 Mb/s "
                           "synthetic clips; decode of tower batches k+1, k+2 overlaps the tower of batch k INSIDE the stage")
            ceil_fps = decode_only(stage._decode_pool, clips, args.ceiling_seconds)
            sintel = ROOT / "tests" / "golden" / "sintel_clip_10s.mp4"
            real = None
            if sintel.exists():
                sd = sintel.read_bytes()
                fps_real = decode_only(stage._decode_pool, [sd], 3.0)
                real = {"clip": "tests/golden/sintel_clip_10s.mp4 (854x480, High profile, CABAC, B-frames-free real content)", "frames_per_sec_per_gpu": fps_real,
                        "macroblocks_per_sec": fps_real * 54 * 30, "as_1080p_frames_per_sec": fps_real * (54 * 30) / (120 * 68)}  # fmt: skip
            ceiling = {"decoder": decoder, "decode_only_frames_per_sec_per_gpu": ceil_fps, "seconds": args.ceiling_seconds, "sessions": args.decoders,
                       "e2e_fraction_of_decode_ceiling": (e2e["decoded_frames_per_sec"] / world) / ceil_fps if ceil_fps > 0 else None,
                       "real_content": real}  # fmt: skip
            stage.destroy()
            stage2 = make_stage(seek=True)  # opt-in mode of the same stage
            e2e_sparse = e2e_measure(stage2, args.e2e_steps)
            e2e_sparse["note"] = "seek_keyframes=True (CB_DECODE_SEEK_SYNC): only GOPs holding sampled frames are decoded (identical frames); closed GOP = 30, 1 fps sampling"
            if world > 1:
                # the one exchange step of the design (BASELINE.json C3/C4): NCCL all-gather of the clip embeddings, then cosine dedup
                from cosmos_curate_b200.dedup import semdedup_cluster
                from cosmos_curate_b200.sharding import all_gather_embeddings

                tasks = stage2.process_data(make_tasks(99))
                local_emb = torch.from_numpy(np.stack([c.openai_embedding for t in tasks for c in t.video.clips + t.video.filtered_clips])).cuda()
                warm, _ = all_gather_embeddings(local_emb)  # warm-up: communicator creation, first-call allocations of the dedup kernels
                semdedup_cluster(np.arange(warm.shape[0]), warm, torch.zeros(warm.shape[0]), eps=0.01)
                barrier()
                g0, g1, g2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                g0.record()
                allemb, _ = all_gather_embeddings(local_emb)
                g1.record()
                res = semdedup_cluster(np.arange(allemb.shape[0]), allemb, torch.zeros(allemb.shape[0]), eps=0.01)
                g2.record()
                torch.cuda.synchronize()
                exchange = {"collective": "NCCL all_gather (padded) of per-rank [n_i, 768] fp32 clip embeddings", "rows_per_rank": int(local_emb.shape[0]),
                            "rows_total": int(allemb.shape[0]), "allgather_ms": max_over_ranks(g0.elapsed_time(g1)), "semdedup_ms": max_over_ranks(g1.elapsed_time(g2)),
                            "kept": res["kept"], "total": res["total"]}  # fmt: skip
            stage2.destroy()
        except Exception as exc:  # noqa: BLE001 - e.g. libnvcuvid missing on the box: report it, keep the device-resident numbers
            import traceback

            e2e_error = f"{type(exc).__name__}: {exc} | {traceback.format_exc()[-600:]}"
            if world > 1:
                raise
    shot = None
    if rank == 0 and not args.no_shots:
        try:
            shot = shot_detection_measure(ctx, torch)
        except Exception as exc:  # noqa: BLE001
            shot = {"error": f"{type(exc).__name__}: {exc}"}
    clocks = sampler.stop() if rank == 0 else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_src = peaks()
    traffic = ncu_traffic()
    gemm_flops = cfg.gemm_flops_per_image() * frames_per_step * args.steps
    gemm_ms, gemm_n = prof["gemm"]["ms"], max(1, prof["gemm"]["launches"])
    ach_tf = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    peak_tf = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    pre_bytes = (1.5 * min(FRAME_W, FRAME_H) ** 2 + 3 * 224 * 224 * 2) * frames_per_step * args.steps
    ln_bytes = 6.0 * cfg.tokens * cfg.hidden * frames_per_step * (2 * cfg.layers) * args.steps  # fp32 in + fp16 out per LayerNorm
    other = {}
    for name, nbytes, key in (("preprocess", pre_bytes, "preprocess"), ("layernorm", ln_bytes, "layernorm")):
        ms = prof[key]["ms"]
        gbs = nbytes / (ms / 1e3) / 1e9 if ms > 0 else 0.0
        other[name] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                       "traffic": traffic.get({"preprocess": "clip_preprocess", "layernorm": "layernorm_kernel"}[name]),
                       "ms_per_step": ms / args.steps, "launches_per_step": prof[key]["launches"] / args.steps}  # fmt: skip
    other["attention"] = {"ms_per_step": prof["attention"]["ms"] / args.steps, "launches_per_step": prof["attention"]["launches"] / args.steps}
    step_ms = 1e3 * dev_s / args.steps
    line = {
        "metric": "clips_per_sec", "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "frames_per_sec": world * frames_per_step * args.steps / dev_s,
        "config": {"workload": WORKLOAD, "implementation": f"one process per B200: {decoder} + fused preprocess kernel + tcgen05 tower behind NvdecClipAestheticStage",
                   "clips_per_step": cps, "frames_per_clip": fpc, "frames_per_step": frames_per_step, "sample_fps": SAMPLE_FPS, "distinct_clips": args.distinct_clips,
                   "clip_bitrate_bps": float(np.mean([8 * len(c) / SECONDS for c in clips])),
                   "clip_stream": "tools/synth_h264.make_coded_clip: Intra16x16 IDR (DC + sparse AC, chroma DC) + P (P_Skip runs, quarter-pel 16x16 motion, sparse 4x4 residuals), CAVLC, deblocking on, GOP 30",
                   "network": "clip-vit-large-patch14, seeded random weights, fp16 operands / fp32 accumulate+residual", "sharding": f"{world} rank(s), clips sharded per rank, no data-path collective",
                   "l2": "inputs (NV12 pool 0.88 GB + activations > 1 GB) exceed the 126 MB L2", "value_inputs": "decoded NV12 surfaces resident in HBM"},
        "decode_backend": backend, "clocks": clocks, "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_2cta_kernel", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf,
                     "traffic": traffic.get("gemm_tcgen05_2cta"), "traffic_source": traffic.get("_source"),
                     "peak_source": f"{pk_src} bf16_tflops_sustained (kernel timed inside a long step)", "launches_per_step": gemm_n / args.steps,
                     "ms_per_step": gemm_ms / args.steps, "share_of_step": gemm_ms / args.steps / step_ms},
        "roofline_other": other,
        "e2e": e2e, "e2e_keyframe_seek": e2e_sparse, "decode_roofline": ceiling, "host": host_cpu_info(),
    }  # fmt: skip
    if exchange is not None:
        line["exchange"] = exchange
    if shot is not None:
        if "tflops_fp32" in shot and clocks:
            peak = ctx.device_info()["sm_count"] * 128 * 2 * clocks["sm_max_mhz"] * 1e6 / 1e12  # FFMA lanes x 2 flop x clock
            shot["fp32_peak_tflops"] = peak
            shot["frac_of_fp32_peak"] = shot["tflops_fp32"] / peak
        line["shot_detection"] = shot
    if e2e_error:
        line["e2e_error"] = e2e_error
    if world == 1 and not args.no_secondary:
        try:
            line["secondary"] = secondary_configs(ctx, torch, clips, clips_4k, args, clips_720, decoder)
        except Exception as exc:  # noqa: BLE001
            import traceback

            line["secondary"] = {"error": f"{type(exc).__name__}: {exc} | {traceback.format_exc()[-500:]}"}
    if world == 1 and not args.no_gpu_library:
        try:
            line["gpu_library_baseline"] = gpu_library_baseline(clips[:4], torch)
        except Exception as exc:  # noqa: BLE001
            line["gpu_library_baseline"] = {"error": f"{type(exc).__name__}: {exc}"}
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(clips[:4])
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Write each output as out_dir/<name>.npy in float32.  The outputs share their leading (frame) dimension; above
    DUMP_LIMIT_BYTES in all, the same seeded sample of rows is kept from each and its row indices go to sample_rows.npy."""
    arrays = {name: t.detach().float().cpu().numpy() for name, t in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        n = next(iter(arrays.values())).shape[0]
        rows = np.sort(np.random.default_rng(0).choice(n, size=DUMP_LIMIT_BYTES // (total // n + 8), replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["sample_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def secondary_configs(ctx, torch, clips_1080p: list[bytes], clips_4k, args, clips_720=None, decoder: str = "NVDEC") -> dict:
    """Bounded secondary rows (N=1, rank 0): BASELINE.json configs[0] (C1) on both arms, a configs[3]-shaped row (4K + SoViT-400m) and
    the transcode-free clip cutter.  Not the headline; each states its own workload."""
    import uuid

    from cosmos_curate_b200.data_model import Clip, SplitPipeTask, Video
    from cosmos_curate_b200.models import weights as W
    from cosmos_curate_b200.models.clip_aesthetics import CLIPAestheticScorer
    from cosmos_curate_b200.models.siglip import SigLIPImageEmbeddings
    from cosmos_curate_b200.runtime import mp4_index
    from cosmos_curate_b200.stages import ClipStreamCopyStage, NvdecClipAestheticStage
    from cosmos_curate_b200.stages.clip_stream_copy import mp4_cut

    out: dict = {}

    def tasks_of(datas, per_task, seconds):
        arrs = [np.frombuffer(d, dtype=np.uint8) for d in datas]
        return [SplitPipeTask(session_id=f"t{t}", video=Video(input_video="v.mp4", clips=[
            Clip(uuid=uuid.uuid4(), source_video="v.mp4", span=(0.0, seconds), encoded_data=arrs[(t * per_task + j) % len(arrs)]) for j in range(per_task)]))
            for t in range(max(1, len(arrs) // per_task))]  # fmt: skip

    def timed(stage, make, reps):
        stage.process_data(make())  # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = 0
        for _ in range(reps):
            for t in stage.process_data(make()):
                n += len(t.video.clips) + len(t.video.filtered_clips)
        torch.cuda.synchronize()
        return n / (time.perf_counter() - t0), n

    # ---- C1: 32 x 480p 5 s clips, CLIP ViT-B/32 (the configuration the reference itself runs on CPU)
    sintel = ROOT / "tests" / "golden" / "sintel_clip_10s.mp4"
    if sintel.exists():
        src = sintel.read_bytes()
        c1 = bytes(mp4_cut(src, 0, 120))  # first 5 s (24 fps) by stream copy: the fixture is a single GOP
        model = CLIPAestheticScorer(seed=0, max_batch=256, config=W.CLIP_VIT_B32)
        st = NvdecClipAestheticStage(score_threshold=-1e9, reduction="min", write_embedding=True, max_batch=256, num_decoders=args.decoders, seek_keyframes=False, model=model)
        st.stage_setup()
        cps, n = timed(st, lambda: tasks_of([c1] * 32, 32, 5.0), 3)
        st.destroy()
        model.tower.close()
        out["c1"] = {"workload": "32 x (854x480 24 fps 5 s H.264 High/CABAC real content: the reference's test fixture cut to 5 s by stream copy) -> 1 fps -> CLIP ViT-B/32 (seeded) + aesthetic head "
                                 "(BASELINE.json configs[0])", "b200_e2e_clips_per_sec": cps, "clips": n, "api": "NvdecClipAestheticStage.process_data, host mp4 bytes in",
                     "cpu": cpu_c1(c1)}  # fmt: skip

    # ---- C4-shaped: 4K clips, 2 fps sampling, SoViT-400m/14 @384 embedding-only (HEVC streams cannot be produced here: H.264 at 4K instead)
    if clips_4k:
        cfg = W.SIGLIP_SO400M_384
        idx = mp4_index(clips_4k[0])
        sig = SigLIPImageEmbeddings(seed=0, max_batch=84, config=cfg)
        st = NvdecClipAestheticStage(score_threshold=None, target_fps=2.0, write_embedding=True, max_batch=84, num_decoders=args.decoders, seek_keyframes=False, model=sig)
        st.stage_setup()
        cps, n = timed(st, lambda: tasks_of(clips_4k * 3, 12, SECONDS), 2)
        decoded = st.last_call_stats["frames_decoded"]
        # resident-input tower rate + roofline of its GEMMs (the dominant kernel of this configuration too)
        from cosmos_curate_b200.runtime import alloc_nv12_pool

        tower = sig.tower
        pool = alloc_nv12_pool(ctx, 84, idx["width"], idx["height"], colour="swscale")
        pool.buf.random_(16, 236)
        for _ in range(2):
            tower.embed_pool(pool, mean=sig.mean, std=sig.std)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.profile_begin()
        ev0.record()
        reps = 3
        for _ in range(reps):
            tower.embed_pool(pool, mean=sig.mean, std=sig.std)
        ev1.record()
        prof = ctx.profile_end()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / reps
        pk, _ = peaks()
        gemm_tf = cfg.gemm_flops_per_image() * 84 * reps / (prof["gemm"]["ms"] / 1e3) / 1e12
        pre_b = (1.5 * 2160**2 + 3 * 384 * 384 * 2) * 84 * reps
        st.destroy()
        tower.close()
        out["c4_shape"] = {
            "workload": "3840x2160 30 fps 10 s H.264 ~16 Mb/s synthetic clips (HEVC cannot be produced in this image; NVDEC accepts hvc1/hev1) -> 2 fps (21 frames/clip) -> "
                        "SigLIP SoViT-400m/14 @384 embedding, seeded weights (BASELINE.json configs[3] shape, one GPU)",
            "e2e_clips_per_sec": cps, "clips": n, "decoded_frames_per_call": decoded, "resident_frames_per_sec": 84 / ms * 1e3, "resident_ms_per_84_frames": ms,
            "gemm": {"achieved_tflops": gemm_tf, "peak": pk.get("bf16_tflops_sustained", pk["bf16_tflops"]), "frac": gemm_tf / pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
                     "ms": prof["gemm"]["ms"] / reps},
            "attention_ms": prof["attention"]["ms"] / reps, "layernorm_ms": prof["layernorm"]["ms"] / reps,
            "preprocess": {"ms": prof["preprocess"]["ms"] / reps, "algorithmic_gbs": pre_b / (prof["preprocess"]["ms"] / 1e3) / 1e9},
            "gflop_per_image": cfg.flops_per_image() / 1e9}  # fmt: skip

    # ---- C5-shaped: 40 % 720p / 40 % 1080p / 20 % 4K in one stream through the aesthetic stage (per-resolution pool rings and batches)
    if clips_4k and clips_720:
        model = CLIPAestheticScorer(seed=0, max_batch=264, config=W.CLIP_VIT_L14)
        st = NvdecClipAestheticStage(score_threshold=5.0, reduction="min", write_embedding=True, max_batch=264, num_decoders=args.decoders, seek_keyframes=False, model=model)
        st.stage_setup()
        mix = []
        for i in range(120):
            mix.append(clips_720[i % len(clips_720)] if i % 5 in (0, 2) else clips_4k[i % len(clips_4k)] if i % 5 == 4 else clips_1080p[i % len(clips_1080p)])
        ctx.profile_begin()
        cps, n = timed(st, lambda: tasks_of(mix, 24, SECONDS), 1)
        prof = ctx.profile_end()
        px = {"720p": 1280 * 720, "1080p": 1920 * 1080, "2160p": 3840 * 2160}
        mean_px = 0.4 * px["720p"] + 0.4 * px["1080p"] + 0.2 * px["2160p"]
        st.destroy()
        model.tower.close()
        out["c5_mix"] = {
            "workload": "120 clips per call: 40 % 1280x720 (2 Mb/s), 40 % 1920x1080 (4 Mb/s), 20 % 3840x2160 (16 Mb/s) H.264 10 s clips interleaved -> 1 fps -> CLIP ViT-L/14 + aesthetic "
                        "filter (BASELINE.json configs[4] mix on one GPU; the reference's split / caption / writer stages around it are out of scope)",
            "e2e_clips_per_sec": cps, "clips": n, "decoded_megapixels_per_sec": cps * 300 * mean_px / 1e6,
            "kernel_ms_over_warmup_and_timed_call": {k: v["ms"] for k, v in prof.items() if v["launches"] and k != "other"},  # "other" would absorb the idle gaps while the SMs wait for NVDEC
            "note": f"decoder: {decoder}; compare decoded_megapixels_per_sec with the 1080p ceiling (decode_roofline.decode_only_frames_per_sec x 2.07 Mpx); one decode session per stream shape per "
                    "worker thread - a session that is fed another resolution is destroyed and re-created by the driver (tools/mixed_decode_probe.py)"}  # fmt: skip

    # ---- video-tower input tubes (N5, formulation only): 1080p clips -> 2 fps -> 8 kept frames -> cv2-bilinear 224 x 224 + ImageNet normalise
    from cosmos_curate_b200.runtime import alloc_nv12_pool
    from cosmos_curate_b200.stages import InternVideo2FrameCreationStage

    st = InternVideo2FrameCreationStage(target_fps=2.0, source="nvdec", num_decoders=args.decoders, stage_batch_size=4)
    st.stage_setup()
    cps, n = timed(st, lambda: tasks_of(clips_1080p[:48], 12, SECONDS), 1)
    pool = alloc_nv12_pool(ctx, 256, 1920, 1080, "swscale")
    pool.buf.random_(0, 256)
    ctx.video_tube(pool, 224, 224)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(10):
        ctx.video_tube(pool, 224, 224)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / 10
    tube_b = 256 * 224 * 224 * (4 * 3 + 3 * 4)  # 4 taps x (Y + UV pair) read, 3 float32 written, per output pixel
    st.destroy()
    del pool
    out["iv2_tubes"] = {
        "workload": "48 1080p 10 s clips -> 2 fps sampling -> frames[::2][:8] -> cv2.resize(224, 224) + ImageNet normalise -> float32 [1,8,3,224,224] on the host "
                    "(InternVideo2FrameCreationStage, source=nvdec; the tower itself is not part of this path)",
        "e2e_clips_per_sec": cps, "clips": n, "d2h_bytes_per_clip": 8 * 3 * 224 * 224 * 4,
        "kernel": {"ms_per_256_frames": ms, "algorithmic_gbs": tube_b / (ms / 1e3) / 1e9, "bound": "hbm (sparse: 4 source pixels per output; sector-granular reads)"},
        "note": f"decode-bound ({decoder}) like the headline: every frame up to the last kept one is decoded"}  # fmt: skip

    # ---- transcode-free clip cutting (N2): 5 s spans out of the 10 s 1080p sources by stream copy
    stage = ClipStreamCopyStage()
    vids = []
    for i in range(16):
        v = Video(input_video=f"v{i}.mp4", encoded_data=clips_1080p[i % len(clips_1080p)], clips=[Clip(uuid=uuid.uuid4(), source_video=f"v{i}.mp4", span=s) for s in ((0.0, 5.0), (5.0, 10.0))])
        v.metadata.duration = SECONDS
        vids.append(SplitPipeTask(session_id=f"c{i}", video=v))
    t0 = time.perf_counter()
    stage.process_data(vids)
    dt = time.perf_counter() - t0
    nb = sum(c.encoded_data.nbytes for t in vids for c in t.video.clips)
    out["clip_cut"] = {"workload": "32 five-second clips cut from sixteen 1080p 10 s sources by stream copy (ClipStreamCopyStage; the reference re-encodes each with libopenh264)",
                       "clips_per_sec": 32 / dt, "mb_per_sec": nb / dt / 1e6, "host_threads": 1}  # fmt: skip
    return out


def cpu_c1(clip: bytes) -> dict:
    """The reference CPU path on C1 (32 x 480p 5 s, ViT-B/32): all usable cores, and one core for per-core normalisation."""
    import torch

    from oracle import cpu_path, vit

    cores = effective_cores()
    cfg = vit.CLIP_VIT_B32
    w, sd = vit.random_weights(cfg, seed=0), vit.random_aesthetic_mlp(seed=0, in_dim=cfg.proj_dim)
    res = {}
    prev = torch.get_num_threads()
    try:
        for name, threads, n in (("all_cores", cores, 32), ("one_core", 1, 4)):
            path = cpu_path.CpuReferencePath(cfg, w, sd, threads=threads)
            path.run([clip], 1.0, decode_workers=1, decode_threads=min(4, threads))  # warm-up
            r = path.run([clip] * n, 1.0, decode_workers=max(1, threads // 4), decode_threads=min(4, threads))
            res[name] = {"clips_per_sec": r["clips"] / r["seconds"], "threads": threads, "clips": n, "decode_s": r["decode_s"], "model_s": r["model_s"]}
    finally:
        torch.set_num_threads(prev)
    return res


def gpu_library_baseline(clips: list[bytes], torch, n_calls: int = 12) -> dict:
    """The reference's GPU *library* path restated without Ray (SURVEY.md 8d; BASELINE.md 2b): frames decoded on the CPU exactly
    as ClipFrameExtractionStage does, then per clip ONE call of `_CLIPImageEmbeddings.__call__` semantics - uint8 frames H2D,
    torchvision Resize(224, bicubic, antialias) / CenterCrop / ConvertImageDtype / Normalize on the GPU, HF `CLIPModel`
    .get_image_features in fp32, L2 norm (clip.py:48-74), the 5-Linear aesthetic MLP (aesthetics.py:44-53) and `.cpu()`
    (aesthetic_filter_stages.py:181-183).  Library code only (torchvision + transformers + cuBLAS/cuDNN); none of this repo's
    kernels.  Weights are random-initialised ViT-L/14 (no checkpoints offline) - the arithmetic is the same."""
    from torchvision import transforms
    from transformers import CLIPConfig, CLIPModel

    from oracle import cpu_path

    dev = torch.device("cuda", torch.cuda.current_device())
    tf = transforms.Compose([transforms.Resize(224, interpolation=transforms.InterpolationMode.BICUBIC, antialias=True), transforms.CenterCrop(224),
                             transforms.ConvertImageDtype(torch.float32),
                             transforms.Normalize(mean=(0.48145466, 0.4578275, 0.40821073), std=(0.26862954, 0.26130258, 0.27577711))])  # fmt: skip
    hf_cfg = CLIPConfig(vision_config={"hidden_size": 1024, "intermediate_size": 4096, "num_hidden_layers": 24, "num_attention_heads": 16, "patch_size": 14,
                                       "image_size": 224, "projection_dim": 768}, projection_dim=768)  # fmt: skip
    torch.manual_seed(0)
    model = CLIPModel(hf_cfg).to(dev).eval()
    mlp = torch.nn.Sequential(torch.nn.Linear(768, 1024), torch.nn.Dropout(0.2), torch.nn.Linear(1024, 128), torch.nn.Dropout(0.2), torch.nn.Linear(128, 64),
                              torch.nn.Dropout(0.1), torch.nn.Linear(64, 16), torch.nn.Linear(16, 1)).to(dev).eval()  # fmt: skip
    t0 = time.perf_counter()
    decoded = [cpu_path.decode_sampled_frames(c, SAMPLE_FPS, 4)[0] for c in clips]
    decode_s = (time.perf_counter() - t0) / len(clips)

    @torch.no_grad()
    def call(frames: np.ndarray) -> np.ndarray:
        x = torch.from_numpy(frames).permute(0, 3, 1, 2).to(dev)
        feats = model.get_image_features(pixel_values=tf(x))
        feats = feats.pooler_output if hasattr(feats, "pooler_output") else feats  # transformers >= 5 returns an output object
        emb = feats / feats.norm(dim=-1, keepdim=True)
        return mlp(emb).cpu().numpy()

    for k in range(3):
        call(decoded[k % len(decoded)])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    frames = 0
    for k in range(n_calls):
        frames += len(decoded[k % len(decoded)])
        call(decoded[k % len(decoded)])
    torch.cuda.synchronize()
    model_s = (time.perf_counter() - t0) / n_calls
    del model, mlp
    torch.cuda.empty_cache()
    cores = effective_cores()
    return {"kind": "reference GPU library path restated without Ray (torch-CUDA torchvision + HF CLIPModel fp32, one call per clip); NOT the reference's Ray pipeline",
            "gpu_model_clips_per_sec": 1.0 / model_s, "gpu_model_frames_per_sec": frames / n_calls / model_s, "gpu_model_ms_per_clip": 1e3 * model_s,
            "cpu_decode_s_per_clip_4_threads": decode_s,
            "pipeline_clips_per_sec_estimate": min(1.0 / model_s, (cores / 4.0) / decode_s),
            "estimate_note": f"min(GPU model stage, CPU decode stage with {cores} usable cores / 4 threads per decode actor) - the reference runs them as separate actors",
            "sample": f"{n_calls} model calls of 11 frames (1080p); {len(clips)} clips decoded with cv2/libavcodec (PyAV stand-in)"}  # fmt: skip


def shot_flops_per_window(frames: int = 100) -> float:
    """2*M*N*K over the convolutions and Linear layers of the shot network for one window (transnetv2.py:66-100)."""
    total = 0.0
    hw = [(27, 48), (13, 24), (6, 12)]
    for s in range(3):
        f = 16 << s
        m = frames * hw[s][0] * hw[s][1]
        for cin in ((3 if s == 0 else 2 * f), 4 * f):  # first block reads the previous stack (4 * f/2 channels), second block 4f
            total += 2.0 * m * (8 * f) * (9 * cin) + 2.0 * m * (4 * f) * (6 * f)
    return total + 2.0 * frames * (4864 * 1024 + 448 * 128 + 1024)


def shot_detection_measure(ctx, torch, n_frames: int = 9000, reps: int = 3) -> dict:
    """Secondary row (SURVEY.md 8a a10): the fp32 shot-transition network over one 5-minute video of resident 27x48 thumbnails."""
    from cosmos_curate_b200.models.transnetv2 import seeded_state_dict
    from cosmos_curate_b200.runtime import ShotNet

    net = ShotNet(ctx, seeded_state_dict(0), max_windows=16)
    frames = torch.randint(0, 256, (n_frames, 27, 48, 3), dtype=torch.uint8, device=f"cuda:{ctx.device}")
    for _ in range(2):
        net.predict(frames)
    torch.cuda.synchronize()
    l0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        net.predict(frames)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    windows = -(-n_frames // 50)
    net.close()
    return {"workload": f"{n_frames} frames 27x48 RGB (5 min @ 30 fps) resident in HBM, {windows} windows of 100 frames / stride 50, fp32",
            "frames_per_sec": n_frames / ms * 1e3, "ms_per_video": ms, "ms_per_window": ms / windows, "gflop_per_window": shot_flops_per_window() / 1e9,
            "tflops_fp32": windows * shot_flops_per_window() / ms / 1e9, "gpu_launches": (ctx.launch_count() - l0) // reps}  # fmt: skip


# the same workload name on both arms (the driver pairs the lines by metric + config)
WORKLOAD = "1080p30 10 s H.264 clips -> 1 fps frame sampling -> preprocess -> CLIP-ViT-L/14 embed + aesthetic score (BASELINE.json configs[1])"


def ncu_traffic() -> dict:
    """DRAM bytes per launch from the committed `ncu --set full` capture (profiles/rNN_traffic.json, newest round); {} if none."""
    import glob

    files = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r*_traffic.json")))
    if not files:
        return {}
    with open(files[-1]) as f:
        d = json.load(f)
    out = {k: v["traffic_bytes_per_launch"] for k, v in d["kernels"].items()}
    out["_source"] = os.path.join("profiles", os.path.basename(files[-1]))
    return out


def cpu_layout(cores: int) -> tuple[int, int]:
    """(worker processes, torch threads each): the reference scales this path by replicating actors, not by threading one model."""
    if os.environ.get("CB_REF_PROCS") and os.environ.get("CB_REF_THREADS"):  # tuning override
        return int(os.environ["CB_REF_PROCS"]), int(os.environ["CB_REF_THREADS"])
    # measured on the 128-thread (64-core) B200 host: 16 workers x 4 threads = 0.58 clips/s, 8 x 8 = 0.51, 8 x 16 = 0.27-0.32,
    # 16 x 8 = 0.36, 4 x 32 = 0.19 -> one torch thread per PHYSICAL core, four per worker
    if cores >= 32:
        return cores // 8, 4
    return max(1, cores // 4), min(4, cores) if cores >= 4 else 1


def cpu_baseline(clips: list[bytes]) -> dict:
    """Bounded CPU sample of the same workload: the oracle's restatement of the reference path (kind 'port')."""
    from oracle import cpu_path, vit

    cores = effective_cores()
    procs, threads = cpu_layout(cores)
    pool = cpu_path.CpuReferencePool(vit.CLIP_VIT_L14, seed=0, procs=procs, threads=threads)
    try:
        pool.run([clips[i % len(clips)] for i in range(procs)], SAMPLE_FPS)  # warm-up: one clip per worker
        n = 2 * procs
        r = pool.run([clips[i % len(clips)] for i in range(n)], SAMPLE_FPS)
    finally:
        pool.close()
    return {"value": r["clips"] / r["seconds"], "unit": "clips/s", "cores": procs * threads, "kind": "port", "host": host_cpu_info(),
            "sample": f"{n} clips (1080p30 10 s, {r['frames']} sampled frames) over {procs} worker processes x {threads} threads: cv2/libavcodec decode + "
                      "torchvision transforms + oracle torch-fp32 ViT-L/14, one model call per clip",
            "frames_per_sec": r["frames"] / r["seconds"], "worker_seconds": {k: r[k] for k in ("decode_s", "preprocess_s", "model_s")}}  # fmt: skip


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--clips-per-step", type=int, default=24)
    ap.add_argument("--distinct-clips", type=int, default=64)
    ap.add_argument("--tasks-per-call", type=int, default=20, help="SplitPipeTasks (of clips-per-step clips each) per process_data call of the e2e measurement")
    ap.add_argument("--ceiling-seconds", type=float, default=5.0, help="duration of the decode-only ceiling measurement")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C1 / C4-shaped / clip-cut secondary rows")
    ap.add_argument("--no-gpu-library", action="store_true", help="skip the reference GPU library-path baseline")
    ap.add_argument("--decoders", type=int, default=20, help="concurrent NVDEC sessions per GPU (7 engines on B200)")
    ap.add_argument("--e2e-steps", type=int, default=2, help="timed process_data calls of the e2e measurement")
    ap.add_argument("--ref-clips", type=int, default=2, help="clips per step of the reference arm (bounded sample)")
    ap.add_argument("--no-shots", action="store_true", help="skip the shot-detection secondary measurement")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's per-frame embeddings and aesthetic scores (rank 0) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
