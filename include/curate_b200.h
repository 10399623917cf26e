/* libcurate_b200 - C ABI of the B200-native decode -> sample -> preprocess -> embed/classify path.
 *
 * The reference (nvidia-cosmos/cosmos-curate) has NO FFI boundary on this path: its stages call
 * Python libraries (PyAV, PyNvVideoCodec, CV-CUDA, torchvision, transformers).  The drop-in boundary
 * is therefore the Python plugin surface (CuratorStage / ModelInterface, mirrored in
 * cosmos_curate_b200/); this header is the thin C ABI those Python stages bind with ctypes.  Every entry
 * point names the reference call it replaces (file:line relative to the reference checkout).
 *
 * Conventions: plain pointers and sizes only (no torch types); every function returns CB_OK (0) or a
 * negative error code and never throws; cb_last_error() returns the message.  Device pointers are
 * caller-owned (torch-allocated is fine); the library owns only its context, cached tables, model
 * weights/workspace and NVDEC sessions.  `stream` is a cudaStream_t passed as void* (NULL = default).
 * Without a CUDA device cb_init fails.  Every kernel runs on the GPU; the one host-side substitute is video decode where the
 * driver exposes no NVDEC engine to the process (cb_decode_backend), and it is reported, never silent.
 */
#ifndef CURATE_B200_H
#define CURATE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CB_OK 0
#define CB_ERR_CUDA (-1)        /* CUDA runtime / driver error */
#define CB_ERR_ARG (-2)         /* bad argument */
#define CB_ERR_UNSUPPORTED (-3) /* valid request this build cannot serve (size, codec, ...) */
#define CB_ERR_NVDEC (-4)       /* libnvcuvid missing or decode failure */
#define CB_ERR_DEMUX (-5)       /* malformed / unsupported container */
#define CB_ERR_STATE (-6)       /* call order (e.g. forward before finalize) */

#define CB_ABI_VERSION 1

typedef struct cb_ctx cb_ctx;
typedef struct cb_vit cb_vit;

/* ---- context ------------------------------------------------------------------------------------ */
int cb_abi_version(void);
/* Creates a context on CUDA device `device` (must be sm_100).  Replaces the implicit torch/CV-CUDA
 * device setup of nvcodec_utils.py:337 (device_id hard-coded to 0 there) and clip.py:39. */
int cb_init(int device, cb_ctx** out);
void cb_destroy(cb_ctx* ctx);
/* Message of the last failing call on `ctx` (or of the last failing cb_init when ctx == NULL). */
const char* cb_last_error(cb_ctx* ctx);
int cb_device_info(cb_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem);
/* PCI bus id of the context's device ("0000:1b:00.0") into buf[len]: the host side uses it to find the GPU's NUMA node
 * (/sys/bus/pci/devices/<id>/numa_node) and pin the NVDEC feeder threads next to it.  The reference leaves placement to
 * Ray/xenna (cosmos-xenna resources.py); one process per GPU needs it spelled out. */
int cb_device_pci_bus_id(cb_ctx* ctx, char* buf, int len);
/* Number of kernels this library has launched on `ctx` since cb_init (bench.py "gpu_launches"). */
unsigned long long cb_launch_count(cb_ctx* ctx);

/* Per-kernel-category device timing: an event is recorded before every launch between begin and end; end
 * returns the summed milliseconds and launch counts per category (bench.py's roofline figures). */
#define CB_PROF_PREPROCESS 0
#define CB_PROF_GEMM 1
#define CB_PROF_LAYERNORM 2
#define CB_PROF_ATTENTION 3
#define CB_PROF_OTHER 4
#define CB_PROF_CONV 5 /* shot-detection network (cb_transnet_*) */
#define CB_PROF_CATEGORIES 6
int cb_profile_begin(cb_ctx* ctx);
int cb_profile_end(cb_ctx* ctx, void* stream, float* ms_by_category, int* launches_by_category, int n_categories);

/* ---- surfaces ----------------------------------------------------------------------------------- */
#define CB_FMT_NV12 0  /* Y plane [luma_rows x pitch] then interleaved UV plane [height/2 x pitch] */
#define CB_FMT_RGB24 1 /* interleaved RGB u8, pitch >= 3*width */
/* NV12 surfaces (same layout as CB_FMT_NV12) whose colour conversion follows libswscale's unscaled yuv420p -> rgb24 converter
 * bit for bit - what the reference's CPU decode hands to CLIP (frame.to_ndarray(format="rgb24"), decoder_utils.py:439-451).
 * CB_FMT_NV12 converts with OpenCV / CV-CUDA semantics (cvcuda.cvtcolor_into, nvcodec_utils.py:35-38,178), the reference's
 * CUDA branch (27x48 shot-detection frames).  Both: ITU-R BT.601 limited range, nearest chroma. */
#define CB_FMT_NV12_SWS 2

/* A pool of equally shaped frames in device memory: frame i starts at base + i*slot_stride.
 * NV12: UV plane of a frame starts `luma_rows * pitch` bytes after its Y plane (NVDEC aligns the coded
 * height, so luma_rows >= height).  base, pitch and slot_stride must be multiples of 16 bytes. */
typedef struct cb_surface_pool {
  const void* base;
  size_t slot_stride;
  int width, height; /* display size in pixels */
  int pitch;         /* bytes per row */
  int luma_rows;     /* NV12 only: rows between the Y plane and the UV plane */
  int format;        /* CB_FMT_* */
} cb_surface_pool;

/* ---- preprocess ---------------------------------------------------------------------------------- */
#define CB_DT_F16 0
#define CB_DT_BF16 1
#define CB_DT_F32 2
#define CB_LAYOUT_NCHW 0  /* out[n][3][res][res]                                   (reference tensor layout) */
#define CB_LAYOUT_PATCH 1 /* out[n][(res/patch)^2][k_pad], k = (c, py, px), zero padded (tower input) */

/* Fused colour-convert + resize + crop + normalise + pack.  Replaces, in one pass over the source
 * frame, cvcuda.cvtcolor_into (nvcodec_utils.py:178) and the reference CLIP transform chain
 * Resize(res, bicubic, antialias) -> CenterCrop(res) -> /255 -> Normalize (clip.py:48-62).
 * slots[n] (host) selects the frames of `pool`; `out` is device memory of the chosen layout/dtype. */
int cb_preprocess_clip(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int res, int layout, int patch,
                       int k_pad, int dtype, const float mean[3], const float std_[3], void* out, void* stream);

/* The same resize/crop with the u8 stage exposed: out u8 [n][3][res][res] (parity tests; this is the
 * tensor torchvision produces before ConvertImageDtype, clip.py:50-55). */
int cb_preprocess_clip_u8(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int res, uint8_t* out,
                          void* stream);

/* Fused NV12->RGB + bilinear resize to out_w x out_h, u8 HWC: out[n][out_h][out_w][3].  Replaces
 * cvcuda.cvtcolor_into + cvcuda.resize_into(Interp.LINEAR) (nvcodec_utils.py:178,189-194), the
 * 27x48 shot-detection frames of VideoFrameExtractionStage (frame_extraction_stages.py:112-116). */
int cb_preprocess_bilinear_u8(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h,
                              uint8_t* out, void* stream);

#define CB_CUBIC_OPENCV 0 /* OpenCV's own fixed-point code: aarch64 wheels, x86 wheels with IPP disabled - bit-exact */
#define CB_CUBIC_IPP 1    /* x86 opencv-python wheels dispatch to Intel IPP: correctly rounded float cubic (<= 1 LSB on ~1e-5 of pixels) */
/* cv2.resize(frame, (out_w, out_h), interpolation=cv2.INTER_CUBIC) of the RGB image of every selected frame (NV12 surfaces
 * are colour-converted per tap), u8 HWC out[n][out_h][out_w][3].  The optional `target_res` square resize of extract_frames
 * (decoder_utils.py:666-670; clip_extraction_target_res = 224 in benchmarks/split_pipeline/invoke.json:38): Keys cubic
 * a = -0.75, 4 taps per axis at any scale (no antialiasing, aspect ratio not preserved), border replicate. */
int cb_resize_cubic_u8(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h, int mode,
                       uint8_t* out, void* stream);

/* The video embedding towers' input formulation, per selected frame: cv2.resize(frame, (out_w, out_h)) [INTER_LINEAR on
 * uint8: OpenCV's fixed-point arithmetic bit for bit, incl. its INTER_AREA reroute of an exact 2x2 decimation] then
 * ((x / 255 - mean) / std) in float32.  Replaces InternVideo2MultiModality._construct_frames / _normalize
 * (cosmos_curate/models/internvideo2_mm.py:385-405), called by InternVideo2FrameCreationStage
 * (pipelines/video/embedding/internvideo2_stages.py:177).  RGB or NV12 pools (NV12 is colour-converted per tap).
 * out_f32 [n][3][out_h][out_w] and/or out_u8 [n][out_h][out_w][3] (the resized frames before normalisation); either may be
 * null, not both. */
int cb_video_tube(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h, const float mean[3],
                  const float std_[3], float* out_f32, uint8_t* out_u8, void* stream);

/* Full-resolution NV12 -> RGB24 (HWC, tightly packed): what decode_video_cpu_frame_ids returns per
 * frame (decoder_utils.py:439-451) / cvcuda.cvtcolor_into (nvcodec_utils.py:178).  Only for callers that
 * must hand RGB frames to an unmodified downstream stage. */
int cb_nv12_to_rgb(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, uint8_t* out, void* stream);

/* ---- image tower (CLIP / SigLIP style ViT) + aesthetic head --------------------------------------- */
#define CB_ACT_QUICK_GELU 0
#define CB_ACT_GELU_TANH 1
#define CB_ARCH_CLIP 0   /* CLS token, pre-LN, post-LN on CLS, bias-free projection (HF CLIPVisionModel) */
#define CB_ARCH_SIGLIP 1 /* no CLS, patch bias, post-LN on all tokens, MAP pooling head (HF SiglipVisionModel) */

typedef struct cb_vit_cfg {
  int image_size, patch, hidden, layers, heads, mlp, proj_dim;
  int act;  /* CB_ACT_* */
  int arch; /* CB_ARCH_* */
  float ln_eps;
} cb_vit_cfg;

/* Replaces CLIPModel.from_pretrained(...).to(device) (clip.py:41) for the image tower. */
int cb_vit_create(cb_ctx* ctx, const cb_vit_cfg* cfg, cb_vit** out);
void cb_vit_destroy(cb_vit* vit);
/* Upload one named tensor (host fp32, row-major, `count` elements).  Names: patch_w[hidden][3*p*p],
 * patch_b, cls, pos[tokens][hidden], pre_ln_w/b, L<i>.{ln1_w,ln1_b,qkv_w[3h][h],qkv_b,out_w,out_b,ln2_w,
 * ln2_b,fc1_w[mlp][h],fc1_b,fc2_w[h][mlp],fc2_b}, post_ln_w/b, proj_w[proj][hidden], map_* (SigLIP). */
int cb_vit_set_tensor(cb_vit* vit, const char* name, const float* data, size_t count);
/* Aesthetic head folded to score = w . embedding + b (the reference MLP, aesthetics.py:44-53, has no
 * non-linearity).  w has proj_dim (or hidden) entries.  Optional. */
int cb_vit_set_aesthetic(cb_vit* vit, const float* w, size_t count, float b);
/* Checks that every tensor arrived and sizes the workspace for batches up to max_batch images. */
int cb_vit_finalize(cb_vit* vit, int max_batch);
/* K padding (in fp16 elements) the tower expects of CB_LAYOUT_PATCH input rows. */
int cb_vit_k_pad(const cb_vit* vit);
/* Forward over n preprocessed images.  patches: device fp16 [n][(image/patch)^2][k_pad] (CB_LAYOUT_PATCH).
 * emb_out: device fp32 [n][proj_dim or hidden], L2-normalised (clip.py:71-74).  feat_out (nullable):
 * the un-normalised features.  score_out (nullable): device fp32 [n] aesthetic scores
 * (clip_aesthetics.py:63-76). */
int cb_vit_forward(cb_vit* vit, const void* patches, int n, float* emb_out, float* feat_out, float* score_out, void* stream);
/* Preprocess + forward in one call: frames of `pool` -> embeddings / scores (the whole
 * CLIPAestheticScorer.__call__, clip_aesthetics.py:63-76, from NV12 or RGB frames). */
int cb_vit_embed_surfaces(cb_vit* vit, const cb_surface_pool* pool, const int32_t* slots, int n, const float mean[3],
                          const float std_[3], float* emb_out, float* feat_out, float* score_out, void* stream);

/* score[i] = w . emb[i] + b over device fp32 embeddings [n][d] (w: device fp32 [d]).  The reference's
 * AestheticScorer.__call__ (aesthetics.py:94-106) on already-computed embeddings. */
int cb_affine_score(cb_ctx* ctx, const float* emb, const float* w, float b, float* out, int n, int d, void* stream);

/* ---- demux + NVDEC ---------------------------------------------------------------------------- */
typedef struct cb_decoder cb_decoder;

typedef struct cb_mp4_info {
  int codec;          /* 4 = H.264, 8 = HEVC (cudaVideoCodec numbering) */
  int width, height;  /* sample-entry (display) size */
  uint32_t timescale; /* mdhd timescale: PTS seconds = pts / timescale */
  int n_samples, n_sync, has_ctts;
  uint64_t duration;     /* mdhd duration in `timescale` ticks */
  uint64_t sample_bytes; /* sum of the video sample sizes (stream bit rate = 8 * sample_bytes / seconds) */
} cb_mp4_info;

typedef struct cb_decode_stats {
  int frames_decoded, frames_emitted;
  int coded_width, coded_height, width, height; /* coded size 0 x 0 when the host decoder ran (it does not report one) */
} cb_decode_stats;

/* Index the first video track of an in-memory MP4: per-sample composition timestamps (decode order, in
 * `timescale` ticks, edit list applied) and sync flags.  Replaces the container open + packet demux of
 * get_video_timestamps (decoder_utils.py:230-278); the caller sorts and converts to float32 seconds exactly
 * as the reference does.  pts_out / sync_out (nullable) receive min(cap, n_samples) entries.  Host-only: ctx may
 * be NULL. */
int cb_mp4_index(cb_ctx* ctx, const uint8_t* data, size_t size, cb_mp4_info* info, int64_t* pts_out, uint8_t* sync_out, int cap);

/* Stream-copy cut (no transcode): samples [first_sample, first_sample + n_samples) of the first video track, decode order,
 * starting on a sync sample, as a standalone MP4 in out[0..*out_size) - sample description copied verbatim, timestamps
 * re-based to 0, coded pictures untouched.  With out == NULL only *out_size is set.  Replaces, for analysis-only runs, the
 * per-clip `ffmpeg -ss/-to ... -c:v libopenh264 -b:v 4M` re-encode of ClipTranscodingStage (clip_extraction_stages.py:318-442;
 * B200 has no NVENC, so that stage is CPU-bound there) with a memcpy of the clip's GOPs.  Host-only: ctx may be NULL. */
int cb_mp4_cut(cb_ctx* ctx, const uint8_t* data, size_t size, int first_sample, int n_samples, uint8_t* out, size_t out_cap,
               size_t* out_size);

#define CB_DECODE_BACKEND_NVDEC 0
#define CB_DECODE_BACKEND_LIBAVCODEC 1
/* Which decoder the sessions of this context use: NVDEC, or - when the driver exposes no NVDEC engine to the process
 * (cuvidGetDecoderCaps -> CUDA_ERROR_NO_DEVICE, e.g. a container granted the compute capability only) - libavcodec on the
 * host, the reference's own decoder, staging each delivered picture as NV12 in device memory.  Callers that report decode
 * (stage stats, benchmarks) must state it.  The host decoder needs libavcodec already mapped into the process (importing
 * cv2 maps opencv-python's copy), $CURATE_B200_LIBAVCODEC, or a system libavcodec. */
int cb_decode_backend(cb_ctx* ctx, int* backend);

/* One decode session (NVDEC parser + decoder + copy stream, or a libavcodec context, see cb_decode_backend); use one per
 * host thread, reuse it across clips. */
int cb_decoder_create(cb_ctx* ctx, cb_decoder** out);
void cb_decoder_destroy(cb_decoder* dec);
/* Decode one clip and deliver ONLY the display-order frames frame_ids[0..n_ids) (ascending; repeats allowed,
 * the counts of sample_closest) as NV12 into slots dst_slots[i] of `dst`.  Decoding stops after the last
 * wanted frame.  Replaces decode_video_cpu_frame_ids (decoder_utils.py:389-461: PyAV decodes every frame,
 * converts the wanted ones to RGB on the host) and NvVideoDecoder.generate_decoded_frames
 * (nvcodec_utils.py:247-295).  Returns only after the copies have completed. */
int cb_decoder_decode(cb_decoder* dec, const uint8_t* data, size_t size, const int32_t* frame_ids, int n_ids,
                      const cb_surface_pool* dst, const int32_t* dst_slots, cb_decode_stats* stats);

#define CB_DECODE_SEEK_SYNC 1   /* skip GOPs without a wanted frame: restart at the sync sample (stss) in front of each one */
#define CB_DECODE_DISCARD_ALL 2 /* decode every picture, deliver none (NVDEC ceiling measurement; frame_ids ignored) */
/* cb_decoder_decode with flags.  CB_DECODE_SEEK_SYNC delivers bit-identical frames while decoding only the closed GOPs
 * that contain sampled frames (streams with composition offsets fall back to sequential decode).  The reference decodes
 * every frame up to the last sampled one (decoder_utils.py:439-455); its sensor library plans sparse seeks the same way
 * (core/sensors/utils/video.py) but the clip path never got them. */
int cb_decoder_decode_ex(cb_decoder* dec, const uint8_t* data, size_t size, const int32_t* frame_ids, int n_ids,
                         const cb_surface_pool* dst, const int32_t* dst_slots, int flags, cb_decode_stats* stats);

/* Decode EVERY frame of the clip (up to max_frames) and write each as an out_w x out_h RGB u8 thumbnail into device
 * memory out[n][out_h][out_w][3]: NV12->RGB + bilinear run directly on the mapped NVDEC surface.  Replaces
 * PyNvcFrameExtractor.__call__ (nvcodec_utils.py:349-381: decode, per-frame reformat, full-resolution colour
 * convert, resize, concat) as used by VideoFrameExtractionStage for the 27x48 shot-detection frames. */
int cb_decoder_decode_thumbnails(cb_decoder* dec, const uint8_t* data, size_t size, int out_w, int out_h, uint8_t* out,
                                 int max_frames, cb_decode_stats* stats);

/* ---- shot-transition network (TransNetV2) -------------------------------------------------------- */
/* Replaces _TransNetV2.forward (cosmos_curate/models/transnetv2.py:103-148, rf=16 rl=3 rs=2 rd=1024 with frame
 * similarity + colour histograms, the only configuration the reference instantiates, :563) and the window
 * stitching of _get_predictions (pipelines/video/clipping/transnetv2_extraction_stages.py:215-264).  fp32 throughout. */
typedef struct cb_transnet cb_transnet;
int cb_transnet_create(cb_ctx* ctx, cb_transnet** out);
void cb_transnet_destroy(cb_transnet* tn);
/* Upload one tensor of the reference state_dict under its own key (host fp32, `count` elements), e.g.
 * "SDDCNN.0.DDCNN.1.Conv3D_4.layers.0.weight", "SDDCNN.2.DDCNN.0.bn.running_var", "fc1.weight",
 * "cls_layer1.bias".  cls_layer2.* and bn.num_batches_tracked are not used by forward() and are not accepted. */
int cb_transnet_set_tensor(cb_transnet* tn, const char* name, const float* data, size_t count);
/* Folds BatchNorm, repacks the convolution weights and sizes the workspace for batches of up to max_windows
 * 100-frame windows (about 150 MB per window). */
int cb_transnet_finalize(cb_transnet* tn, int max_windows);
/* The model call: windows = device uint8 [n_windows][frames_per_window][27][48][3] RGB, 1 <= frames_per_window <= 100;
 * prob_out = device fp32 [n_windows][frames_per_window], sigmoid(one_hot) of transnetv2.py:142-148. */
int cb_transnet_forward(cb_transnet* tn, const uint8_t* windows, int n_windows, int frames_per_window, float* prob_out, void* stream);
/* A whole video: frames = device uint8 [n_frames][27][48][3]; prob_out = device fp32 [n_frames], the concatenation of
 * one_hot[0, 25:75] over the reference's 100-frame / stride-50 windows (first window front-padded with frame 0,
 * the tail windows left short exactly as _get_batches leaves them).  Thresholding (prob > threshold) is the caller's. */
int cb_transnet_predict(cb_transnet* tn, const uint8_t* frames, int n_frames, float* prob_out, void* stream);

/* ---- semantic dedup on the gathered embeddings (fp32) ------------------------------------------------ */
#define CB_ROWDOT_UPPER 1 /* a == b: only candidates i < j count (strict upper triangle) */
#define CB_ROWDOT_CLIP 2  /* clamp scores to [-1, 1] before comparing */
/* For every row j of b[nb][d]: the maximum over rows i of a[na][d] of (a_i . b_j + bias_i) and the FIRST index attaining
 * it; a candidate must be strictly greater than init_val, else out_idx[j] = -1 and out_val[j] = init_val.  All pointers
 * are device fp32 / int32, d a multiple of 16.  Replaces the tiled `E[i0:i1] @ E[j0:j1].T -> clip -> argmax -> where`
 * loop of SemanticDedupActor.dedup (cosmos_curate/pipelines/video/dedup/dedup_actor.py:420-462) with UPPER|CLIP and
 * init_val = -1, and the nearest-centroid assignment of its KMeansMG call (:232-241) with bias_i = -|c_i|^2 / 2. */
int cb_rowdot_argmax(cb_ctx* ctx, const float* a, int na, const float* b, int nb, int d, const float* bias, int flags, float init_val, float* out_val,
                     int* out_idx, void* stream);
/* x[row] /= max(|x[row]|_2, 1e-12) in place (dedup_actor.py:224-225, :407-408); norms_out (nullable) receives |x[row]|. */
int cb_rows_l2_normalize(cb_ctx* ctx, float* x, int rows, int d, float* norms_out, void* stream);
/* sums[c][:] += sum of x[order[t]][:] for t in [seg[c], seg[c+1]): the centroid-update reduction of k-means, rows added
 * in the given order by one thread per (cluster, dimension) - bit-reproducible.  order/seg are device int64. */
int cb_cluster_sums(cb_ctx* ctx, const float* x, const long long* order, const long long* seg, int n_clusters, int d, float* sums, void* stream);

/* ---- building blocks exported for the parity tests ------------------------------------------------ */
#define CB_EPI_NONE 0       /* C = A W^T (+ bias) */
#define CB_EPI_QUICK_GELU 1 /* C = quick_gelu(A W^T + bias) */
#define CB_EPI_GELU_TANH 2  /* C = gelu_tanh(A W^T + bias) */
/* C[M][N] = epilogue(A[M][K] . W[N][K]^T + bias[N]) (+ residual).  A, W fp16 row-major (K contiguous,
 * K % 8 == 0); bias fp32 or NULL.  If out_f32 != NULL: out_f32[M][N] (fp32) = result + (residual ?
 * residual[M][N] : 0) - residual may alias out_f32.  Else out_f16[M][N] = fp16(result).
 * The tcgen05 GEMM under every Linear of the tower (HF CLIPEncoderLayer q/k/v/out/fc1/fc2). */
int cb_gemm_f16(cb_ctx* ctx, const void* A, const void* W, const float* bias, const float* residual, float* out_f32,
                void* out_f16, int M, int N, int K, int epilogue, void* stream);
/* y[rows][d] fp16 = LayerNorm(x[rows][d] fp32) * gamma + beta. */
int cb_layernorm_f16(cb_ctx* ctx, const float* x, const float* gamma, const float* beta, void* y, int rows, int d, float eps,
                     void* stream);
/* Multi-head self-attention over qkv fp16 [n][tokens][3*hidden] (q | k | v, heads contiguous):
 * out fp16 [n][tokens][hidden]; softmax in fp32, scale = head_dim^-1/2. */
int cb_attention_f16(cb_ctx* ctx, const void* qkv, void* out, int n, int tokens, int heads, int head_dim, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CURATE_B200_H */
