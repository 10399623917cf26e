// NVDEC decode of sampled frames straight from in-memory MP4 bytes (C ABI: cb_mp4_index, cb_decoder_*).
//
// Replaces, for the clips the pipeline itself produces:
//   * PyAV demux + software decode + swscale  (decoder_utils.py:230-278, 389-461)  - the reference's per-clip path
//   * PyNvDemuxer / PyNvDecoder               (nvcodec_utils.py:224-234, 247-295)  - its only NVDEC path
// Differences by design: no temp file (frame_extraction_stages.py:152-156 writes one), only the SAMPLED
// display-order frames are mapped and copied (as NV12, into a caller-owned surface pool the fused
// preprocess kernel reads), nothing is converted to RGB or copied to the host.
//
// libnvcuvid ships with the driver, not with the toolkit, and the Video Codec SDK headers are not in this
// image: the handful of structs the parser-driven flow needs are declared here by hand (layout of
// nvcuvid.h / cuviddec.h, SDK 12.x) and the library is dlopen'ed at first use.  CUVIDPICPARAMS is passed
// through opaquely from the parser to cuvidDecodePicture.
#include <dlfcn.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <cstdlib>
#include <string>
#include <vector>

#include "common.h"
#include "mp4_demux.h"
#include "swdec.h"

namespace {

// ---- hand-declared cuvid ABI --------------------------------------------------------------------------
typedef void* CUvideodecoder;
typedef void* CUvideoparser;
typedef void* CUvideoctxlock;
typedef long long CUvideotimestamp;

struct CUVIDEOFORMAT {
  int codec;
  struct {
    unsigned numerator, denominator;
  } frame_rate;
  unsigned char progressive_sequence, bit_depth_luma_minus8, bit_depth_chroma_minus8, min_num_decode_surfaces;
  unsigned coded_width, coded_height;
  struct {
    int left, top, right, bottom;
  } display_area;
  int chroma_format;
  unsigned bitrate;
  struct {
    int x, y;
  } display_aspect_ratio;
  struct {
    unsigned char video_format : 3, video_full_range_flag : 1, reserved_zero_bits : 4;
    unsigned char color_primaries, transfer_characteristics, matrix_coefficients;
  } video_signal_description;
  unsigned seqhdr_data_length;
};
static_assert(sizeof(CUVIDEOFORMAT) == 64, "CUVIDEOFORMAT layout");

struct CUVIDPARSERDISPINFO {
  int picture_index, progressive_frame, top_field_first, repeat_first_field;
  CUvideotimestamp timestamp;
};

struct CUVIDSOURCEDATAPACKET {
  unsigned long flags, payload_size;
  const unsigned char* payload;
  CUvideotimestamp timestamp;
};
enum { CUVID_PKT_ENDOFSTREAM = 1, CUVID_PKT_TIMESTAMP = 2, CUVID_PKT_DISCONTINUITY = 4, CUVID_PKT_ENDOFPICTURE = 8 };

typedef int (*PFNVIDSEQUENCECALLBACK)(void*, CUVIDEOFORMAT*);
typedef int (*PFNVIDDECODECALLBACK)(void*, void* /*CUVIDPICPARAMS*/);
typedef int (*PFNVIDDISPLAYCALLBACK)(void*, CUVIDPARSERDISPINFO*);

struct CUVIDPARSERPARAMS {
  int CodecType;
  unsigned ulMaxNumDecodeSurfaces, ulClockRate, ulErrorThreshold, ulMaxDisplayDelay;
  unsigned bAnnexb : 1, uReserved : 31;
  unsigned uReserved1[4];
  void* pUserData;
  PFNVIDSEQUENCECALLBACK pfnSequenceCallback;
  PFNVIDDECODECALLBACK pfnDecodePicture;
  PFNVIDDISPLAYCALLBACK pfnDisplayPicture;
  void* pfnGetOperatingPoint;
  void* pfnGetSEIMsg;
  void* pvReserved2[5];
  void* pExtVideoInfo;
};
static_assert(sizeof(CUVIDPARSERPARAMS) == 136, "CUVIDPARSERPARAMS layout");

struct CUVIDDECODECREATEINFO {
  unsigned long ulWidth, ulHeight, ulNumDecodeSurfaces;
  int CodecType, ChromaFormat;
  unsigned long ulCreationFlags, bitDepthMinus8, ulIntraDecodeOnly, ulMaxWidth, ulMaxHeight, Reserved1;
  struct {
    short left, top, right, bottom;
  } display_area;
  int OutputFormat, DeinterlaceMode;
  unsigned long ulTargetWidth, ulTargetHeight, ulNumOutputSurfaces;
  CUvideoctxlock vidLock;
  struct {
    short left, top, right, bottom;
  } target_rect;
  unsigned long enableHistogram;
  unsigned long Reserved2[4];
};
static_assert(sizeof(CUVIDDECODECREATEINFO) == 176, "CUVIDDECODECREATEINFO layout");

struct CUVIDDECODECAPS {
  int eCodecType, eChromaFormat;
  unsigned nBitDepthMinus8, reserved1[3];
  unsigned char bIsSupported, nNumNVDECs;
  unsigned short nOutputFormatMask;
  unsigned nMaxWidth, nMaxHeight, nMaxMBCount;
  unsigned short nMinWidth, nMinHeight;
  unsigned char bIsHistogramSupported, nCounterBitDepth;
  unsigned short nMaxHistogramBins;
  unsigned reserved3[10];
};

struct CUVIDPROCPARAMS {
  int progressive_frame, second_field, top_field_first, unpaired_field;
  unsigned reserved_flags, reserved_zero;
  unsigned long long raw_input_dptr;
  unsigned raw_input_pitch, raw_input_format;
  unsigned long long raw_output_dptr;
  unsigned raw_output_pitch, Reserved1;
  void* output_stream;
  unsigned Reserved[46];
  unsigned long long* histogram_dptr;
  void* Reserved2[1];
};
static_assert(sizeof(CUVIDPROCPARAMS) == 264, "CUVIDPROCPARAMS layout");

struct CuvidApi {
  void* handle = nullptr;
  int (*CreateVideoParser)(CUvideoparser*, CUVIDPARSERPARAMS*) = nullptr;
  int (*ParseVideoData)(CUvideoparser, CUVIDSOURCEDATAPACKET*) = nullptr;
  int (*DestroyVideoParser)(CUvideoparser) = nullptr;
  int (*CreateDecoder)(CUvideodecoder*, CUVIDDECODECREATEINFO*) = nullptr;
  int (*DestroyDecoder)(CUvideodecoder) = nullptr;
  int (*DecodePicture)(CUvideodecoder, void*) = nullptr;
  int (*MapVideoFrame64)(CUvideodecoder, int, unsigned long long*, unsigned*, CUVIDPROCPARAMS*) = nullptr;
  int (*UnmapVideoFrame64)(CUvideodecoder, unsigned long long) = nullptr;
  int (*CtxLockCreate)(CUvideoctxlock*, void* /*CUcontext*/) = nullptr;
  int (*CtxLockDestroy)(CUvideoctxlock) = nullptr;
  int (*GetDecoderCaps)(CUVIDDECODECAPS*) = nullptr;  // optional: only used to find out whether the device has an engine
  std::string error;
};

CuvidApi* load_cuvid() {
  static CuvidApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[] = {"libnvcuvid.so.1", "/usr/local/nvidia/lib/libnvcuvid.so.1", "/usr/local/nvidia/lib64/libnvcuvid.so.1",
                           "/usr/lib/x86_64-linux-gnu/libnvcuvid.so.1", "libnvcuvid.so"};
    const char* env = getenv("CURATE_B200_NVCUVID");
    if (env) api.handle = dlopen(env, RTLD_NOW);
    for (size_t i = 0; i < sizeof(names) / sizeof(names[0]) && !api.handle; ++i) api.handle = dlopen(names[i], RTLD_NOW);
    if (!api.handle) {
      api.error = "libnvcuvid.so.1 not found (driver video library); set CURATE_B200_NVCUVID to its path";
      return;
    }
#define CB_SYM(field, name)                                                  \
  *(void**)(&api.field) = dlsym(api.handle, name);                           \
  if (!api.field && api.error.empty()) api.error = std::string("libnvcuvid lacks ") + name;
    CB_SYM(CreateVideoParser, "cuvidCreateVideoParser")
    CB_SYM(ParseVideoData, "cuvidParseVideoData")
    CB_SYM(DestroyVideoParser, "cuvidDestroyVideoParser")
    CB_SYM(CreateDecoder, "cuvidCreateDecoder")
    CB_SYM(DestroyDecoder, "cuvidDestroyDecoder")
    CB_SYM(DecodePicture, "cuvidDecodePicture")
    CB_SYM(MapVideoFrame64, "cuvidMapVideoFrame64")
    CB_SYM(UnmapVideoFrame64, "cuvidUnmapVideoFrame64")
    CB_SYM(CtxLockCreate, "cuvidCtxLockCreate")
    CB_SYM(CtxLockDestroy, "cuvidCtxLockDestroy")
#undef CB_SYM
    *(void**)(&api.GetDecoderCaps) = dlsym(api.handle, "cuvidGetDecoderCaps");
  });
  return &api;
}

struct NvdecShared {  // per cb_ctx
  CUvideoctxlock lock = nullptr;
  bool software = false;  // the driver exposes no NVDEC engine to this process: sessions decode with libavcodec (swdec.h)
};

}  // namespace

struct cb_decoder {
  cb_ctx* ctx = nullptr;
  CuvidApi* api = nullptr;
  CUvideodecoder dec = nullptr;
  cudaStream_t stream = nullptr;
  // geometry of the live decoder
  int codec = -1;
  unsigned coded_w = 0, coded_h = 0;
  int disp_w = 0, disp_h = 0, n_surfaces = 0;
  // per-call state (callbacks run on the calling thread inside cuvidParseVideoData)
  const int32_t* ids = nullptr;
  const int32_t* slots = nullptr;
  int n_ids = 0, next_id = 0, display_index = 0, decoded = 0, emitted = 0;
  uint8_t* dst_base = nullptr;
  size_t dst_slot_stride = 0;
  int dst_pitch = 0, dst_luma_rows = 0, dst_w = 0, dst_h = 0;
  bool done = false;
  bool discard = false;            // decode everything, deliver nothing (decode-rate ceiling measurement)
  std::vector<int32_t> rank;       // sample index (decode order) -> display-order frame index
  // thumbnail mode (cb_decoder_decode_thumbnails): every displayed frame -> out_w x out_h RGB, no surface copy
  uint8_t* thumb_out = nullptr;
  int thumb_w = 0, thumb_h = 0, thumb_cap = 0;
  std::string error;
  std::vector<uint8_t> scratch;
  // host decode (NvdecShared::software): libavcodec session, NV12 staging on the host and in device memory
  bool software = false;
  cb::SwDecoder* sw = nullptr;
  int sw_codec = -1;
  bool sw_low_delay = false;
  std::vector<uint8_t> sw_host;
  uint8_t* sw_dev = nullptr;
  size_t sw_dev_bytes = 0;
};

namespace {

int on_sequence(void* user, CUVIDEOFORMAT* f) {
  cb_decoder* d = (cb_decoder*)user;
  const int dw = f->display_area.right - f->display_area.left, dh = f->display_area.bottom - f->display_area.top;
  if (f->chroma_format != 1 || f->bit_depth_luma_minus8 != 0) {
    d->error = "only 8-bit 4:2:0 streams are supported";
    return 0;
  }
  const int want_surfaces = std::max<int>(f->min_num_decode_surfaces, 4) + 2;
  if (d->dec && d->codec == f->codec && d->coded_w == f->coded_width && d->coded_h == f->coded_height && d->disp_w == dw && d->disp_h == dh &&
      d->n_surfaces >= want_surfaces)
    return d->n_surfaces;  // same stream shape as the previous clip: keep the session
  if (d->dec) {
    d->api->DestroyDecoder(d->dec);
    d->dec = nullptr;
  }
  CUVIDDECODECREATEINFO ci;
  memset(&ci, 0, sizeof ci);
  ci.ulWidth = f->coded_width, ci.ulHeight = f->coded_height;
  ci.ulNumDecodeSurfaces = want_surfaces;
  ci.CodecType = f->codec, ci.ChromaFormat = f->chroma_format;
  ci.ulCreationFlags = 4;  // cudaVideoCreate_PreferCUVID: fixed-function NVDEC
  ci.bitDepthMinus8 = 0;
  ci.ulMaxWidth = f->coded_width, ci.ulMaxHeight = f->coded_height;
  ci.display_area.left = (short)f->display_area.left, ci.display_area.top = (short)f->display_area.top;
  ci.display_area.right = (short)f->display_area.right, ci.display_area.bottom = (short)f->display_area.bottom;
  ci.OutputFormat = 0;     // cudaVideoSurfaceFormat_NV12
  ci.DeinterlaceMode = 0;  // weave (progressive content)
  ci.ulTargetWidth = (dw + 1) & ~1, ci.ulTargetHeight = (dh + 1) & ~1;
  ci.ulNumOutputSurfaces = 2;
  // One context lock shared by the sessions of this device: cuvid pushes the lock's context around its own work, so a session
  // keeps working when its callbacks run on a thread whose current device is another GPU (one process, several devices; worker
  // threads start on device 0).  Measured cost: none (16.43 vs 16.46 clips/s end to end with 12 sessions).  CB_NVDEC_CTX_LOCK=0
  // drops it for A/B on single-GPU processes.
  static const bool use_lock = [] {
    const char* e = getenv("CB_NVDEC_CTX_LOCK");
    return !(e && e[0] == '0');
  }();
  ci.vidLock = use_lock ? ((NvdecShared*)d->ctx->nvdec)->lock : nullptr;
  const int rc = d->api->CreateDecoder(&d->dec, &ci);
  if (rc != 0) {
    d->dec = nullptr;
    d->error = "cuvidCreateDecoder failed with CUresult " + std::to_string(rc);
    return 0;
  }
  d->codec = f->codec, d->coded_w = f->coded_width, d->coded_h = f->coded_height, d->disp_w = dw, d->disp_h = dh, d->n_surfaces = want_surfaces;
  return want_surfaces;
}

int on_decode(void* user, void* pic) {
  cb_decoder* d = (cb_decoder*)user;
  if (!d->dec) return 0;
  if (d->done) return 1;  // everything wanted is out: skip the remaining pictures
  const int rc = d->api->DecodePicture(d->dec, pic);
  if (rc != 0) {
    d->error = "cuvidDecodePicture failed with CUresult " + std::to_string(rc);
    return 0;
  }
  d->decoded++;
  return 1;
}

// One displayed picture, NV12 in device memory (luma rows rounded up to even, then the chroma rows) at `pitch`: scaled into
// the thumbnail output, or copied into every surface slot that asked for display index `idx`.
int deliver(cb_decoder* d, int idx, const uint8_t* src, size_t pitch) {
  if (d->thumb_out) {
    const int th = (d->disp_h + 1) & ~1;
    int trc = cb::bilinear_from_surface(d->ctx, src, (int)pitch, th, d->disp_w, d->disp_h, d->thumb_w, d->thumb_h,
                                        d->thumb_out + (size_t)idx * d->thumb_w * d->thumb_h * 3, d->stream);
    cudaError_t te = cudaStreamSynchronize(d->stream);
    if (trc != 0 || te != cudaSuccess) {
      d->error = "thumbnail kernel failed";
      return 0;
    }
    d->emitted++;
    return 1;
  }
  if (((d->disp_w + 1) & ~1) != d->dst_w || ((d->disp_h + 1) & ~1) != d->dst_h) {
    d->error = "clip is " + std::to_string(d->disp_w) + "x" + std::to_string(d->disp_h) + " but the surface pool is " + std::to_string(d->dst_w) +
               "x" + std::to_string(d->dst_h);
    return 0;
  }
  const int th = d->dst_h;  // target height (even)
  cudaError_t e = cudaSuccess;
  while (d->next_id < d->n_ids && d->ids[d->next_id] == idx) {  // a repeated id (supersampling) fills several slots
    uint8_t* dst = d->dst_base + (size_t)d->slots[d->next_id] * d->dst_slot_stride;
    e = cudaMemcpy2DAsync(dst, d->dst_pitch, src, pitch, d->dst_w, th, cudaMemcpyDeviceToDevice, d->stream);
    if (e == cudaSuccess)
      e = cudaMemcpy2DAsync(dst + (size_t)d->dst_luma_rows * d->dst_pitch, d->dst_pitch, src + pitch * th, pitch, d->dst_w, th / 2,
                            cudaMemcpyDeviceToDevice, d->stream);
    if (e != cudaSuccess) break;
    d->next_id++;
    d->emitted++;
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(d->stream);  // the source must outlive the copy
  if (e != cudaSuccess) {
    d->error = std::string("surface copy failed: ") + cudaGetErrorString(e);
    return 0;
  }
  if (d->next_id >= d->n_ids) d->done = true;
  return 1;
}

int on_display(void* user, CUVIDPARSERDISPINFO* info) {
  cb_decoder* d = (cb_decoder*)user;
  if (!info || d->done) return 1;
  d->display_index++;
  if (d->discard) return 1;
  const long long smp = info->timestamp;
  if (smp < 0 || smp >= (long long)d->rank.size()) {
    d->error = "decoder returned an unknown picture timestamp";
    return 0;
  }
  const int idx = d->rank[(size_t)smp];  // display-order index of this picture within the clip
  if (d->thumb_out) {
    if (idx >= d->thumb_cap) {
      d->done = true;
      return 1;
    }
  } else if (d->next_id >= d->n_ids || idx != d->ids[d->next_id]) {
    return 1;
  }
  CUVIDPROCPARAMS pp;
  memset(&pp, 0, sizeof pp);
  pp.progressive_frame = info->progressive_frame;
  pp.top_field_first = info->top_field_first;
  pp.output_stream = d->stream;
  unsigned long long src = 0;
  unsigned pitch = 0;
  int rc = d->api->MapVideoFrame64(d->dec, info->picture_index, &src, &pitch, &pp);
  if (rc != 0) {
    d->error = "cuvidMapVideoFrame64 failed with CUresult " + std::to_string(rc);
    return 0;
  }
  const int ok = deliver(d, idx, (const uint8_t*)src, pitch);
  d->api->UnmapVideoFrame64(d->dec, src);
  return ok;
}

int ensure_shared(cb_ctx* ctx, CuvidApi* api) {
  std::lock_guard<std::mutex> lk(ctx->mu);
  if (ctx->nvdec) return CB_OK;
  CB_CUDA(ctx, cudaSetDevice(ctx->device));
  CB_CUDA(ctx, cudaFree(0));
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuCtxGetCurrent", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn)
    return cb::fail(ctx, CB_ERR_CUDA, "cuCtxGetCurrent not found");
  void* cuctx = nullptr;
  if (((int (*)(void**))fn)(&cuctx) != 0 || !cuctx) return cb::fail(ctx, CB_ERR_CUDA, "no current CUDA context");
  NvdecShared* s = new NvdecShared();
  if (api->GetDecoderCaps) {
    CUVIDDECODECAPS caps;
    memset(&caps, 0, sizeof caps);
    caps.eCodecType = 4, caps.eChromaFormat = 1;  // H.264 4:2:0
    s->software = api->GetDecoderCaps(&caps) == 100;  // CUDA_ERROR_NO_DEVICE: no video engine behind this context
  }
  if (s->software) {
    fprintf(stderr, "cosmos_curate_b200: the driver exposes no NVDEC engine (CUDA_ERROR_NO_DEVICE); decoding on the host with libavcodec\n");
    ctx->nvdec = s;
    return CB_OK;
  }
  const int rc = api->CtxLockCreate(&s->lock, cuctx);
  if (rc != 0) {
    delete s;
    return cb::fail(ctx, CB_ERR_NVDEC, "cuvidCtxLockCreate failed with CUresult %d", rc);
  }
  ctx->nvdec = s;
  return CB_OK;
}

}  // namespace

extern "C" {

void cb_nvdec_release(cb_ctx* ctx) {
  if (!ctx || !ctx->nvdec) return;
  NvdecShared* s = (NvdecShared*)ctx->nvdec;
  CuvidApi* api = load_cuvid();
  if (s->lock && api->CtxLockDestroy) api->CtxLockDestroy(s->lock);
  delete s;
  ctx->nvdec = nullptr;
}

int cb_mp4_index(cb_ctx* ctx, const uint8_t* data, size_t size, cb_mp4_info* info, int64_t* pts_out, uint8_t* sync_out, int cap) {
  // pure host parsing: ctx may be NULL (the message then goes to cb_last_error(NULL))
  if (!data || !info) return cb::fail(ctx, CB_ERR_ARG, "mp4_index: null argument");
  cb::Mp4Track t;
  const std::string err = cb::mp4_parse(data, size, &t);
  if (!err.empty()) return cb::fail(ctx, CB_ERR_DEMUX, "mp4: %s", err.c_str());
  info->codec = t.codec, info->width = t.width, info->height = t.height, info->timescale = t.timescale;
  info->n_samples = (int)t.size.size(), info->has_ctts = t.has_ctts ? 1 : 0, info->duration = t.duration;
  int nsync = 0;
  for (uint8_t s : t.sync) nsync += s;
  info->sample_bytes = 0;
  for (uint32_t b : t.size) info->sample_bytes += b;
  info->n_sync = nsync;
  const int n = std::min<int>(cap, info->n_samples);
  for (int i = 0; i < n; ++i) {
    if (pts_out) pts_out[i] = t.pts[i];
    if (sync_out) sync_out[i] = t.sync[i];
  }
  return CB_OK;
}

int cb_mp4_cut(cb_ctx* ctx, const uint8_t* data, size_t size, int first_sample, int n_samples, uint8_t* out, size_t out_cap, size_t* out_size) {
  // pure host work like cb_mp4_index: ctx may be NULL
  if (!data || !out_size || first_sample < 0 || n_samples <= 0) return cb::fail(ctx, CB_ERR_ARG, "mp4_cut: bad argument");
  cb::Mp4Track t;
  std::string err = cb::mp4_parse(data, size, &t);
  if (!err.empty()) return cb::fail(ctx, CB_ERR_DEMUX, "mp4: %s", err.c_str());
  std::vector<uint8_t> buf;
  err = cb::mp4_cut(data, size, t, (size_t)first_sample, (size_t)n_samples, &buf);
  if (!err.empty()) return cb::fail(ctx, CB_ERR_ARG, "mp4_cut: %s", err.c_str());
  *out_size = buf.size();
  if (!out) return CB_OK;  // size query
  if (out_cap < buf.size()) return cb::fail(ctx, CB_ERR_ARG, "mp4_cut: output buffer of %zu bytes needed, %zu given", buf.size(), out_cap);
  memcpy(out, buf.data(), buf.size());
  return CB_OK;
}

int cb_decode_backend(cb_ctx* ctx, int* backend) {
  if (!ctx) return CB_ERR_ARG;
  if (!backend) return cb::fail(ctx, CB_ERR_ARG, "decode_backend: null argument");
  CuvidApi* api = load_cuvid();
  if (!api->error.empty()) return cb::fail(ctx, CB_ERR_NVDEC, "%s", api->error.c_str());
  const int rc = ensure_shared(ctx, api);
  if (rc) return rc;
  *backend = ((NvdecShared*)ctx->nvdec)->software ? CB_DECODE_BACKEND_LIBAVCODEC : CB_DECODE_BACKEND_NVDEC;
  return CB_OK;
}

int cb_decoder_create(cb_ctx* ctx, cb_decoder** out) {
  if (!ctx) return CB_ERR_ARG;
  if (!out) return cb::fail(ctx, CB_ERR_ARG, "decoder_create: null argument");
  *out = nullptr;
  CuvidApi* api = load_cuvid();
  if (!api->error.empty()) return cb::fail(ctx, CB_ERR_NVDEC, "%s", api->error.c_str());
  int rc = ensure_shared(ctx, api);
  if (rc) return rc;
  CB_CUDA(ctx, cudaSetDevice(ctx->device));  // the session's stream must live on this context's device, whatever thread creates it
  const bool software = ((NvdecShared*)ctx->nvdec)->software;
  if (software) {
    const std::string why = cb::swdec_available();
    if (!why.empty()) return cb::fail(ctx, CB_ERR_NVDEC, "the driver exposes no NVDEC engine (CUDA_ERROR_NO_DEVICE) and host decode is unavailable: %s", why.c_str());
  }
  cb_decoder* d = new cb_decoder();
  d->ctx = ctx, d->api = api;
  d->software = software;
  // highest priority: the post-processing kernel cuvidMapVideoFrame launches and the two surface copies are tiny, and the
  // decode surface is only handed back to NVDEC once they are done - they must not queue behind the tower's persistent CTAs
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (cudaStreamCreateWithPriority(&d->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
    delete d;
    return cb::fail(ctx, CB_ERR_CUDA, "decoder_create: stream creation failed");
  }
  *out = d;
  return CB_OK;
}

void cb_decoder_destroy(cb_decoder* d) {
  if (!d) return;
  cudaSetDevice(d->ctx->device);
  if (d->dec) d->api->DestroyDecoder(d->dec);
  cb::swdec_destroy(d->sw);
  if (d->sw_dev) cudaFree(d->sw_dev);
  if (d->stream) cudaStreamDestroy(d->stream);
  delete d;
}

static int run_parser(cb_decoder* d, const uint8_t* data, size_t size, const cb::Mp4Track& t, cb_decode_stats* stats, int expect, int flags);

int cb_decoder_decode_thumbnails(cb_decoder* d, const uint8_t* data, size_t size, int out_w, int out_h, uint8_t* out, int max_frames,
                                 cb_decode_stats* stats) {
  if (!d) return CB_ERR_ARG;
  cb_ctx* ctx = d->ctx;
  if (stats) memset(stats, 0, sizeof *stats);
  if (!data || !out || out_w <= 0 || out_h <= 0 || max_frames < 0) return cb::fail(ctx, CB_ERR_ARG, "decode_thumbnails: bad argument");
  cb::Mp4Track t;
  const std::string err = cb::mp4_parse(data, size, &t);
  if (!err.empty()) return cb::fail(ctx, CB_ERR_DEMUX, "mp4: %s", err.c_str());
  cudaSetDevice(ctx->device);
  d->ids = nullptr, d->slots = nullptr, d->n_ids = 0, d->next_id = 0, d->display_index = 0, d->decoded = 0, d->emitted = 0;
  d->done = (max_frames == 0);
  d->error.clear();
  d->thumb_out = out, d->thumb_w = out_w, d->thumb_h = out_h, d->thumb_cap = max_frames;
  const int want = std::min<int>(max_frames, (int)t.size.size());
  d->discard = false;
  const int rc = run_parser(d, data, size, t, stats, want, 0);
  d->thumb_out = nullptr;
  return rc;
}

int cb_decoder_decode(cb_decoder* d, const uint8_t* data, size_t size, const int32_t* frame_ids, int n_ids, const cb_surface_pool* dst,
                      const int32_t* dst_slots, cb_decode_stats* stats) {
  return cb_decoder_decode_ex(d, data, size, frame_ids, n_ids, dst, dst_slots, 0, stats);
}

int cb_decoder_decode_ex(cb_decoder* d, const uint8_t* data, size_t size, const int32_t* frame_ids, int n_ids, const cb_surface_pool* dst,
                         const int32_t* dst_slots, int flags, cb_decode_stats* stats) {
  if (!d) return CB_ERR_ARG;
  cb_ctx* ctx = d->ctx;
  if (stats) memset(stats, 0, sizeof *stats);
  if (!data || n_ids < 0 || (n_ids > 0 && (!frame_ids || !dst_slots || !dst || !dst->base))) return cb::fail(ctx, CB_ERR_ARG, "decode: null argument");
  if (dst && n_ids > 0 && dst->format != CB_FMT_NV12 && dst->format != CB_FMT_NV12_SWS) return cb::fail(ctx, CB_ERR_ARG, "decode: destination pool must be NV12");
  for (int i = 1; i < n_ids; ++i)
    if (frame_ids[i] < frame_ids[i - 1]) return cb::fail(ctx, CB_ERR_ARG, "decode: frame ids must be ascending");
  if (n_ids > 0 && frame_ids[0] < 0) return cb::fail(ctx, CB_ERR_ARG, "decode: negative frame id");
  cb::Mp4Track t;
  const std::string err = cb::mp4_parse(data, size, &t);
  if (!err.empty()) return cb::fail(ctx, CB_ERR_DEMUX, "mp4: %s", err.c_str());
  if (n_ids > 0 && frame_ids[n_ids - 1] >= (int)t.size.size())
    return cb::fail(ctx, CB_ERR_ARG, "decode: frame id %d beyond the %zu samples of the clip", frame_ids[n_ids - 1], t.size.size());
  cudaSetDevice(ctx->device);

  d->ids = frame_ids, d->slots = dst_slots, d->n_ids = n_ids, d->next_id = 0, d->display_index = 0, d->decoded = 0, d->emitted = 0;
  d->discard = (flags & CB_DECODE_DISCARD_ALL) != 0;
  d->done = (n_ids == 0) && !d->discard;
  d->error.clear();
  if (dst) {
    d->dst_base = (uint8_t*)dst->base, d->dst_slot_stride = dst->slot_stride, d->dst_pitch = dst->pitch, d->dst_luma_rows = dst->luma_rows;
    d->dst_w = dst->width, d->dst_h = dst->height;
  }

  return run_parser(d, data, size, t, stats, d->discard ? 0 : n_ids, flags);
}

static int run_software(cb_decoder* d, const uint8_t* data, size_t size, const cb::Mp4Track& t, cb_decode_stats* stats, int expect, int flags);

static int run_parser(cb_decoder* d, const uint8_t* data, size_t size, const cb::Mp4Track& t, cb_decode_stats* stats, int expect, int flags) {
  if (d->software) return run_software(d, data, size, t, stats, expect, flags);
  cb_ctx* ctx = d->ctx;
  CUVIDPARSERPARAMS pp;
  memset(&pp, 0, sizeof pp);
  pp.CodecType = t.codec;
  pp.ulMaxNumDecodeSurfaces = 1;  // the sequence callback returns the real DPB size
  pp.ulClockRate = t.timescale;
  pp.ulMaxDisplayDelay = t.has_ctts ? 4 : 0;
  pp.pUserData = d;
  pp.pfnSequenceCallback = on_sequence, pp.pfnDecodePicture = on_decode, pp.pfnDisplayPicture = on_display;
  CUvideoparser parser = nullptr;
  int rc = d->api->CreateVideoParser(&parser, &pp);
  if (rc != 0) return cb::fail(ctx, CB_ERR_NVDEC, "cuvidCreateVideoParser failed with CUresult %d", rc);

  bool failed = false;
  const size_t n = t.size.size();
  // display-order index of every sample: rank of its composition time (stable for equal times)
  {
    std::vector<int32_t> order(n);
    for (size_t i = 0; i < n; ++i) order[i] = (int32_t)i;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return t.pts[a] < t.pts[b]; });
    d->rank.assign(n, 0);
    for (size_t r = 0; r < n; ++r) d->rank[order[r]] = (int32_t)r;
  }
  auto feed = [&](size_t i) {
    d->scratch.clear();
    if (i == 0 || t.sync[i]) d->scratch.insert(d->scratch.end(), t.param_sets_annexb.begin(), t.param_sets_annexb.end());
    if (!cb::mp4_sample_annexb(data, size, t, i, &d->scratch)) {
      d->error = "malformed sample " + std::to_string(i);
      failed = true;
      return;
    }
    CUVIDSOURCEDATAPACKET pkt;
    memset(&pkt, 0, sizeof pkt);
    pkt.flags = CUVID_PKT_TIMESTAMP | CUVID_PKT_ENDOFPICTURE;
    pkt.payload = d->scratch.data(), pkt.payload_size = d->scratch.size(), pkt.timestamp = (CUvideotimestamp)i;  // sample index
    rc = d->api->ParseVideoData(parser, &pkt);
    if (rc != 0 || !d->error.empty()) failed = true;
  };
  auto flush = [&]() {  // end-of-stream: every decoded picture is displayed, the parser restarts at the next IDR
    CUVIDSOURCEDATAPACKET pkt;
    memset(&pkt, 0, sizeof pkt);
    pkt.flags = CUVID_PKT_ENDOFSTREAM;
    rc = d->api->ParseVideoData(parser, &pkt);
    if (rc != 0 || !d->error.empty()) failed = true;
  };
  size_t pos = 0;
  const bool seek = (flags & CB_DECODE_SEEK_SYNC) != 0 && !t.has_ctts && !d->thumb_out && !d->discard && d->n_ids > 0;
  if (seek) {
    // Without reordering (no ctts) display index == sample index.  Jump to the sync sample in front of every wanted frame that
    // lies beyond the current position: the GOPs in between hold no wanted frame and are never decoded.
    for (int k = 0; k < d->n_ids && !failed && !d->done; ++k) {
      const size_t j = (size_t)d->ids[k];
      if (j < pos) continue;  // repeated id, already delivered
      size_t gsync = j;
      while (gsync > pos && !t.sync[gsync]) --gsync;
      if (gsync > pos && t.sync[gsync]) {
        if (pos > 0) flush();
        pos = gsync;
      }
      for (; pos <= j && !failed && !d->done; ++pos) feed(pos);
    }
  }
  for (; pos < n && !d->done && !failed; ++pos) feed(pos);
  if (!failed && !d->done) flush();  // frames still queued for display
  d->api->DestroyVideoParser(parser);
  if (stats) {
    stats->frames_decoded = d->decoded, stats->frames_emitted = d->emitted;
    stats->coded_width = (int)d->coded_w, stats->coded_height = (int)d->coded_h, stats->width = d->disp_w, stats->height = d->disp_h;
  }
  if (failed) return cb::fail(ctx, CB_ERR_NVDEC, "decode: %s", d->error.empty() ? ("cuvidParseVideoData CUresult " + std::to_string(rc)).c_str() : d->error.c_str());
  if (d->emitted != expect) return cb::fail(ctx, CB_ERR_NVDEC, "decode: stream ended after %d displayed frames, %d of %d sampled frames delivered", d->display_index, d->emitted, expect);
  return CB_OK;
}

// The same walk over the samples as run_parser (sync-sample seeks included), decoded by libavcodec on the host.  Every packet
// carries its sample index as pts, and a picture's display index is the rank of that sample's composition time, exactly as
// on_display maps NVDEC's timestamps; each wanted picture is staged as NV12 in device memory and delivered like a mapped
// NVDEC surface.
static int run_software(cb_decoder* d, const uint8_t* data, size_t size, const cb::Mp4Track& t, cb_decode_stats* stats, int expect, int flags) {
  cb_ctx* ctx = d->ctx;
  std::string err;
  if (!d->sw || d->sw_codec != t.codec || d->sw_low_delay != !t.has_ctts) {
    cb::swdec_destroy(d->sw);
    d->sw = cb::swdec_create(t.codec, !t.has_ctts, &err);
    if (!d->sw) return cb::fail(ctx, CB_ERR_NVDEC, "decode: %s", err.c_str());
    d->sw_codec = t.codec, d->sw_low_delay = !t.has_ctts;
  }
  const size_t n = t.size.size();
  {
    std::vector<int32_t> order(n);
    for (size_t i = 0; i < n; ++i) order[i] = (int32_t)i;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return t.pts[a] < t.pts[b]; });
    d->rank.assign(n, 0);
    for (size_t r = 0; r < n; ++r) d->rank[order[r]] = (int32_t)r;
  }
  auto on_picture = [&](const cb::SwPicture& p) -> bool {
    if (d->done) return true;
    d->display_index++;
    d->disp_w = p.width, d->disp_h = p.height, d->coded_w = 0, d->coded_h = 0;  // libavcodec does not report the coded size
    if (d->discard) return true;
    if (p.pts < 0 || p.pts >= (int64_t)n) {
      d->error = "decoder returned an unknown picture timestamp";
      return false;
    }
    const int idx = d->rank[(size_t)p.pts];
    if (d->thumb_out) {
      if (idx >= d->thumb_cap) {
        d->done = true;
        return true;
      }
    } else if (d->next_id >= d->n_ids || idx != d->ids[d->next_id]) {
      return true;
    }
    const int w2 = (p.width + 1) & ~1, h2 = (p.height + 1) & ~1, cw = (p.width + 1) / 2, ch = (p.height + 1) / 2;
    const size_t pitch = (size_t)w2, bytes = pitch * h2 * 3 / 2;
    d->sw_host.assign(bytes, 0);
    for (int y = 0; y < h2; ++y) memcpy(&d->sw_host[y * pitch], p.plane[0] + (size_t)std::min(y, p.height - 1) * p.pitch[0], p.width);
    for (int y = 0; y < ch; ++y) {
      uint8_t* row = &d->sw_host[(h2 + y) * pitch];
      const uint8_t *u = p.plane[1] + (size_t)y * p.pitch[1], *v = p.plane[2] + (size_t)y * p.pitch[2];
      for (int x = 0; x < cw; ++x) row[2 * x] = u[x], row[2 * x + 1] = v[x];
    }
    if (d->sw_dev_bytes < bytes) {
      if (d->sw_dev) cudaFree(d->sw_dev);
      d->sw_dev = nullptr, d->sw_dev_bytes = 0;
      if (cudaMalloc(&d->sw_dev, bytes) != cudaSuccess) {
        d->error = "staging surface allocation failed";
        return false;
      }
      d->sw_dev_bytes = bytes;
    }
    if (cudaMemcpyAsync(d->sw_dev, d->sw_host.data(), bytes, cudaMemcpyHostToDevice, d->stream) != cudaSuccess) {
      d->error = "staging surface upload failed";
      return false;
    }
    return deliver(d, idx, d->sw_dev, pitch) != 0;
  };
  bool failed = false;
  auto decode = [&](const uint8_t* buf, size_t len, int64_t pts) {
    if (!cb::swdec_decode(d->sw, buf, len, pts, on_picture, &err)) failed = true;
  };
  auto feed = [&](size_t i) {
    d->scratch.clear();
    if (i == 0 || t.sync[i]) d->scratch.insert(d->scratch.end(), t.param_sets_annexb.begin(), t.param_sets_annexb.end());
    if (!cb::mp4_sample_annexb(data, size, t, i, &d->scratch)) {
      d->error = "malformed sample " + std::to_string(i);
      failed = true;
      return;
    }
    d->decoded++;
    decode(d->scratch.data(), d->scratch.size(), (int64_t)i);
  };
  size_t pos = 0;
  const bool seek = (flags & CB_DECODE_SEEK_SYNC) != 0 && !t.has_ctts && !d->thumb_out && !d->discard && d->n_ids > 0;
  if (seek) {
    for (int k = 0; k < d->n_ids && !failed && !d->done; ++k) {
      const size_t j = (size_t)d->ids[k];
      if (j < pos) continue;  // repeated id, already delivered
      size_t gsync = j;
      while (gsync > pos && !t.sync[gsync]) --gsync;
      if (gsync > pos && t.sync[gsync]) {
        if (pos > 0) decode(nullptr, 0, 0);
        pos = gsync;
      }
      for (; pos <= j && !failed && !d->done; ++pos) feed(pos);
    }
  }
  for (; pos < n && !d->done && !failed; ++pos) feed(pos);
  if (!failed) decode(nullptr, 0, 0);  // queued pictures out; the session is ready for the next clip
  if (stats) {
    stats->frames_decoded = d->decoded, stats->frames_emitted = d->emitted;
    stats->coded_width = (int)d->coded_w, stats->coded_height = (int)d->coded_h, stats->width = d->disp_w, stats->height = d->disp_h;
  }
  if (failed) {
    cb::swdec_destroy(d->sw);  // state after a failure is unknown: the next call starts a fresh session
    d->sw = nullptr;
    return cb::fail(ctx, CB_ERR_NVDEC, "decode: %s", d->error.empty() ? err.c_str() : d->error.c_str());
  }
  if (d->emitted != expect) return cb::fail(ctx, CB_ERR_NVDEC, "decode: stream ended after %d displayed frames, %d of %d sampled frames delivered", d->display_index, d->emitted, expect);
  return CB_OK;
}

}  // extern "C"
