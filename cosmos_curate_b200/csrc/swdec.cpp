// libavcodec host decode behind cb_decoder (see swdec.h).
#include "swdec.h"

#include <dlfcn.h>
#include <string.h>

#include <cstdlib>
#include <fstream>
#include <mutex>

namespace cb {
namespace {

// Leading fields of AVPacket / AVFrame: unchanged since FFmpeg 1.x.
struct AVPacketHead {
  void* buf;
  int64_t pts, dts;
  uint8_t* data;
  int size;
};
struct AVFrameHead {
  uint8_t* data[8];
  int linesize[8];
  uint8_t** extended_data;
  int width, height, nb_samples, format;
  int pict_type;
  int sample_aspect_ratio[2];
  int64_t pts;  // offset 136 in FFmpeg 6 (after key_frame) and 7/8 (key_frame removed, 8-byte alignment)
};
static_assert(offsetof(AVFrameHead, pts) == 136, "AVFrame.pts offset");
enum { AV_PIX_FMT_YUV420P = 0, AV_PIX_FMT_YUVJ420P = 12 };
enum { AV_CODEC_ID_H264 = 27, AV_CODEC_ID_HEVC = 173 };
constexpr int AVERROR_EAGAIN = -11;
constexpr int AVERROR_EOF_ = -(int)('E' | ('O' << 8) | ('F' << 16) | ((unsigned)' ' << 24));

struct AvApi {
  void* handle = nullptr;
  const void* (*find_decoder)(int) = nullptr;
  void* (*alloc_context3)(const void*) = nullptr;
  int (*open2)(void*, const void*, void**) = nullptr;
  void (*free_context)(void**) = nullptr;
  int (*send_packet)(void*, const void*) = nullptr;
  int (*receive_frame)(void*, void*) = nullptr;
  void (*flush_buffers)(void*) = nullptr;
  void* (*packet_alloc)() = nullptr;
  void (*packet_free)(void**) = nullptr;
  void* (*frame_alloc)() = nullptr;
  void (*frame_free)(void**) = nullptr;
  void (*frame_unref)(void*) = nullptr;
  int (*opt_set)(void*, const char*, const char*, int) = nullptr;
  std::string error;
};

AvApi* load_av() {
  static AvApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* env = getenv("CURATE_B200_LIBAVCODEC");
    if (env && *env) api.handle = dlopen(env, RTLD_NOW);
    if (!api.handle) {  // already mapped with its dependencies, e.g. by cv2
      std::ifstream maps("/proc/self/maps");
      for (std::string line; !api.handle && std::getline(maps, line);) {
        const size_t p = line.find('/');
        if (p != std::string::npos && line.find("/libavcodec", p) != std::string::npos) api.handle = dlopen(line.c_str() + p, RTLD_NOW | RTLD_NOLOAD);
      }
    }
    const char* names[] = {"libavcodec.so.62", "libavcodec.so.61", "libavcodec.so.60", "libavcodec.so.59", "libavcodec.so"};
    for (size_t i = 0; i < sizeof(names) / sizeof(names[0]) && !api.handle; ++i) api.handle = dlopen(names[i], RTLD_NOW);
    if (!api.handle) {
      api.error = "libavcodec not found; set CURATE_B200_LIBAVCODEC to its path";
      return;
    }
#define CB_AV(field, name)                                   \
  *(void**)(&api.field) = dlsym(api.handle, name);           \
  if (!api.field && api.error.empty()) api.error = std::string("libavcodec lacks ") + name;
    CB_AV(find_decoder, "avcodec_find_decoder")
    CB_AV(alloc_context3, "avcodec_alloc_context3")
    CB_AV(open2, "avcodec_open2")
    CB_AV(free_context, "avcodec_free_context")
    CB_AV(send_packet, "avcodec_send_packet")
    CB_AV(receive_frame, "avcodec_receive_frame")
    CB_AV(flush_buffers, "avcodec_flush_buffers")
    CB_AV(packet_alloc, "av_packet_alloc")
    CB_AV(packet_free, "av_packet_free")
    CB_AV(frame_alloc, "av_frame_alloc")  // libavutil, reached through libavcodec's dependencies
    CB_AV(frame_free, "av_frame_free")
    CB_AV(frame_unref, "av_frame_unref")
    CB_AV(opt_set, "av_opt_set")
#undef CB_AV
  });
  return &api;
}

}  // namespace

struct SwDecoder {
  AvApi* api = nullptr;
  void* ctx = nullptr;
  void* pkt = nullptr;
  void* frame = nullptr;
};

std::string swdec_available() { return load_av()->error; }

void swdec_destroy(SwDecoder* s) {
  if (!s) return;
  if (s->frame) s->api->frame_free(&s->frame);
  if (s->pkt) s->api->packet_free(&s->pkt);
  if (s->ctx) s->api->free_context(&s->ctx);
  delete s;
}

SwDecoder* swdec_create(int codec, bool low_delay, std::string* err) {
  AvApi* api = load_av();
  if (!api->error.empty()) {
    *err = api->error;
    return nullptr;
  }
  const void* c = api->find_decoder(codec == 8 ? AV_CODEC_ID_HEVC : AV_CODEC_ID_H264);
  if (!c || (codec != 4 && codec != 8)) {
    *err = "libavcodec: no decoder for codec " + std::to_string(codec);
    return nullptr;
  }
  SwDecoder* s = new SwDecoder();
  s->api = api;
  s->ctx = api->alloc_context3(c);
  s->pkt = api->packet_alloc();
  s->frame = api->frame_alloc();
  if (!s->ctx || !s->pkt || !s->frame || api->opt_set(s->ctx, "threads", "1", 0) < 0 ||
      (low_delay && api->opt_set(s->ctx, "flags", "+low_delay", 0) < 0) || api->open2(s->ctx, c, nullptr) < 0) {
    *err = "libavcodec: decoder setup failed";
    swdec_destroy(s);
    return nullptr;
  }
  return s;
}

bool swdec_decode(SwDecoder* s, const uint8_t* data, size_t size, int64_t pts, const std::function<bool(const SwPicture&)>& on_picture,
                  std::string* err) {
  AvApi* api = s->api;
  AVPacketHead* p = (AVPacketHead*)s->pkt;
  p->data = (uint8_t*)data, p->size = (int)size, p->pts = p->dts = pts;
  int rc = api->send_packet(s->ctx, data ? s->pkt : nullptr);
  p->data = nullptr, p->size = 0;
  if (rc < 0 && rc != AVERROR_EOF_) {
    *err = "libavcodec: avcodec_send_packet failed (" + std::to_string(rc) + ")";
    return false;
  }
  for (;;) {
    rc = api->receive_frame(s->ctx, s->frame);
    if (rc == AVERROR_EAGAIN) return true;
    if (rc == AVERROR_EOF_) {
      api->flush_buffers(s->ctx);  // drained: ready for the next stream
      return true;
    }
    if (rc < 0) {
      *err = "libavcodec: avcodec_receive_frame failed (" + std::to_string(rc) + ")";
      return false;
    }
    const AVFrameHead* f = (const AVFrameHead*)s->frame;
    if (f->format != AV_PIX_FMT_YUV420P && f->format != AV_PIX_FMT_YUVJ420P) {
      api->frame_unref(s->frame);
      *err = "only 8-bit 4:2:0 streams are supported";
      return false;
    }
    SwPicture pic;
    for (int i = 0; i < 3; ++i) pic.plane[i] = f->data[i], pic.pitch[i] = f->linesize[i];
    pic.width = f->width, pic.height = f->height, pic.pts = f->pts;
    const bool ok = on_picture(pic);
    api->frame_unref(s->frame);
    if (!ok) return false;
  }
}

}  // namespace cb
