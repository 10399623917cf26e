// Host decode of Annex-B access units with libavcodec, for devices whose driver exposes no NVDEC engine to the process
// (cuvidGetDecoderCaps -> CUDA_ERROR_NO_DEVICE, e.g. a container granted the compute capability only).  libavcodec is the
// decoder the reference itself runs (PyAV); the library is dlopen'ed like libnvcuvid, with the handful of entry points and
// the stable leading fields of AVPacket / AVFrame declared by hand.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <functional>
#include <string>

namespace cb {

struct SwPicture {
  const uint8_t* plane[3];  // Y, U, V (8-bit 4:2:0)
  int pitch[3];
  int width, height;        // display size (cropping applied)
  int64_t pts;              // the pts of the packet the picture came from
};

struct SwDecoder;

// "" when libavcodec can be loaded, else why not.  Searched: $CURATE_B200_LIBAVCODEC, a libavcodec already mapped into the
// process (importing cv2 maps opencv-python's copy with its dependencies), the system's libavcodec.
std::string swdec_available();
// codec: cudaVideoCodec numbering (4 = H.264, 8 = HEVC).  low_delay: the stream has no reordering, output every picture as
// soon as it is decoded.
SwDecoder* swdec_create(int codec, bool low_delay, std::string* err);
void swdec_destroy(SwDecoder* s);
// Decodes one access unit (data == nullptr: end of stream, every queued picture is output and the decoder is ready for a new
// stream).  on_picture is called per output picture in display order; returning false stops with `err` left to the caller.
bool swdec_decode(SwDecoder* s, const uint8_t* data, size_t size, int64_t pts, const std::function<bool(const SwPicture&)>& on_picture,
                  std::string* err);

}  // namespace cb
