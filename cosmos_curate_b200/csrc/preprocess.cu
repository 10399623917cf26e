// Fused frame preprocess kernels (sm_100a).
//
//  clip_preprocess_v2_kernel : NV12 (or RGB24) frame -> YUV->RGB u8 (OpenCV BT.601 or libswscale fixed point) ->
//      antialiased bicubic resize (ATen _upsample_bicubic2d_aa arithmetic, horizontal then vertical,
//      fp32 FMA chains in tap order) -> centre crop -> clamp/round to u8 -> (v/255 - mean)/std LUT ->
//      fp16/bf16/fp32, NCHW or patch-major rows for the tower's patch-embed GEMM.
//      Replaces nvcodec_utils.py:178 + clip.py:48-62 of the reference in ONE pass over the source frame.
//      Source strips are staged into shared memory by TMA (cp.async.bulk.tensor, mbarrier double buffer);
//      a CTA owns one frame x one tile of output columns and walks down the source rows keeping a ring
//      of horizontally filtered rows, so every source byte is fetched once per column tile.
//      By default the horizontal pass runs on the tensor pipe instead (preprocess_tc.cu); this SIMT kernel takes RGB24
//      pools, more than 40 vertical taps and the plans the tensor-pipe kernel rejects, and CB_PRE_KERNEL=2 forces it.
//  bilinear_u8_kernel     : NV12 -> RGB -> 4-tap bilinear (half-pixel centres) -> u8 HWC (27x48 frames).
//  nv12_to_rgb_kernel     : full-resolution NV12 -> RGB24.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "common.h"
#include "ptx.cuh"

namespace cb {

// OpenCV ITUR_BT_601 fixed-point constants (shift 20)
__device__ __forceinline__ void yuv_to_rgb(int y, int u, int v, int& r, int& g, int& b) {
  const int yy = max(y - 16, 0) * 1220542;
  u -= 128;
  v -= 128;
  r = (yy + (1 << 19) + 1673527 * v) >> 20;
  g = (yy + (1 << 19) - 852492 * v - 409993 * u) >> 20;
  b = (yy + (1 << 19) + 2116026 * u) >> 20;
  r = min(max(r, 0), 255);
  g = min(max(g, 0), 255);
  b = min(max(b, 0), 255);
}

// libswscale's unscaled yuv420p -> rgb24 converter (x86 SIMD path, libswscale/x86/yuv_2_rgb.asm; coefficients from
// ff_yuv2rgb_c_init_tables for ITU-R BT.601 limited range, the default PyAV / cv2 leave in place): 16-bit fixed point,
// every product truncated by pmulhw - (8Y - 128) * 9539 >> 16 etc. - nearest chroma.  This is what the reference's CPU decode
// (decode_video_cpu_frame_ids -> frame.to_ndarray(format="rgb24"), decoder_utils.py:439-451) feeds the CLIP transforms.
// Pinned bit-exactly against cv2/libswscale over the whole u8 range (tests/test_oracle_cpu.py).
__device__ __forceinline__ void yuv_to_rgb_sws(int y, int u, int v, int& r, int& g, int& b) {
  const int yy = (((y << 3) - 128) * 9539) >> 16;
  const int uu = (u << 3) - 1024, vv = (v << 3) - 1024;
  r = yy + ((vv * 13075) >> 16);
  g = yy + ((uu * -3209) >> 16) + ((vv * -6660) >> 16);
  b = yy + ((uu * 16525) >> 16);
  r = min(max(r, 0), 255);
  g = min(max(g, 0), 255);
  b = min(max(b, 0), 255);
}
__host__ __device__ __forceinline__ constexpr bool is_nv12(int fmt) { return fmt == CB_FMT_NV12 || fmt == CB_FMT_NV12_SWS; }

constexpr int kThreads = 256;
constexpr int kSR = 32;  // source rows per strip (= lanes of a warp in the horizontal pass)

struct ClipArgs {
  const int* slots;  // device [n]
  int n, src_w, src_h, res;
  int res_out;  // rows/columns actually emitted: res, or (res / patch) * patch for the patch layout (a stride-p conv drops the rest)
  const int *xmin, *xsize, *ymin, *ysize;  // cropped tap tables, [res]
  const float *wx, *wy;                    // [res][tx], [res][ty]
  int tx, ty;
  int y_begin, n_strips;  // first source row fetched (even), number of kSR-row strips
  int tc;                 // output columns per CTA
  int swa;                // strip width in pixels (multiple of 16)
  int ring;               // ring rows (power of two >= kSR + ty)
  const float* lut;       // [3][256]
  int out_mode;           // 0 = u8 NCHW, 1 = typed NCHW, 2 = typed patch rows
  int x_align;            // source window start is aligned down to this many pixels (TMA: 16-byte aligned box start)
  int gu;                 // rows of the per-group dense weight table (>= widest 4-column union window)
  int dtype, patch, k_pad;
  void* out;
};

template <typename T>
__device__ __forceinline__ T cvt_out(float v);
template <>
__device__ __forceinline__ __half cvt_out<__half>(float v) {
  return __float2half_rn(v);
}
template <>
__device__ __forceinline__ __nv_bfloat16 cvt_out<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}
template <>
__device__ __forceinline__ float cvt_out<float>(float v) {
  return v;
}

__device__ __forceinline__ void store_typed(void* out, size_t idx, float v, int dtype) {
  if (dtype == CB_DT_F16) ((__half*)out)[idx] = __float2half_rn(v);
  else if (dtype == CB_DT_BF16) ((__nv_bfloat16*)out)[idx] = __float2bfloat16_rn(v);
  else ((float*)out)[idx] = v;
}

// ------------------------------------------------------------------------------------------------
// Tiled so that the horizontal pass is not shared-memory bound:
//   * output columns are processed in groups of 4 adjacent columns; their tap windows overlap by ~75 %, so one
//     lane (= one source row) walks the UNION window once, loading each pixel once (3 x LDS.32) and applying it to
//     the 4 columns with a dense, zero-padded weight row fetched as one broadcast LDS.128: 12 FMAs per 4 loads, where
//     a lane walking one column's own window does 1 FMA per 2 loads.  fma(x, 0, acc) == acc, so the result is
//     bit-identical to the tap-order chain.
//   * colour conversion clamps with add-min-relu (DPX) instead of separate add / shift / clamp chains;
//   * all output rows that became ready in a strip are emitted in one parallel sweep.
template <int FMT>
__global__ void __launch_bounds__(kThreads, 2) clip_preprocess_v2_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                          const __grid_constant__ CUtensorMap map_b, const ClipArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int frame = blockIdx.y;
  const int c0 = blockIdx.x * a.tc;
  const int ncol = min(a.tc, a.res_out - c0);
  const int slot = a.slots[frame];
  const int ngroups = (ncol + 3) >> 2;

  const int raw_stage = is_nv12(FMT) ? (a.swa * kSR + a.swa * (kSR / 2)) : (3 * a.swa * kSR);
  const int swp = a.swa + 1;
  const int tcp = a.tc | 1;
  uint8_t* raw = smem;
  float* rgbf = (float*)(smem + 2 * raw_stage);
  float* ringb = rgbf + 3 * kSR * swp;
  float4* wg = (float4*)(((uintptr_t)(ringb + 3 * a.ring * tcp) + 15) & ~(uintptr_t)15);  // [groups][gu] x 4 columns
  int* gbase = (int*)(wg + ((a.tc + 3) >> 2) * a.gu);                                      // [groups] first source column, [groups] length
  uint16_t* obuf = (uint16_t*)(((uintptr_t)(gbase + 2 * ((a.tc + 3) >> 2)) + 15) & ~(uintptr_t)15);
  const int npx = (a.out_mode == 2) ? a.tc / a.patch : 0;
  uint64_t* bars = (uint64_t*)(((uintptr_t)(obuf + npx * a.k_pad) + 7) & ~(uintptr_t)7);

  const int x_lo = a.xmin[c0] & ~(a.x_align - 1);

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_barrier_init();
  }
  // dense weight table of this column tile
  for (int i = tid; i < ngroups * a.gu; i += kThreads) wg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (a.out_mode == 2)
    for (int i = tid; i < npx * a.k_pad; i += kThreads) obuf[i] = 0;
  __syncthreads();
  if (tid < ngroups) {
    const int cfirst = c0 + 4 * tid, base = a.xmin[cfirst];
    int len = 0;
    for (int k = 0; k < 4 && 4 * tid + k < ncol; ++k) len = max(len, a.xmin[cfirst + k] + a.xsize[cfirst + k] - base);
    gbase[tid] = base, gbase[ngroups + tid] = len;
  }
  for (int i = tid; i < ncol * a.tx; i += kThreads) {
    const int c = i / a.tx, j = i - c * a.tx;
    if (j < a.xsize[c0 + c]) {
      const int g = c >> 2, k = c & 3;
      const int d = a.xmin[c0 + c] - a.xmin[c0 + 4 * g];
      ((float*)&wg[g * a.gu + d + j])[k] = a.wx[(size_t)(c0 + c) * a.tx + j];
    }
  }
  __syncthreads();

  // NOTE: x_lo is a multiple of 16 pixels: a TMA box whose first byte is not 16-byte aligned in global memory
  // faults with "illegal instruction" (measured on B200; u8 elements make this easy to hit).
#define CB_ISSUE_STRIP(S_)                                                                                        \
  do {                                                                                                            \
    const int s_ = (S_);                                                                                          \
    uint8_t* dst_ = raw + (s_ & 1) * raw_stage;                                                                   \
    uint64_t* bar_ = &bars[s_ & 1];                                                                               \
    const int ys_ = a.y_begin + s_ * kSR;                                                                         \
    mbar_expect_tx(bar_, raw_stage);                                                                              \
    if (is_nv12(FMT)) {                                                                                     \
      tma_load_3d(dst_, &map_a, bar_, x_lo, ys_, slot);                                                           \
      tma_load_3d(dst_ + a.swa * kSR, &map_b, bar_, x_lo, ys_ >> 1, slot);                                        \
    } else {                                                                                                      \
      tma_load_3d(dst_, &map_a, bar_, x_lo * 3, ys_, slot);                                                       \
      tma_load_3d(dst_ + a.swa * kSR, &map_a, bar_, x_lo * 3 + a.swa, ys_, slot);                                 \
      tma_load_3d(dst_ + 2 * a.swa * kSR, &map_a, bar_, x_lo * 3 + 2 * a.swa, ys_, slot);                         \
    }                                                                                                             \
  } while (0)
  if (tid == 0) {
    CB_ISSUE_STRIP(0);
    if (a.n_strips > 1) CB_ISSUE_STRIP(1);
  }

  int next_out = 0;
  for (int s = 0; s < a.n_strips; ++s) {
    const int y0 = a.y_begin + s * kSR;
    const uint8_t* rs = raw + (s & 1) * raw_stage;
    mbar_wait(&bars[s & 1], (s >> 1) & 1);

    // ---- phase 1: colour conversion; one thread owns a 2-row x 4-pixel block (two chroma samples, three 32-bit loads)
    if (is_nv12(FMT)) {
      const int q4 = a.swa >> 2;
      const uint8_t* ry = rs;
      const uint8_t* ruv = rs + a.swa * kSR;
      constexpr int kMax = (256 << 20) - 1;
      for (int i = tid; i < (kSR / 2) * q4; i += kThreads) {
        const int rp = i / q4, x = (i - rp * q4) * 4, r = rp * 2;
        const uint32_t ya = *(const uint32_t*)(ry + r * a.swa + x), yb = *(const uint32_t*)(ry + (r + 1) * a.swa + x);
        const uint32_t uv4 = *(const uint32_t*)(ruv + rp * a.swa + x);
        float* p = rgbf + r * swp + x;
#pragma unroll
        for (int h = 0; h < 2; ++h) {  // the two chroma samples of the block
          if (FMT == CB_FMT_NV12_SWS) {  // swscale arithmetic (see yuv_to_rgb_sws): truncating 16-bit products, clamp 0..255
            const int uu = ((int)((uv4 >> (16 * h)) & 0xff) << 3) - 1024, vv = ((int)((uv4 >> (16 * h + 8)) & 0xff) << 3) - 1024;
            const int ruv_ = (vv * 13075) >> 16, guv_ = ((uu * -3209) >> 16) + ((vv * -6660) >> 16), buv_ = (uu * 16525) >> 16;
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
              const uint32_t yw = rr ? yb : ya;
#pragma unroll
              for (int k = 0; k < 2; ++k) {
                const int yv = ((((int)((yw >> (16 * h + 8 * k)) & 0xff) << 3) - 128) * 9539) >> 16;
                float* q = p + rr * swp + 2 * h + k;
                q[0] = (float)__viaddmin_s32_relu(yv, ruv_, 255);
                q[kSR * swp] = (float)__viaddmin_s32_relu(yv, guv_, 255);
                q[2 * kSR * swp] = (float)__viaddmin_s32_relu(yv, buv_, 255);
              }
            }
            continue;
          }
          const int u = (int)((uv4 >> (16 * h)) & 0xff) - 128, v = (int)((uv4 >> (16 * h + 8)) & 0xff) - 128;
          const int ruv_ = 1673527 * v, guv_ = -852492 * v - 409993 * u, buv_ = 2116026 * u;
#pragma unroll
          for (int rr = 0; rr < 2; ++rr) {
            const uint32_t yw = rr ? yb : ya;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const int yv = max((int)((yw >> (16 * h + 8 * k)) & 0xff) - 16, 0) * 1220542 + (1 << 19);
              float* q = p + rr * swp + 2 * h + k;
              q[0] = (float)(__viaddmin_s32_relu(yv, ruv_, kMax) >> 20);
              q[kSR * swp] = (float)(__viaddmin_s32_relu(yv, guv_, kMax) >> 20);
              q[2 * kSR * swp] = (float)(__viaddmin_s32_relu(yv, buv_, kMax) >> 20);
            }
          }
        }
      }
    } else {
      for (int i = tid; i < kSR * a.swa; i += kThreads) {
        const int r = i / a.swa, x = i - r * a.swa;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          const int b = 3 * x + ch;
          const int blk = b / a.swa, within = b - blk * a.swa;
          rgbf[(ch * kSR + r) * swp + x] = (float)rs[(blk * kSR + r) * a.swa + within];
        }
      }
    }
    __syncthreads();
    if (tid == 0 && s + 2 < a.n_strips) {
      fence_proxy_async();
      CB_ISSUE_STRIP(s + 2);
    }

    // ---- phase 2: horizontal filter, 4 columns x 3 channels per lane (lane = source row)
    for (int g = warp; g < ngroups; g += kThreads / 32) {
      const int len = gbase[ngroups + g];
      const float* px = rgbf + lane * swp + (gbase[g] - x_lo);
      const float4* w = wg + g * a.gu;
      float acc[3][4];
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) acc[ch][0] = acc[ch][1] = acc[ch][2] = acc[ch][3] = 0.f;
#pragma unroll 4
      for (int p = 0; p < len; ++p) {
        const float4 wv = w[p];
        const float r = px[p], gg = px[kSR * swp + p], b = px[2 * kSR * swp + p];
        acc[0][0] = fmaf(r, wv.x, acc[0][0]), acc[0][1] = fmaf(r, wv.y, acc[0][1]), acc[0][2] = fmaf(r, wv.z, acc[0][2]), acc[0][3] = fmaf(r, wv.w, acc[0][3]);
        acc[1][0] = fmaf(gg, wv.x, acc[1][0]), acc[1][1] = fmaf(gg, wv.y, acc[1][1]), acc[1][2] = fmaf(gg, wv.z, acc[1][2]), acc[1][3] = fmaf(gg, wv.w, acc[1][3]);
        acc[2][0] = fmaf(b, wv.x, acc[2][0]), acc[2][1] = fmaf(b, wv.y, acc[2][1]), acc[2][2] = fmaf(b, wv.z, acc[2][2]), acc[2][3] = fmaf(b, wv.w, acc[2][3]);
      }
      const int slot_row = (y0 + lane) & (a.ring - 1);
#pragma unroll
      for (int ch = 0; ch < 3; ++ch)
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (4 * g + k < ncol) ringb[(ch * a.ring + slot_row) * tcp + 4 * g + k] = acc[ch][k];
    }
    __syncthreads();

    // ---- phase 3: emit all output rows whose vertical window is complete, one patch row at a time
    int last = next_out;
    const bool final_strip = (s == a.n_strips - 1);
    while (last < a.res_out && (final_strip || a.ymin[last] + a.ysize[last] <= y0 + kSR)) ++last;
    int seg = next_out;
    while (seg < last) {
      const int seg_end = (a.out_mode == 2) ? min(last, (seg / a.patch + 1) * a.patch) : last;
      for (int yo = seg + warp; yo < seg_end; yo += kThreads / 32) {  // one warp per output row, lane = column
        const int ym = a.ymin[yo], ys = a.ysize[yo];
        const float* wrow = a.wy + (size_t)yo * a.ty;
        const float w_lo = lane < ys ? __ldg(wrow + lane) : 0.f, w_hi = lane + 32 < ys ? __ldg(wrow + lane + 32) : 0.f;
        const int c = min(lane, ncol - 1);
        const float* rb = ringb + c;
        const int chs = a.ring * tcp;
        float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f;
        for (int k = 0; k < ys; ++k) {
          const float w = __shfl_sync(0xffffffffu, k < 32 ? w_lo : w_hi, k & 31);
          const float* rr = rb + ((ym + k) & (a.ring - 1)) * tcp;
          acc0 = fmaf(rr[0], w, acc0), acc1 = fmaf(rr[chs], w, acc1), acc2 = fmaf(rr[2 * chs], w, acc2);
        }
        if (lane < ncol) {
          const int x = c0 + c;
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            float acc = ch == 0 ? acc0 : (ch == 1 ? acc1 : acc2);
            acc = fminf(fmaxf(acc, 0.f), 255.f);
            const int v = __float2int_rn(acc);
            if (a.out_mode == 0) {
              ((uint8_t*)a.out)[(((size_t)frame * 3 + ch) * a.res + yo) * a.res + x] = (uint8_t)v;
            } else {
              const float f = a.lut[ch * 256 + v];
              if (a.out_mode == 1) {
                store_typed(a.out, (((size_t)frame * 3 + ch) * a.res + yo) * a.res + x, f, a.dtype);
              } else {
                const int ip = c / a.patch, px_ = c - ip * a.patch, py = yo % a.patch;
                const uint16_t bits = (a.dtype == CB_DT_F16) ? __half_as_ushort(__float2half_rn(f))
                                                             : __bfloat16_as_ushort(__float2bfloat16_rn(f));
                obuf[ip * a.k_pad + (ch * a.patch + py) * a.patch + px_] = bits;
              }
            }
          }
        }
      }
      if (a.out_mode == 2 && (seg_end % a.patch) == 0) {  // a row of patches is complete: 128-bit stores
        __syncthreads();
        const int gsz = a.res / a.patch, prow = (seg_end - 1) / a.patch, vec = a.k_pad >> 3;
        const int np = ncol / a.patch;
        for (int i = tid; i < np * vec; i += kThreads) {
          const int ip = i / vec, q = i - ip * vec;
          uint4* dst = (uint4*)((uint16_t*)a.out + ((size_t)frame * gsz * gsz + (size_t)prow * gsz + (c0 / a.patch + ip)) * a.k_pad);
          dst[q] = ((const uint4*)(obuf + ip * a.k_pad))[q];
        }
        __syncthreads();
      }
      seg = seg_end;
    }
    next_out = last;
  }
}

// ------------------------------------------------------------------------------------------------
struct SimpleArgs {
  const uint8_t* base;
  size_t slot_stride;
  const int* slots;
  int n, w, h, pitch, luma_rows, out_w, out_h, format;
  uint8_t* out;
};

__device__ __forceinline__ void fetch_rgb_nv12(const uint8_t* f, int pitch, int luma_rows, int x, int y, int& r, int& g, int& b, int format = CB_FMT_NV12) {
  const int Y = f[(size_t)y * pitch + x];
  const uint8_t* uv = f + (size_t)luma_rows * pitch + (size_t)(y >> 1) * pitch + (x & ~1);
  if (format == CB_FMT_NV12_SWS) yuv_to_rgb_sws(Y, uv[0], uv[1], r, g, b);
  else yuv_to_rgb(Y, uv[0], uv[1], r, g, b);
}

// cvcuda.resize_into(LINEAR) semantics: half-pixel centres, clamp-to-edge taps, fp32, round-to-nearest-even.
__global__ void bilinear_u8_kernel(const SimpleArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per = a.out_w * a.out_h;
  if (i >= a.n * per) return;
  const int f = i / per, p = i - f * per, yo = p / a.out_w, xo = p - yo * a.out_w;
  const uint8_t* fr = a.base + (size_t)(a.slots ? a.slots[f] : f) * a.slot_stride;
  const float sx = (float)a.w / (float)a.out_w, sy = (float)a.h / (float)a.out_h;
  const float fx = (xo + 0.5f) * sx - 0.5f, fy = (yo + 0.5f) * sy - 0.5f;
  const int x0 = (int)floorf(fx), y0 = (int)floorf(fy);
  const float wx = fx - (float)x0, wy = fy - (float)y0;
  const int xa = min(max(x0, 0), a.w - 1), xb = min(max(x0 + 1, 0), a.w - 1);
  const int ya = min(max(y0, 0), a.h - 1), yb = min(max(y0 + 1, 0), a.h - 1);
  int p00[3], p01[3], p10[3], p11[3];
  fetch_rgb_nv12(fr, a.pitch, a.luma_rows, xa, ya, p00[0], p00[1], p00[2], a.format);
  fetch_rgb_nv12(fr, a.pitch, a.luma_rows, xb, ya, p01[0], p01[1], p01[2], a.format);
  fetch_rgb_nv12(fr, a.pitch, a.luma_rows, xa, yb, p10[0], p10[1], p10[2], a.format);
  fetch_rgb_nv12(fr, a.pitch, a.luma_rows, xb, yb, p11[0], p11[1], p11[2], a.format);
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const float top = __fadd_rn(__fmul_rn((float)p00[ch], 1.f - wx), __fmul_rn((float)p01[ch], wx));
    const float bot = __fadd_rn(__fmul_rn((float)p10[ch], 1.f - wx), __fmul_rn((float)p11[ch], wx));
    float v = __fadd_rn(__fmul_rn(top, 1.f - wy), __fmul_rn(bot, wy));
    v = fminf(fmaxf(v, 0.f), 255.f);
    a.out[(size_t)i * 3 + ch] = (uint8_t)__float2int_rn(v);
  }
}

__global__ void nv12_to_rgb_kernel(const SimpleArgs a) {
  // one thread per horizontal pixel pair; out tightly packed [n][h][w][3]
  const int pairs_w = (a.w + 1) >> 1;
  const size_t per = (size_t)pairs_w * a.h;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per * a.n) return;
  const int f = (int)(i / per);
  const size_t p = i - (size_t)f * per;
  const int y = (int)(p / pairs_w), x = (int)(p - (size_t)y * pairs_w) * 2;
  const uint8_t* fr = a.base + (size_t)a.slots[f] * a.slot_stride;
  const uint8_t* uv = fr + (size_t)a.luma_rows * a.pitch + (size_t)(y >> 1) * a.pitch + x;
  const int U = uv[0], V = uv[1];
  uint8_t* o = a.out + (((size_t)f * a.h + y) * a.w + x) * 3;
  int r, g, b;
  const bool sws = a.format == CB_FMT_NV12_SWS;
  if (sws) yuv_to_rgb_sws(fr[(size_t)y * a.pitch + x], U, V, r, g, b);
  else yuv_to_rgb(fr[(size_t)y * a.pitch + x], U, V, r, g, b);
  o[0] = r, o[1] = g, o[2] = b;
  if (x + 1 < a.w) {
    if (sws) yuv_to_rgb_sws(fr[(size_t)y * a.pitch + x + 1], U, V, r, g, b);
    else yuv_to_rgb(fr[(size_t)y * a.pitch + x + 1], U, V, r, g, b);
    o[3] = r, o[4] = g, o[5] = b;
  }
}


// ------------------------------------------------------------------------------------------------
// cv2.resize(frame, (out_w, out_h), INTER_CUBIC) on the RGB image of a surface: the optional `target_res` resize of
// extract_frames (decoder_utils.py:666-670).  Keys cubic a = -0.75, 4 taps per axis whatever the scale (no antialiasing),
// border replicate.  Two arithmetic variants, because opencv-python-headless (the reference's pin) ships two:
//   CB_CUBIC_OPENCV : OpenCV's own code (aarch64 wheels; x86 wheels with IPP off) - int16 weights at 2^11, exact int32
//                     horizontal sums, vertical S0*b0 + (S1*b1 + (S2*b2 + S3*b3)) in fp32 without contraction, round half
//                     even (vector body) or (sum + 2^21) >> 22 (scalar row tail).  Bit-exact.
//   CB_CUBIC_IPP    : x86 wheels dispatch to Intel IPP, whose result is the correctly rounded real-valued cubic up to fp32
//                     noise (measured: differs from exact arithmetic on < 3e-5 of the pixels, always at ties): unquantised
//                     weights and accumulation in double (fp32 accumulation alone flips ~3e-4 of the pixels), round half even.
struct CubicArgs {
  const uint8_t* base;
  size_t slot_stride;
  const int* slots;
  int n, w, h, pitch, luma_rows, format, out_w, out_h, mode, n_vec;
  const int *x0, *y0;
  const short *wxq, *wyq;
  const double *wxf, *wyf;
  uint8_t* out;
};

__global__ void resize_cubic_kernel(const CubicArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per = a.out_w * a.out_h;
  if (i >= a.n * per) return;
  const int f = i / per, p = i - f * per, yo = p / a.out_w, xo = p - yo * a.out_w;
  const uint8_t* fr = a.base + (size_t)a.slots[f] * a.slot_stride;
  const int xs = a.x0[xo], ys = a.y0[yo];
  int hs[4][3];
  double hf[4][3];  // IPP variant in double: fp32 accumulation alone moves ~3e-4 of the pixels across a rounding tie (measured)
#pragma unroll
  for (int ky = 0; ky < 4; ++ky) {
    const int y = min(max(ys + ky, 0), a.h - 1);
    int acc[3] = {0, 0, 0};
    double accf[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int kx = 0; kx < 4; ++kx) {
      const int x = min(max(xs + kx, 0), a.w - 1);
      int r, g, b;
      if (is_nv12(a.format)) {
        fetch_rgb_nv12(fr, a.pitch, a.luma_rows, x, y, r, g, b, a.format);
      } else {
        const uint8_t* px = fr + (size_t)y * a.pitch + 3 * x;
        r = px[0], g = px[1], b = px[2];
      }
      if (a.mode == CB_CUBIC_OPENCV) {
        const int wq = a.wxq[xo * 4 + kx];
        acc[0] += r * wq, acc[1] += g * wq, acc[2] += b * wq;
      } else {
        const double wf = a.wxf[xo * 4 + kx];
        accf[0] = fma((double)r, wf, accf[0]), accf[1] = fma((double)g, wf, accf[1]), accf[2] = fma((double)b, wf, accf[2]);
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) hs[ky][c] = acc[c], hf[ky][c] = accf[c];
  }
  uint8_t* o = a.out + (size_t)i * 3;
  if (a.mode == CB_CUBIC_OPENCV) {
    const float sc = 1.0f / 4194304.0f;  // 2^-22, exact
    const int b0i = a.wyq[yo * 4 + 0], b1i = a.wyq[yo * 4 + 1], b2i = a.wyq[yo * 4 + 2], b3i = a.wyq[yo * 4 + 3];
    const float b0 = (float)b0i * sc, b1 = (float)b1i * sc, b2 = (float)b2i * sc, b3 = (float)b3i * sc;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      int v;
      if (xo * 3 + c < a.n_vec) {
        float t = __fmul_rn((float)hs[3][c], b3);
        t = __fadd_rn(__fmul_rn((float)hs[2][c], b2), t);
        t = __fadd_rn(__fmul_rn((float)hs[1][c], b1), t);
        t = __fadd_rn(__fmul_rn((float)hs[0][c], b0), t);
        v = __float2int_rn(t);
      } else {
        const long long e = (long long)hs[0][c] * b0i + (long long)hs[1][c] * b1i + (long long)hs[2][c] * b2i + (long long)hs[3][c] * b3i;
        v = (int)((e + (1ll << 21)) >> 22);
      }
      o[c] = (uint8_t)min(max(v, 0), 255);
    }
  } else {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      double t = 0.0;
#pragma unroll
      for (int ky = 0; ky < 4; ++ky) t = fma(hf[ky][c], a.wyf[yo * 4 + ky], t);
      o[c] = (uint8_t)min(max(__double2int_rn(t), 0), 255);
    }
  }
}


// ------------------------------------------------------------------------------------------------ video-tower tubes
// cv2.resize(frame, (out_w, out_h)) [INTER_LINEAR, u8] + ((x / 255 - mean) / std) -> fp32 CHW: the input formulation of the
// video embedding towers (InternVideo2MultiModality._construct_frames / _normalize, models/internvideo2_mm.py:385-405).
// OpenCV's fixed-point arithmetic, bit for bit: int16 weights at 2^11 (each of the pair rounded on its own), horizontal pass
// in int32, vertical pass (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2; an exact 2x2 decimation is what
// cv2 reroutes to INTER_AREA ((a + b + c + d + 2) >> 2); equal sizes copy.  HBM-bound and sparse: 4 source pixels per output.
struct TubeArgs {
  const uint8_t* base;
  size_t slot_stride;
  const int* slots;
  int n, w, h, pitch, luma_rows, format, out_w, out_h, mode;  // mode 0 linear, 1 area 2x2, 2 copy
  const int *x0, *y0;
  const short *ax, *by;
  float mean[3], std_[3];
  float* out_f32;    // [n][3][out_h][out_w] or null
  uint8_t* out_u8;   // [n][out_h][out_w][3] or null
};

__device__ __forceinline__ void fetch_rgb_any(const TubeArgs& a, const uint8_t* fr, int x, int y, int& r, int& g, int& b) {
  if (is_nv12(a.format)) {
    fetch_rgb_nv12(fr, a.pitch, a.luma_rows, x, y, r, g, b, a.format);
  } else {
    const uint8_t* px = fr + (size_t)y * a.pitch + 3 * x;
    r = px[0], g = px[1], b = px[2];
  }
}

__global__ void video_tube_kernel(const TubeArgs a) {
  __shared__ float lut[3][256];
  for (int t = threadIdx.x; t < 768; t += blockDim.x) {
    const int c = t >> 8, v = t & 255;
    lut[c][v] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)v, 255.0f), a.mean[c]), a.std_[c]);
  }
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int per = a.out_w * a.out_h;
  if (i >= a.n * per) return;
  const int f = i / per, p = i - f * per, yo = p / a.out_w, xo = p - yo * a.out_w;
  const uint8_t* fr = a.base + (size_t)a.slots[f] * a.slot_stride;
  int v[3];
  if (a.mode == 2) {
    fetch_rgb_any(a, fr, xo, yo, v[0], v[1], v[2]);
  } else if (a.mode == 1) {
    int s[3] = {2, 2, 2};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      int r, g, b;
      fetch_rgb_any(a, fr, 2 * xo + (k & 1), 2 * yo + (k >> 1), r, g, b);
      s[0] += r, s[1] += g, s[2] += b;
    }
    v[0] = s[0] >> 2, v[1] = s[1] >> 2, v[2] = s[2] >> 2;
  } else {
    const int xs = a.x0[xo], ys = a.y0[yo];
    const int xa = min(max(xs, 0), a.w - 1), xb = min(max(xs + 1, 0), a.w - 1);
    const int ya = min(max(ys, 0), a.h - 1), yb = min(max(ys + 1, 0), a.h - 1);
    const int a0 = a.ax[2 * xo], a1 = a.ax[2 * xo + 1], b0 = a.by[2 * yo], b1 = a.by[2 * yo + 1];
    int p00[3], p01[3], p10[3], p11[3];
    fetch_rgb_any(a, fr, xa, ya, p00[0], p00[1], p00[2]);
    fetch_rgb_any(a, fr, xb, ya, p01[0], p01[1], p01[2]);
    fetch_rgb_any(a, fr, xa, yb, p10[0], p10[1], p10[2]);
    fetch_rgb_any(a, fr, xb, yb, p11[0], p11[1], p11[2]);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int s0 = p00[c] * a0 + p01[c] * a1, s1 = p10[c] * a0 + p11[c] * a1;
      v[c] = (((b0 * (s0 >> 4)) >> 16) + ((b1 * (s1 >> 4)) >> 16) + 2) >> 2;
    }
  }
  if (a.out_u8) {
    uint8_t* o = a.out_u8 + (size_t)i * 3;
    o[0] = (uint8_t)v[0], o[1] = (uint8_t)v[1], o[2] = (uint8_t)v[2];
  }
  if (a.out_f32) {
    float* o = a.out_f32 + (size_t)f * 3 * per + p;
#pragma unroll
    for (int c = 0; c < 3; ++c) o[(size_t)c * per] = lut[c][v[c] & 255];
  }
}

// ------------------------------------------------------------------------------------------------ host
static float cubic_aa(float x) {  // Keys a = -0.5, float32 like ATen's bicubic_filter
  const float a = -0.5f;
  if (x < 0.f) x = -x;
  if (x < 1.f) return ((a + 2.f) * x - (a + 3.f)) * x * x + 1.f;
  if (x < 2.f) return (((x - 5.f) * x + 8.f) * x - 4.f) * a;
  return 0.f;
}

const TapTable* get_taps(cb_ctx* ctx, int in_size, int out_size, int crop_off, int crop_len) {
  auto key = std::make_tuple(in_size, out_size, crop_off, crop_len);
  auto it = ctx->taps.find(key);
  if (it != ctx->taps.end()) return &it->second;
  TapTable t;
  t.in_size = in_size, t.out_size = out_size, t.crop_off = crop_off, t.crop_len = crop_len;
  // ATen upsample_antialias::_compute_weights_span / _compute_weights in float32
  volatile float scale = (float)in_size / (float)out_size;
  const float support = (scale >= 1.f) ? 2.0f * scale : 2.0f;
  const float invscale = (scale >= 1.f) ? 1.0f / scale : 1.0f;
  t.h_min.resize(crop_len), t.h_size.resize(crop_len);
  std::vector<std::vector<float>> w(crop_len);
  t.src_begin = in_size, t.src_end = 0;
  for (int o = 0; o < crop_len; ++o) {
    const int i = o + crop_off;
    volatile float center = scale * ((float)i + 0.5f);
    volatile float lo = center - support;
    volatile float hi = center + support;
    const int xmin = std::max((int)(lo + 0.5f), 0);
    const int xsize = std::min((int)(hi + 0.5f), in_size) - xmin;
    volatile float xmin_m_center = (float)xmin - center;
    volatile float total = 0.f;
    w[o].resize(xsize);
    for (int j = 0; j < xsize; ++j) {
      volatile float arg = ((float)j + xmin_m_center + 0.5f);
      arg = arg * invscale;
      const float wv = cubic_aa(arg);
      w[o][j] = wv;
      total = total + wv;
    }
    if (total != 0.f)
      for (int j = 0; j < xsize; ++j) w[o][j] = w[o][j] / total;
    t.h_min[o] = xmin, t.h_size[o] = xsize;
    t.max_taps = std::max(t.max_taps, xsize);
    t.src_begin = std::min(t.src_begin, xmin);
    t.src_end = std::max(t.src_end, xmin + xsize);
  }
  std::vector<float> flat((size_t)crop_len * t.max_taps, 0.f);
  for (int o = 0; o < crop_len; ++o) std::copy(w[o].begin(), w[o].end(), flat.begin() + (size_t)o * t.max_taps);
  if (cudaMalloc(&t.d_min, crop_len * sizeof(int)) != cudaSuccess || cudaMalloc(&t.d_size, crop_len * sizeof(int)) != cudaSuccess ||
      cudaMalloc(&t.d_w, flat.size() * sizeof(float)) != cudaSuccess)
    return nullptr;
  cudaMemcpy(t.d_min, t.h_min.data(), crop_len * sizeof(int), cudaMemcpyHostToDevice);
  cudaMemcpy(t.d_size, t.h_size.data(), crop_len * sizeof(int), cudaMemcpyHostToDevice);
  cudaMemcpy(t.d_w, flat.data(), flat.size() * sizeof(float), cudaMemcpyHostToDevice);
  t.h_w = flat;
  auto res = ctx->taps.emplace(key, std::move(t));
  return &res.first->second;
}

int ensure_norm_lut(cb_ctx* ctx, const float mean[3], const float std_[3], cudaStream_t stream) {
  bool same = ctx->d_norm_lut != nullptr;
  for (int c = 0; c < 3 && same; ++c) same = ctx->lut_mean[c] == mean[c] && ctx->lut_std[c] == std_[c];
  if (same) return CB_OK;
  if (!ctx->d_norm_lut) CB_CUDA(ctx, cudaMalloc(&ctx->d_norm_lut, 3 * 256 * sizeof(float)));
  float lut[3 * 256];
  for (int c = 0; c < 3; ++c)
    for (int v = 0; v < 256; ++v) {
      volatile float x = (float)v / 255.0f;  // ConvertImageDtype: u8 -> float32 then / 255
      volatile float d = x - mean[c];        // Normalize: sub_ then div_
      lut[c * 256 + v] = d / std_[c];
    }
  // synchronous copy on the caller's stream order: the table is tiny and rarely changes
  CB_CUDA(ctx, cudaMemcpyAsync(ctx->d_norm_lut, lut, sizeof(lut), cudaMemcpyHostToDevice, stream));
  CB_CUDA(ctx, cudaStreamSynchronize(stream));
  for (int c = 0; c < 3; ++c) ctx->lut_mean[c] = mean[c], ctx->lut_std[c] = std_[c];
  return CB_OK;
}

static int python_round_half_even(double v) { return (int)std::nearbyint(v); }  // default FE_TONEAREST

static int upload_slots(cb_ctx* ctx, const int32_t* slots, int n, cudaStream_t stream, const int** out) {
  if (ctx->slots_cap < n) {
    if (ctx->d_slots) {
      CB_CUDA(ctx, cudaStreamSynchronize(stream));  // a previous launch may still read the old list
      cudaFree(ctx->d_slots);
    }
    ctx->slots_cap = std::max(1024, n);
    CB_CUDA(ctx, cudaMalloc(&ctx->d_slots, ctx->slots_cap * sizeof(int)));
  }
  CB_CUDA(ctx, cudaMemcpyAsync(ctx->d_slots, slots, n * sizeof(int), cudaMemcpyHostToDevice, stream));
  *out = ctx->d_slots;
  return CB_OK;
}

static int check_pool(cb_ctx* ctx, const cb_surface_pool* pool, int n, const int32_t* slots) {
  if (!ctx) return CB_ERR_ARG;
  if (!pool || !pool->base || n < 0 || (n > 0 && !slots)) return fail(ctx, CB_ERR_ARG, "null pool/slots");
  if (!is_nv12(pool->format) && pool->format != CB_FMT_RGB24) return fail(ctx, CB_ERR_ARG, "unknown surface format %d", pool->format);
  if (pool->width <= 0 || pool->height <= 0) return fail(ctx, CB_ERR_ARG, "bad surface size %dx%d", pool->width, pool->height);
  const int min_pitch = is_nv12(pool->format) ? pool->width : 3 * pool->width;
  if (pool->pitch < min_pitch) return fail(ctx, CB_ERR_ARG, "pitch %d < row bytes %d", pool->pitch, min_pitch);
  if (is_nv12(pool->format) && pool->luma_rows < pool->height) return fail(ctx, CB_ERR_ARG, "luma_rows < height");
  for (int i = 0; i < n; ++i)
    if (slots[i] < 0) return fail(ctx, CB_ERR_ARG, "negative slot index");
  return CB_OK;
}

int run_clip_preprocess(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int res, int out_mode, int layout_patch,
                        int k_pad, int dtype, const float mean[3], const float std_[3], void* out, cudaStream_t stream) {
  int rc = check_pool(ctx, pool, n, slots);
  if (rc) return rc;
  if (n == 0) return CB_OK;
  if (!out) return fail(ctx, CB_ERR_ARG, "null output");
  if (res <= 0 || res > 1024) return fail(ctx, CB_ERR_ARG, "bad output resolution %d", res);
  if (((uintptr_t)pool->base & 15) || (pool->pitch & 15) || (pool->slot_stride & 15))
    return fail(ctx, CB_ERR_ARG, "TMA needs base/pitch/slot_stride multiples of 16 bytes");
  if (is_nv12(pool->format) && ((pool->width | pool->height) & 1)) return fail(ctx, CB_ERR_UNSUPPORTED, "NV12 needs even dimensions");
  const int W = pool->width, H = pool->height;
  // torchvision: short side -> res, long side -> int(res * long / short); centre crop res x res
  int new_w, new_h;
  if (W <= H) new_w = res, new_h = (int)((long long)res * H / W);
  else new_h = res, new_w = (int)((long long)res * W / H);
  const int top = python_round_half_even((new_h - res) / 2.0), left = python_round_half_even((new_w - res) / 2.0);
  const TapTable* tx = get_taps(ctx, W, new_w, left, res);
  const TapTable* ty = get_taps(ctx, H, new_h, top, res);
  if (!tx || !ty) return fail(ctx, CB_ERR_CUDA, "tap table allocation failed");

  ClipArgs a{};
  a.n = n, a.src_w = W, a.src_h = H, a.res = res;
  a.xmin = tx->d_min, a.xsize = tx->d_size, a.wx = tx->d_w, a.tx = tx->max_taps;
  a.ymin = ty->d_min, a.ysize = ty->d_size, a.wy = ty->d_w, a.ty = ty->max_taps;
  a.out_mode = out_mode, a.dtype = dtype, a.patch = layout_patch, a.k_pad = k_pad, a.out = out;
  if (out_mode == 2) {
    if (layout_patch <= 0 || layout_patch > 32 || res < layout_patch) return fail(ctx, CB_ERR_UNSUPPORTED, "patch %d unsupported for res %d", layout_patch, res);
    if (k_pad < 3 * layout_patch * layout_patch || (k_pad & 7)) return fail(ctx, CB_ERR_ARG, "k_pad %d must be >= 3*p*p and a multiple of 8", k_pad);
    if (dtype != CB_DT_F16 && dtype != CB_DT_BF16) return fail(ctx, CB_ERR_ARG, "patch layout needs a 16-bit dtype");
    a.tc = layout_patch * (32 / layout_patch);
    a.res_out = (res / layout_patch) * layout_patch;
  } else {
    a.tc = 32;
    a.res_out = res;
  }
  a.y_begin = ty->src_begin & ~1;
  a.n_strips = (ty->src_end - a.y_begin + kSR - 1) / kSR;
  int ring = 64;
  while (ring < kSR + ty->max_taps) ring <<= 1;
  a.ring = ring;
  a.x_align = 16;  // cp.async.bulk.tensor needs the box to start on a 16-byte boundary of the innermost dimension
  // widest source span of any column tile; strong downscales (4K -> 224: 9.6 source pixels per output column) halve the tile so that
  // the window still fits one TMA box (256 bytes of the innermost dimension)
  int span = 0, tiles = 0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    span = 0;
    tiles = (a.res_out + a.tc - 1) / a.tc;
    for (int t = 0; t < tiles; ++t) {
      const int c0 = t * a.tc, c1 = std::min(a.res_out, c0 + a.tc);
      int lo = tx->h_min[c0] & ~(a.x_align - 1), hi = 0;
      for (int c = c0; c < c1; ++c) hi = std::max(hi, tx->h_min[c] + tx->h_size[c]);
      span = std::max(span, hi - lo);
    }
    if (span <= 256 || attempt == 1) break;
    a.tc = out_mode == 2 ? layout_patch * std::max(1, 16 / layout_patch) : 16;
  }
  a.swa = (span + 15) & ~15;
  // widest union window of any group of 4 adjacent output columns
  int gu = 1;
  for (int c = 0; c < res; c += 4) {
    if ((c % a.tc) + 4 > a.tc && (c % a.tc) % 4) continue;
    const int cl = std::min(res, std::min(c + 4, (c / a.tc + 1) * a.tc));
    int hi = 0;
    for (int k = c; k < cl; ++k) hi = std::max(hi, tx->h_min[k] + tx->h_size[k] - tx->h_min[c]);
    gu = std::max(gu, hi);
  }
  a.gu = gu;
  if (ty->max_taps > 64 || tx->max_taps > 64) return fail(ctx, CB_ERR_UNSUPPORTED, "downscale factor too large (%d vertical taps)", ty->max_taps);

  rc = ensure_norm_lut(ctx, mean, std_, stream);
  if (rc) return rc;
  a.lut = ctx->d_norm_lut;
  rc = upload_slots(ctx, slots, n, stream, &a.slots);
  if (rc) return rc;

  int max_slot = 0;
  for (int i = 0; i < n; ++i) max_slot = std::max(max_slot, (int)slots[i]);
  // default: horizontal pass on the tensor pipe (preprocess_tc.cu), which returns 1 for plans it does not take
  const char* kver = getenv("CB_PRE_KERNEL");
  if (!kver || std::strcmp(kver, "2") != 0) {
    rc = run_clip_preprocess_tc(ctx, pool, a.slots, n, max_slot, res, out_mode, layout_patch, k_pad, dtype, tx, ty, out, stream);
    if (rc <= 0) return rc;
  }
  if (a.swa > 256) return fail(ctx, CB_ERR_UNSUPPORTED, "downscale too large for one TMA box (%d source columns per tile)", a.swa);
  CUtensorMap map_a, map_b;
  if (is_nv12(pool->format)) {
    uint64_t dims[3] = {(uint64_t)W, (uint64_t)H, (uint64_t)max_slot + 1};
    uint64_t strides[2] = {(uint64_t)pool->pitch, (uint64_t)pool->slot_stride};
    uint32_t box[3] = {(uint32_t)a.swa, (uint32_t)kSR, 1};
    rc = make_tensor_map(ctx, &map_a, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, pool->base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    uint64_t dims_uv[3] = {(uint64_t)W, (uint64_t)(H / 2), (uint64_t)max_slot + 1};
    uint32_t box_uv[3] = {(uint32_t)a.swa, (uint32_t)(kSR / 2), 1};
    rc = make_tensor_map(ctx, &map_b, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (const uint8_t*)pool->base + (size_t)pool->luma_rows * pool->pitch,
                         dims_uv, strides, box_uv, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
  } else {
    uint64_t dims[3] = {(uint64_t)W * 3, (uint64_t)H, (uint64_t)max_slot + 1};
    uint64_t strides[2] = {(uint64_t)pool->pitch, (uint64_t)pool->slot_stride};
    uint32_t box[3] = {(uint32_t)a.swa, (uint32_t)kSR, 1};
    rc = make_tensor_map(ctx, &map_a, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, pool->base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    map_b = map_a;
  }

  const int raw_stage = is_nv12(pool->format) ? (a.swa * kSR * 3 / 2) : (3 * a.swa * kSR);
  const int npx = out_mode == 2 ? a.tc / a.patch : 0;
  size_t smem = 2 * (size_t)raw_stage + (size_t)3 * kSR * (a.swa + 1) * 4 + (size_t)3 * a.ring * (a.tc | 1) * 4 + (size_t)npx * k_pad * 2 + 32;
  smem += 48 + (size_t)((a.tc + 3) / 4) * a.gu * 16 + (size_t)2 * ((a.tc + 3) / 4) * 4;
  if (smem > 227 * 1024) return fail(ctx, CB_ERR_UNSUPPORTED, "preprocess tile needs %zu bytes of shared memory", smem);
  dim3 grid(tiles, n);
  mark_launch(ctx, CB_PROF_PREPROCESS, stream);
#define CB_LAUNCH_PRE(KERNEL, F)                                                                                         \
  do {                                                                                                                  \
    CB_CUDA(ctx, cudaFuncSetAttribute(KERNEL<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));               \
    KERNEL<F><<<grid, kThreads, smem, stream>>>(map_a, map_b, a);                                                        \
  } while (0)
  if (pool->format == CB_FMT_NV12) CB_LAUNCH_PRE(clip_preprocess_v2_kernel, CB_FMT_NV12);
  else if (pool->format == CB_FMT_NV12_SWS) CB_LAUNCH_PRE(clip_preprocess_v2_kernel, CB_FMT_NV12_SWS);
  else CB_LAUNCH_PRE(clip_preprocess_v2_kernel, CB_FMT_RGB24);
#undef CB_LAUNCH_PRE
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

static int run_simple(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h, uint8_t* out, bool bilinear,
                      cudaStream_t stream) {
  int rc = check_pool(ctx, pool, n, slots);
  if (rc) return rc;
  if (n == 0) return CB_OK;
  if (!out) return fail(ctx, CB_ERR_ARG, "null output");
  if (!is_nv12(pool->format)) return fail(ctx, CB_ERR_UNSUPPORTED, "NV12 surfaces only");
  SimpleArgs a{};
  a.base = (const uint8_t*)pool->base, a.slot_stride = pool->slot_stride;
  a.n = n, a.w = pool->width, a.h = pool->height, a.pitch = pool->pitch, a.luma_rows = pool->luma_rows;
  a.out_w = out_w, a.out_h = out_h, a.out = out, a.format = pool->format;
  rc = upload_slots(ctx, slots, n, stream, &a.slots);
  if (rc) return rc;
  if (bilinear && (out_w <= 0 || out_h <= 0)) return fail(ctx, CB_ERR_ARG, "bad output size");
  mark_launch(ctx, CB_PROF_PREPROCESS, stream);
  if (bilinear) {
    const long long total = (long long)n * out_w * out_h;
    bilinear_u8_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(a);
  } else {
    const long long total = (long long)n * a.h * ((a.w + 1) / 2);
    nv12_to_rgb_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(a);
  }
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

// OpenCV resize(): fx = float((dx + 0.5) * scale - 0.5) with scale = 1 / (dst / src) in double; interpolateCubic in float.
static const CubicTaps* get_cubic_taps(cb_ctx* ctx, int src, int dst) {
  std::lock_guard<std::mutex> lk(ctx->mu);
  auto key = std::make_pair(src, dst);
  auto it = ctx->cubic_taps.find(key);
  if (it != ctx->cubic_taps.end()) return &it->second;
  std::vector<int> first(dst);
  std::vector<short> wq(4 * (size_t)dst);
  std::vector<double> wf(4 * (size_t)dst);
  const double inv_scale = (double)dst / (double)src, scale = 1.0 / inv_scale;
  for (int d = 0; d < dst; ++d) {
    float fx = (float)((d + 0.5) * scale - 0.5);
    const int sx = (int)std::floor(fx);
    fx -= (float)sx;
    first[d] = sx - 1;
    const float A = -0.75f;
    float c[4];
    c[0] = ((A * (fx + 1.f) - 5.f * A) * (fx + 1.f) + 8.f * A) * (fx + 1.f) - 4.f * A;
    c[1] = ((A + 2.f) * fx - (A + 3.f)) * fx * fx + 1.f;
    c[2] = ((A + 2.f) * (1.f - fx) - (A + 3.f)) * (1.f - fx) * (1.f - fx) + 1.f;
    c[3] = 1.f - c[0] - c[1] - c[2];
    // float path: the same Keys kernel evaluated in double at the double-precision phase (what a correctly rounded result needs)
    const double pos = (d + 0.5) * scale - 0.5, fr = pos - std::floor(pos), Ad = -0.75;
    const double cd[4] = {((Ad * (fr + 1) - 5 * Ad) * (fr + 1) + 8 * Ad) * (fr + 1) - 4 * Ad, ((Ad + 2) * fr - (Ad + 3)) * fr * fr + 1,
                          ((Ad + 2) * (1 - fr) - (Ad + 3)) * (1 - fr) * (1 - fr) + 1, 0.0};
    for (int k = 0; k < 4; ++k) {
      const float q = std::nearbyint(c[k] * 2048.f);  // saturate_cast<short>(float) = cvRound: half to even
      wq[4 * (size_t)d + k] = (short)std::min(32767.f, std::max(-32768.f, q));
      wf[4 * (size_t)d + k] = k < 3 ? cd[k] : 1.0 - cd[0] - cd[1] - cd[2];
    }
  }
  CubicTaps t;
  if (cudaMalloc(&t.d_first, dst * sizeof(int)) != cudaSuccess || cudaMalloc(&t.d_wq, 4 * (size_t)dst * sizeof(short)) != cudaSuccess ||
      cudaMalloc(&t.d_wf, 4 * (size_t)dst * sizeof(double)) != cudaSuccess)
    return nullptr;
  cudaMemcpy(t.d_first, first.data(), dst * sizeof(int), cudaMemcpyHostToDevice);
  cudaMemcpy(t.d_wq, wq.data(), 4 * (size_t)dst * sizeof(short), cudaMemcpyHostToDevice);
  cudaMemcpy(t.d_wf, wf.data(), 4 * (size_t)dst * sizeof(double), cudaMemcpyHostToDevice);
  return &(ctx->cubic_taps[key] = t);
}

static int run_resize_cubic(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h, int mode, uint8_t* out,
                            cudaStream_t stream) {
  int rc = check_pool(ctx, pool, n, slots);
  if (rc) return rc;
  if (n == 0) return CB_OK;
  if (!out) return fail(ctx, CB_ERR_ARG, "null output");
  if (out_w <= 0 || out_h <= 0 || out_w > 8192 || out_h > 8192) return fail(ctx, CB_ERR_ARG, "bad output size %dx%d", out_w, out_h);
  if (mode != CB_CUBIC_OPENCV && mode != CB_CUBIC_IPP) return fail(ctx, CB_ERR_ARG, "unknown cubic mode %d", mode);
  if (is_nv12(pool->format) && ((pool->width | pool->height) & 1)) return fail(ctx, CB_ERR_UNSUPPORTED, "NV12 needs even dimensions");
  const CubicTaps* tx = get_cubic_taps(ctx, pool->width, out_w);
  const CubicTaps* ty = get_cubic_taps(ctx, pool->height, out_h);
  if (!tx || !ty) return fail(ctx, CB_ERR_CUDA, "cubic tap table allocation failed");
  CubicArgs a{};
  a.base = (const uint8_t*)pool->base, a.slot_stride = pool->slot_stride;
  a.n = n, a.w = pool->width, a.h = pool->height, a.pitch = pool->pitch, a.luma_rows = pool->luma_rows, a.format = pool->format;
  a.out_w = out_w, a.out_h = out_h, a.mode = mode, a.out = out;
  a.n_vec = (out_w * 3) / 8 * 8;  // elements of a row handled by the 8-lane vector body of VResizeCubicVec_32s8u
  a.x0 = tx->d_first, a.wxq = tx->d_wq, a.wxf = tx->d_wf, a.y0 = ty->d_first, a.wyq = ty->d_wq, a.wyf = ty->d_wf;
  rc = upload_slots(ctx, slots, n, stream, &a.slots);
  if (rc) return rc;
  mark_launch(ctx, CB_PROF_PREPROCESS, stream);
  const long long total = (long long)n * out_w * out_h;
  resize_cubic_kernel<<<(unsigned)((total + 127) / 128), 128, 0, stream>>>(a);
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

// OpenCV resize() linear taps: the column table zeroes fx at the borders, the row table clamps rows instead (resize.cpp).
static const CubicTaps* get_linear_taps(cb_ctx* ctx, int src, int dst, bool zero_at_border) {
  std::lock_guard<std::mutex> lk(ctx->mu);
  auto key = std::make_tuple(src, dst, zero_at_border ? 1 : 0);
  auto it = ctx->linear_taps.find(key);
  if (it != ctx->linear_taps.end()) return &it->second;
  std::vector<int> first(dst);
  std::vector<short> wq(2 * (size_t)dst);
  const double inv_scale = (double)dst / (double)src, scale = 1.0 / inv_scale;
  for (int d = 0; d < dst; ++d) {
    float fx = (float)((d + 0.5) * scale - 0.5);
    int sx = (int)std::floor(fx);
    fx -= (float)sx;
    if (zero_at_border) {
      if (sx < 0) fx = 0.f, sx = 0;
      if (sx >= src - 1) fx = 0.f, sx = src - 1;
    }
    first[d] = sx;
    const float c[2] = {1.f - fx, fx};
    for (int k = 0; k < 2; ++k) {
      const float q = std::nearbyint(c[k] * 2048.f);  // saturate_cast<short>(float) = cvRound: half to even
      wq[2 * (size_t)d + k] = (short)std::min(32767.f, std::max(-32768.f, q));
    }
  }
  CubicTaps t;
  if (cudaMalloc(&t.d_first, dst * sizeof(int)) != cudaSuccess || cudaMalloc(&t.d_wq, 2 * (size_t)dst * sizeof(short)) != cudaSuccess)
    return nullptr;
  cudaMemcpy(t.d_first, first.data(), dst * sizeof(int), cudaMemcpyHostToDevice);
  cudaMemcpy(t.d_wq, wq.data(), 2 * (size_t)dst * sizeof(short), cudaMemcpyHostToDevice);
  return &(ctx->linear_taps[key] = t);
}

static int run_video_tube(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h, const float mean[3],
                          const float std_[3], float* out_f32, uint8_t* out_u8, cudaStream_t stream) {
  int rc = check_pool(ctx, pool, n, slots);
  if (rc) return rc;
  if (n == 0) return CB_OK;
  if (!out_f32 && !out_u8) return fail(ctx, CB_ERR_ARG, "null output");
  if (out_w <= 0 || out_h <= 0 || out_w > 8192 || out_h > 8192) return fail(ctx, CB_ERR_ARG, "bad output size %dx%d", out_w, out_h);
  if (out_f32 && (!mean || !std_)) return fail(ctx, CB_ERR_ARG, "null mean/std");
  if (is_nv12(pool->format) && ((pool->width | pool->height) & 1)) return fail(ctx, CB_ERR_UNSUPPORTED, "NV12 needs even dimensions");
  if ((long long)n * out_w * out_h > 0x7fffffffLL) return fail(ctx, CB_ERR_ARG, "too many output pixels for one call");
  TubeArgs a{};
  a.base = (const uint8_t*)pool->base, a.slot_stride = pool->slot_stride;
  a.n = n, a.w = pool->width, a.h = pool->height, a.pitch = pool->pitch, a.luma_rows = pool->luma_rows, a.format = pool->format;
  a.out_w = out_w, a.out_h = out_h, a.out_f32 = out_f32, a.out_u8 = out_u8;
  for (int c = 0; c < 3; ++c) a.mean[c] = mean ? mean[c] : 0.f, a.std_[c] = std_ ? std_[c] : 1.f;
  if (a.w == out_w && a.h == out_h) {
    a.mode = 2;
  } else if (a.w == 2 * out_w && a.h == 2 * out_h) {
    a.mode = 1;
  } else {
    a.mode = 0;
    const CubicTaps* tx = get_linear_taps(ctx, a.w, out_w, true);
    const CubicTaps* ty = get_linear_taps(ctx, a.h, out_h, false);
    if (!tx || !ty) return fail(ctx, CB_ERR_CUDA, "linear tap table allocation failed");
    a.x0 = tx->d_first, a.ax = tx->d_wq, a.y0 = ty->d_first, a.by = ty->d_wq;
  }
  rc = upload_slots(ctx, slots, n, stream, &a.slots);
  if (rc) return rc;
  mark_launch(ctx, CB_PROF_PREPROCESS, stream);
  const long long total = (long long)n * out_w * out_h;
  video_tube_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(a);
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

int bilinear_from_surface(cb_ctx* ctx, const void* base, int pitch, int luma_rows, int w, int h, int out_w, int out_h, uint8_t* out,
                          cudaStream_t stream) {
  SimpleArgs a{};
  a.base = (const uint8_t*)base, a.slot_stride = 0, a.slots = nullptr;
  a.n = 1, a.w = w, a.h = h, a.pitch = pitch, a.luma_rows = luma_rows, a.out_w = out_w, a.out_h = out_h, a.out = out, a.format = CB_FMT_NV12;
  mark_launch(ctx, CB_PROF_PREPROCESS, stream);
  bilinear_u8_kernel<<<(out_w * out_h + 255) / 256, 256, 0, stream>>>(a);
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

}  // namespace cb

extern "C" {

int cb_preprocess_clip(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int res, int layout, int patch, int k_pad,
                       int dtype, const float mean[3], const float std_[3], void* out, void* stream) {
  if (!ctx) return CB_ERR_ARG;
  if (!mean || !std_) return cb::fail(ctx, CB_ERR_ARG, "null mean/std");
  if (layout != CB_LAYOUT_NCHW && layout != CB_LAYOUT_PATCH) return cb::fail(ctx, CB_ERR_ARG, "unknown layout %d", layout);
  if (dtype < CB_DT_F16 || dtype > CB_DT_F32) return cb::fail(ctx, CB_ERR_ARG, "unknown dtype %d", dtype);
  return cb::run_clip_preprocess(ctx, pool, slots, n, res, layout == CB_LAYOUT_PATCH ? 2 : 1, patch, k_pad, dtype, mean, std_, out,
                                 (cudaStream_t)stream);
}

int cb_preprocess_clip_u8(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int res, uint8_t* out, void* stream) {
  if (!ctx) return CB_ERR_ARG;
  const float m[3] = {0, 0, 0}, s[3] = {1, 1, 1};
  return cb::run_clip_preprocess(ctx, pool, slots, n, res, 0, 0, 0, CB_DT_F32, m, s, out, (cudaStream_t)stream);
}

int cb_preprocess_bilinear_u8(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h, uint8_t* out,
                              void* stream) {
  if (!ctx) return CB_ERR_ARG;
  return cb::run_simple(ctx, pool, slots, n, out_w, out_h, out, true, (cudaStream_t)stream);
}

int cb_resize_cubic_u8(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h, int mode, uint8_t* out,
                       void* stream) {
  if (!ctx) return CB_ERR_ARG;
  return cb::run_resize_cubic(ctx, pool, slots, n, out_w, out_h, mode, out, (cudaStream_t)stream);
}

int cb_video_tube(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, int out_w, int out_h, const float mean[3],
                  const float std_[3], float* out_f32, uint8_t* out_u8, void* stream) {
  if (!ctx) return CB_ERR_ARG;
  return cb::run_video_tube(ctx, pool, slots, n, out_w, out_h, mean, std_, out_f32, out_u8, (cudaStream_t)stream);
}

int cb_nv12_to_rgb(cb_ctx* ctx, const cb_surface_pool* pool, const int32_t* slots, int n, uint8_t* out, void* stream) {
  if (!ctx) return CB_ERR_ARG;
  return cb::run_simple(ctx, pool, slots, n, 0, 0, out, false, (cudaStream_t)stream);
}

}  // extern "C"
