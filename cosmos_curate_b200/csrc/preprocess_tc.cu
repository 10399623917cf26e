// Third-generation fused preprocess: the horizontal antialiased-bicubic pass on the tensor pipe (tcgen05), everything else SIMT.
//
// Same arithmetic contract as clip_preprocess_v2_kernel (preprocess.cu): NV12 -> RGB u8 (OpenCV or libswscale arithmetic) ->
// torchvision Resize(res, bicubic, antialias) + CenterCrop(res) with fp32 intermediates -> round half even -> u8.  The v2
// kernel is issue / shared-memory bound (ncu: 1.16 M shared wavefronts per 1080p frame, tensor pipe idle): 83 % of its FMAs
// are the ~20-tap horizontal pass.  Here that pass is a banded GEMM on the tensor cores:
//
//   D[(row, colour plane), x] = sum_k  A[(row, colour plane), k] * (Wh[x, k] + Wl[x, k])
//
//   * A = the colour-converted pixels as fp16 (0..255 is exact in fp16), written by the SIMT threads straight into the
//     128-byte-swizzled K-major UMMA layout.  The M dimension stacks 40 source rows x 3 colour planes = 120 of the 128 UMMA
//     rows, so one 128-row operand tile holds a whole unit of work and all three planes share the B operand (the weights).
//   * B = the fp32 tap weights split into two fp16 terms (hi + lo, 22 significant bits: products with u8 pixels are exact in
//     the fp32 accumulator, only the summation order differs from ATen's - the <= 1 LSB on <= 1e-4 of the pixels budget the
//     fp32 paths already share).  An N-tile is 16 output columns; its K window is the ~100 source columns those columns
//     tap (7 k-steps of 16), so the band is ~70 % dense instead of a dense 1080-wide GEMM.  The hi and lo terms of a tile sit
//     side by side in the B tile (N = 32): a UMMA with M = 128 streams its A rows from shared memory in ~128 cycles whatever N
//     is, so the number of instructions, not their width, is what costs (14 per unit).
//   * accumulators in TMEM (64 columns per CTA: N-tile x weight term), read back with tcgen05.ld, hi + lo added, into a 64-row
//     ring of filtered rows in shared memory; the vertical pass (17 % of the FMAs) stays on the FMA pipe in ATen's order (it
//     runs while the next unit's MMAs are in flight), then round / clamp / store u8.
//
// A CTA owns (frame, 32 output columns) and walks the source rows top to bottom in units of 40 rows: TMA load of the NV12
// window (Y + UV boxes) -> convert -> 14 MMAs -> epilogue -> vertical pass for the output rows that became complete.
// ~105 KB of shared memory per CTA: two CTAs per SM overlap each other's phases.  Output: u8 [n][3][res][res]; normalisation +
// patch packing is a second, bandwidth-trivial kernel (pack_patches_kernel / normalize_pack_kernel) so that this one stays small.
#include <algorithm>
#include <cstring>
#include <vector>

#include <cuda_bf16.h>

#include "common.h"
#include "ptx.cuh"

namespace cb {

constexpr int kNC = 32;          // output columns per CTA = two UMMA N-tiles of 16
constexpr int kRingRows = 64;    // ring of horizontally filtered rows
constexpr int kRingStride = 3 * kNC + 4;  // floats per ring row: +16 B so that the epilogue's row-per-lane 16-byte stores spread over the banks
constexpr int kMaxUnits = 128;            // units per frame column (4K: 55)
constexpr int kVRows = 16, kVTaps = 40;   // vertical-pass weights of one unit staged in shared memory (rows x taps)
constexpr int kTcThreads = 320;  // 10 warps: 20 row pairs x kw / 4 column groups of the convert phase divide evenly (kw = 128 / 192 / 256)
// mbarrier waits suspend in hardware for up to this long instead of re-polling, which spares the co-resident CTA's issue
// slots; spin, 32, 200 and 2000 ns measured the same
constexpr int kWaitNs = 2000;

struct TcArgs {
  const int* slots;
  int n, res, ru, n_units, y_begin, kw, kb, colour;
  int nc;                  // output columns per CTA slab: 32 (two N-tiles), or 16 when the downscale is so strong that 32 columns' window exceeds a TMA box
  const int* x_lo;         // [n_slabs] first source column of the slab window (multiple of 16)
  const int* tile_k0;      // [n_slabs * 2] first k-step (16 source columns) of the N-tile inside the window
  const int* tile_nk;      // [n_slabs * 2] k-steps of the N-tile (0 = tile beyond the image)
  const uint8_t* wtiles;   // [n_slabs][2 tiles][kb / 64][32 rows (hi | lo)][128 B] fp16, already in the swizzled UMMA layout
  const int *ymin, *ysize;
  const int* unit_last;    // [n_units] output rows complete once unit u has been filtered
  const float* wy;
  int ty;
  uint8_t* out;  // [n][3][res][res]
};

__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

// two integers 0..255 -> packed fp16 pair, exactly: 0x6400 | v is the fp16 1024 + v, and (1024 + v) - 1024 is exact
__device__ __forceinline__ uint32_t pack_u8_pair_f16(int a, int b) {
  uint32_t p = (uint32_t)(a | (b << 16)) | 0x64006400u;
  __half2 h = *reinterpret_cast<__half2*>(&p);
  h = __hsub2(h, __half2half2(__ushort_as_half((unsigned short)0x6400)));
  return *reinterpret_cast<uint32_t*>(&h);
}

__global__ void __launch_bounds__(kTcThreads, 2)
    clip_preprocess_tc_kernel(const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_uv, const TcArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  const int kw = a.kw, ru = a.ru;
  const int b_tile = (a.kb >> 6) * 4096;  // one N-tile of the B operand: 32 rows (16 columns x {hi, lo} weight term) x kb
  uint8_t* sA = smem;                // [kw / 64][16 row groups][8 rows][128 B]
  uint8_t* sB = sA + kw * 256;       // [tile][kb / 64][32 rows: hi 0..15 | lo 16..31][128 B]
  uint8_t* sRaw = sB + 2 * b_tile;   // ru luma rows then ru / 2 chroma rows, kw bytes each
  const int raw_bytes = (((ru + ru / 2) * kw) + 127) & ~127;
  float* ring = reinterpret_cast<float*>(sRaw + raw_bytes);  // [kRingRows][kRingStride]: row = [3 planes][kNC] + pad
  float* sW = ring + kRingRows * kRingStride;                 // [kVRows][kVTaps] vertical taps of the output rows this unit completes
  int* sY = reinterpret_cast<int*>(sW + kVRows * kVTaps);     // [kVRows][2] first ring row, tap count
  int* sUL = sY + 2 * kVRows;                                 // [kMaxUnits] copy of unit_last (a global load per phase would sit on the critical path)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sUL + kMaxUnits);
  uint64_t* raw_full = bars;
  uint64_t* mma_done = bars + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int slab = blockIdx.x, frame = blockIdx.y;
  const int slot = a.slots[frame];
  const int x_lo = a.x_lo[slab], x0 = slab * a.nc;
  const int ncols = min(a.nc, a.res - x0);

  if (tid == 0) {
    mbar_init(raw_full, 1), mbar_init(mma_done, 1);
    fence_barrier_init();
    tma_prefetch_desc(&map_y), tma_prefetch_desc(&map_uv);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 64);
    tmem_relinquish();
  }
  {
    const uint4* src = reinterpret_cast<const uint4*>(a.wtiles + (size_t)slab * 2 * b_tile);
    uint4* dst = reinterpret_cast<uint4*>(sB);
    for (int i = tid; i < (2 * b_tile) >> 4; i += kTcThreads) dst[i] = src[i];
    for (int i = tid; i < a.n_units; i += kTcThreads) sUL[i] = a.unit_last[i];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t raw_tx = (uint32_t)((ru + ru / 2) * kw);
  auto issue = [&](int u) {
    const int ys = a.y_begin + u * ru;
    mbar_expect_tx(raw_full, raw_tx);
    tma_load_3d(sRaw, &map_y, raw_full, x_lo, ys, slot);
    tma_load_3d(sRaw + ru * kw, &map_uv, raw_full, x_lo, ys >> 1, slot);
  };
  if (tid == 0) issue(0);

  constexpr uint32_t idesc = umma_idesc_f16(128, 32, 0);  // N = 32: the hi and lo weight terms of 16 output columns side by side
  // per-CTA constants of the MMA issuer: k-step windows of the two N-tiles and the operand descriptor bases (16-byte units)
  const int nk0 = a.tile_nk[slab * 2], nk1 = a.tile_nk[slab * 2 + 1], k00 = a.tile_k0[slab * 2], k01 = a.tile_k0[slab * 2 + 1];
  const int nkm = nk0 > nk1 ? nk0 : nk1;
  const uint64_t desc_a0 = umma_desc_sw128(smem_u32(sA)), desc_b0 = umma_desc_sw128(smem_u32(sB));
  const uint32_t b_tile16 = (uint32_t)b_tile >> 4;
  const int q4 = kw >> 2;
  const int rp0 = tid / q4, xg0 = tid - rp0 * q4, drp = kTcThreads / q4, dxg = kTcThreads - drp * q4;  // item walk of the convert phase
  const int plane_bytes = (ru >> 3) << 10;                                                             // ru rows = ru / 8 row groups of 1 KB
  const bool sws = a.colour == CB_FMT_NV12_SWS;
  int next_out = 0;
  // vertical taps of the output rows unit `uv` completes -> shared memory (global loads off the FMA loop's critical path)
  auto stage_taps = [&](int uv) {
    const int last = sUL[uv], nrow = last - next_out;
    if (nrow > 0 && nrow <= kVRows && a.ty <= kVTaps) {
      for (int i = tid; i < nrow * a.ty; i += kTcThreads) {
        const int rr = i / a.ty, k = i - rr * a.ty;
        sW[rr * kVTaps + k] = a.wy[(size_t)(next_out + rr) * a.ty + k];
      }
      if (tid < nrow) sY[2 * tid] = (a.ymin[next_out + tid] - a.y_begin) & (kRingRows - 1), sY[2 * tid + 1] = a.ysize[next_out + tid];
    }
  };
  // vertical pass for the output rows completed by unit `uv` (ATen order: first product, then FMAs), round half even.  It runs while
  // the NEXT unit's MMAs are in flight (their issue-to-commit latency, ~2 k cycles of dependent accumulation, used to be a sleep).
  auto vertical = [&](int uv) {
    const int u = uv;
    (void)u;

    const int last = sUL[u];
    if ((ncols & 3) == 0 && (a.res & 3) == 0 && last - next_out <= kVRows && a.ty <= kVTaps) {
      // four columns per thread: one 16-byte ring read feeds four FMAs, taps from shared memory, one 4-byte store
      const int q = ncols >> 2, items = (last - next_out) * 3 * q;
      for (int i = tid; i < items; i += kTcThreads) {
        const int xq = i % q, t = i / q, yr = t / 3, ch = t - 3 * yr, y = next_out + yr;
        const int nt = sY[2 * yr + 1];
        const float* w = sW + yr * kVTaps;
        const float* col = ring + ch * kNC + 4 * xq;
        int rr = sY[2 * yr];
        float4 v = *reinterpret_cast<const float4*>(col + rr * kRingStride);
        float w0 = w[0];
        float a0 = v.x * w0, a1 = v.y * w0, a2 = v.z * w0, a3 = v.w * w0;
        for (int k = 1; k < nt; ++k) {
          rr = (rr + 1) & (kRingRows - 1);
          v = *reinterpret_cast<const float4*>(col + rr * kRingStride);
          w0 = w[k];
          a0 = fmaf(v.x, w0, a0), a1 = fmaf(v.y, w0, a1), a2 = fmaf(v.z, w0, a2), a3 = fmaf(v.w, w0, a3);
        }
        const uint32_t packed = (uint32_t)min(max(__float2int_rn(a0), 0), 255) | ((uint32_t)min(max(__float2int_rn(a1), 0), 255) << 8) |
                                ((uint32_t)min(max(__float2int_rn(a2), 0), 255) << 16) | ((uint32_t)min(max(__float2int_rn(a3), 0), 255) << 24);
        *reinterpret_cast<uint32_t*>(a.out + (((size_t)frame * 3 + ch) * a.res + y) * a.res + x0 + 4 * xq) = packed;
      }
    } else {
      const int items = (last - next_out) * 3 * ncols;
      for (int i = tid; i < items; i += kTcThreads) {
        const int x = i % ncols, t = i / ncols, yr = t / 3, ch = t - 3 * yr, y = next_out + yr;
        const int y0 = a.ymin[y] - a.y_begin, nt = a.ysize[y];
        const float* w = a.wy + (size_t)y * a.ty;
        float acc = ring[(y0 & (kRingRows - 1)) * kRingStride + ch * kNC + x] * w[0];
        for (int k = 1; k < nt; ++k) acc = fmaf(ring[((y0 + k) & (kRingRows - 1)) * kRingStride + ch * kNC + x], w[k], acc);
        a.out[(((size_t)frame * 3 + ch) * a.res + y) * a.res + x0 + x] = (uint8_t)min(max(__float2int_rn(acc), 0), 255);
      }
    }
    next_out = last;
  };
  for (int u = 0; u < a.n_units; ++u) {
    if (u > 0) stage_taps(u - 1);  // for the vertical pass of the previous unit, which runs below while this unit's MMAs execute
    mbar_wait_parked(raw_full, u & 1, kWaitNs);
    // ---- colour conversion straight into the A operand: a thread owns 2 rows x 4 pixels (two chroma samples)
    {
      const uint8_t* ry = sRaw;
      const uint8_t* ruv = sRaw + ru * kw;
      for (int rp = rp0, xg = xg0; rp < (ru >> 1);) {
        const int x = xg << 2, r = rp << 1;
        const uint32_t yw[2] = {*reinterpret_cast<const uint32_t*>(ry + r * kw + x), *reinterpret_cast<const uint32_t*>(ry + (r + 1) * kw + x)};
        const uint32_t uv4 = *reinterpret_cast<const uint32_t*>(ruv + rp * kw + x);
        int px[2][4][3];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int U = (int)((uv4 >> (16 * h)) & 0xff), V = (int)((uv4 >> (16 * h + 8)) & 0xff);
          int cr, cg, cb_;
          if (sws) {
            const int uu = (U << 3) - 1024, vv = (V << 3) - 1024;
            cr = (vv * 13075) >> 16, cg = ((uu * -3209) >> 16) + ((vv * -6660) >> 16), cb_ = (uu * 16525) >> 16;
          } else {
            const int uo = U - 128, vo = V - 128;
            cr = 1673527 * vo, cg = -852492 * vo - 409993 * uo, cb_ = 2116026 * uo;
          }
#pragma unroll
          for (int rr = 0; rr < 2; ++rr) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const int Y = (int)((yw[rr] >> (16 * h + 8 * k)) & 0xff);
              int* o = px[rr][2 * h + k];
              if (sws) {
                const int yv = (((Y << 3) - 128) * 9539) >> 16;
                o[0] = __viaddmin_s32_relu(yv, cr, 255), o[1] = __viaddmin_s32_relu(yv, cg, 255), o[2] = __viaddmin_s32_relu(yv, cb_, 255);
              } else {
                constexpr int kMax = (256 << 20) - 1;
                const int yv = max(Y - 16, 0) * 1220542 + (1 << 19);
                o[0] = __viaddmin_s32_relu(yv, cr, kMax) >> 20, o[1] = __viaddmin_s32_relu(yv, cg, kMax) >> 20, o[2] = __viaddmin_s32_relu(yv, cb_, kMax) >> 20;
              }
            }
          }
        }
        // operand address of (m, k): chunk of 64 k-elements, 8-row group, row, 16-byte unit XOR row (128-byte swizzle), element.
        // ru is a multiple of 8, so the plane offset ch * ru only moves whole 8-row groups: one row offset serves the three planes.
        const int koff = ((x >> 6) << 14) + ((x & 7) << 1), unit = (x & 63) >> 3;
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const int mr = r + rr;
          uint8_t* row = sA + koff + ((mr >> 3) << 10) + ((mr & 7) << 7) + ((unit ^ (mr & 7)) << 4);
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            uint2 v;
            v.x = pack_u8_pair_f16(px[rr][0][ch], px[rr][1][ch]);
            v.y = pack_u8_pair_f16(px[rr][2][ch], px[rr][3][ch]);
            *reinterpret_cast<uint2*>(row + ch * plane_bytes) = v;
          }
        }
        xg += dxg, rp += drp;
        if (xg >= q4) xg -= q4, ++rp;
      }
    }
    fence_proxy_async();  // generic-proxy writes of the operand -> visible to the tensor core (async proxy)
    __syncthreads();
    if (tid == 0) {
      if (u + 1 < a.n_units) issue(u + 1);  // the raw window is free again
      tc_fence_after();
      // Four independent accumulators - (N-tile, weight term) - interleaved k-step by k-step: a chain of accumulations into ONE
      // TMEM tile serialises on the MMA pipeline latency (measured: 28 back-to-back dependent MMAs cost ~3.5 k cycles, 44 % of the
      // warp samples slept on the commit barrier); hi and lo partial sums are added in the epilogue instead.
      // One MMA per (N-tile, k-step): a UMMA with M = 128 streams its 128 A rows from shared memory in ~128 cycles whatever N is
      // (measured: 28 N=16 MMAs per unit cost ~3.5 k cycles, 44 % of the warp samples slept on the commit), so the hi and lo weight
      // terms ride in the SAME instruction as N = 32 - two accumulators per tile (TMEM columns 0..15 | 16..31), added in the epilogue.
      for (int kk = 0; kk < nkm; ++kk) {
        const uint64_t kb_off = (uint64_t)(((kk >> 2) << 8) + ((kk & 3) << 1));  // chunk of 64 k: 32 rows x 128 B = 4096 B, k-step: 32 B
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (kk >= (j ? nk1 : nk0)) continue;
          const int qa = (j ? k01 : k00) + kk;
          const uint64_t da = desc_a0 + (uint64_t)(((qa >> 2) << 10) + ((qa & 3) << 1));  // chunk: 16384 B
          umma_f16(tmem + (uint32_t)(j * 32), da, desc_b0 + (uint64_t)(j * b_tile16) + kb_off, idesc, kk != 0);
        }
      }
      umma_commit(mma_done);
    }
    if (u > 0) vertical(u - 1);
    __syncthreads();  // the epilogue below overwrites ring rows the vertical pass was still reading
    mbar_wait_parked(mma_done, u & 1, kWaitNs);
    tc_fence_after();
    // ---- epilogue: the filtered rows of this unit -> ring (warp = lane quarter x N-tile)
    if (warp < 8) {
      const int lq = warp & 3, half = warp >> 2;
      uint32_t v[16], vl[16];
      tmem_ld_32x32b_x16(tmem + ((uint32_t)(lq * 32) << 16) + (uint32_t)(half * 32), v);        // hi-weight partial sums
      tmem_ld_32x32b_x16(tmem + ((uint32_t)(lq * 32) << 16) + (uint32_t)(half * 32 + 16), vl);  // lo-weight partial sums
      tmem_ld_wait();
      const int l = lq * 32 + lane;
      if (l < 3 * ru) {
        const int ch = l / ru, r = l - ch * ru;
        float4* dst = reinterpret_cast<float4*>(ring + ((u * ru + r) & (kRingRows - 1)) * kRingStride + ch * kNC + half * 16);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          dst[q] = make_float4(__uint_as_float(v[4 * q]) + __uint_as_float(vl[4 * q]), __uint_as_float(v[4 * q + 1]) + __uint_as_float(vl[4 * q + 1]),
                               __uint_as_float(v[4 * q + 2]) + __uint_as_float(vl[4 * q + 2]), __uint_as_float(v[4 * q + 3]) + __uint_as_float(vl[4 * q + 3]));
      }
    }
    tc_fence_before();
    __syncthreads();
  }
  stage_taps(a.n_units - 1);
  __syncthreads();
  vertical(a.n_units - 1);
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 64);
}

// u8 [n][3][res][res] -> normalised output: typed NCHW (mode 1) or zero-padded patch rows [n][(res/p)^2][k_pad] (mode 2)
struct PackArgs {
  const uint8_t* src;
  const float* lut;  // [3][256]
  int n, res, mode, dtype, patch, k_pad;
  void* out;
};

__device__ __forceinline__ void store_out(void* out, size_t idx, float v, int dtype) {
  if (dtype == CB_DT_F16) reinterpret_cast<__half*>(out)[idx] = __float2half_rn(v);
  else if (dtype == CB_DT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[idx] = __float2bfloat16_rn(v);
  else reinterpret_cast<float*>(out)[idx] = v;
}

__global__ void normalize_pack_kernel(const PackArgs a) {  // mode 1: typed NCHW, one element per thread (parity-test output)
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t plane = (size_t)a.res * a.res;
  if (i >= 3 * plane * a.n) return;
  const int ch = (int)((i / plane) % 3);
  store_out(a.out, i, a.lut[ch * 256 + a.src[i]], a.dtype);
}

// mode 2: one CTA per (frame, patch row): the k -> (plane, y, x) map of a patch is built once in shared memory, then every thread
// emits 8 consecutive elements of a zero-padded patch row per iteration as one 16-byte store.
__global__ void __launch_bounds__(256) pack_patches_kernel(const PackArgs a) {
  extern __shared__ int koff[];  // [k_pad]: (plane << 24) | offset inside the patch origin's plane, -1 = padding
  const int g = a.res / a.patch, pp = a.patch * a.patch;
  for (int k = threadIdx.x; k < a.k_pad; k += blockDim.x) {
    int v = -1;
    if (k < 3 * pp) {
      const int ch = k / pp, yy = (k - ch * pp) / a.patch, xx = k - ch * pp - yy * a.patch;
      v = (ch << 24) | (yy * a.res + xx);
    }
    koff[k] = v;
  }
  __syncthreads();
  const int py = blockIdx.x, f = blockIdx.y;
  const size_t plane = (size_t)a.res * a.res;
  const uint8_t* img = a.src + (size_t)f * 3 * plane + (size_t)py * a.patch * a.res;
  const int k8 = a.k_pad >> 3;
  const bool bf = a.dtype == CB_DT_BF16;
  for (int i = threadIdx.x; i < g * k8; i += blockDim.x) {
    const int px = i / k8, kk = (i - px * k8) << 3;
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float v[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int o = koff[kk + 2 * e + h];
        const int ch = o >> 24;
        v[h] = o < 0 ? 0.f : a.lut[ch * 256 + img[(size_t)ch * plane + (o & 0xFFFFFF) + px * a.patch]];
      }
      if (bf) {
        __nv_bfloat162 b = __floats2bfloat162_rn(v[0], v[1]);
        w[e] = *reinterpret_cast<uint32_t*>(&b);
      } else {
        __half2 hh = __floats2half2_rn(v[0], v[1]);
        w[e] = *reinterpret_cast<uint32_t*>(&hh);
      }
    }
    uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(a.out) + (((size_t)f * g + py) * g + px) * a.k_pad + kk);
    *dst = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ------------------------------------------------------------------------------------------------ host
namespace {

struct TcPlan {  // per (source size, taps): slab windows + pre-swizzled weight tiles on the device
  int n_slabs = 0, kw = 0, kb = 0, ru = 0, n_units = 0, y_begin = 0, nc = kNC;
  int *d_x_lo = nullptr, *d_k0 = nullptr, *d_nk = nullptr, *d_unit_last = nullptr;
  uint8_t* d_w = nullptr;
  bool ok = false;
};

uint16_t f32_to_f16_bits(float f) {
  __half h = __float2half_rn(f);
  uint16_t b;
  memcpy(&b, &h, 2);
  return b;
}
float f16_bits_to_f32(uint16_t b) {
  __half h;
  memcpy(&h, &b, 2);
  return __half2float(h);
}

}  // namespace

static std::map<std::tuple<const TapTable*, const TapTable*>, TcPlan>& plans(cb_ctx* ctx) {
  static std::map<cb_ctx*, std::map<std::tuple<const TapTable*, const TapTable*>, TcPlan>> all;  // tap tables live as long as the ctx
  return all[ctx];
}

static const TcPlan* get_plan(cb_ctx* ctx, const TapTable* tx, const TapTable* ty, int res) {
  auto key = std::make_tuple(tx, ty);
  auto& cache = plans(ctx);
  auto it = cache.find(key);
  if (it != cache.end()) return &it->second;
  TcPlan p;
  std::vector<int> x_lo, k0, nk;
  int kw = 0, kbmax = 0;
  for (int nc : {kNC, 16}) {  // 32 columns per slab unless their source window exceeds one TMA box (4K -> 224: 9.6x downscale)
    p.nc = nc, p.n_slabs = (res + nc - 1) / nc;
    x_lo.assign(p.n_slabs, 0), k0.assign(p.n_slabs * 2, 0), nk.assign(p.n_slabs * 2, 0);
    kw = 0, kbmax = 0;
    for (int s = 0; s < p.n_slabs; ++s) {
      const int c0 = s * nc, c1 = std::min(res, c0 + nc);
      x_lo[s] = tx->h_min[c0] & ~15;
      int hi = 0;
      for (int c = c0; c < c1; ++c) hi = std::max(hi, tx->h_min[c] + tx->h_size[c]);
      kw = std::max(kw, hi - x_lo[s]);
      for (int j = 0; j < 2; ++j) {
        const int t0 = c0 + 16 * j, t1 = std::min(c1, t0 + 16);
        if (t0 >= t1) continue;
        const int first = (tx->h_min[t0] - x_lo[s]) / 16;
        int end = 0;
        for (int c = t0; c < t1; ++c) end = std::max(end, tx->h_min[c] + tx->h_size[c] - x_lo[s]);
        k0[s * 2 + j] = first, nk[s * 2 + j] = (end - first * 16 + 15) / 16;
        kbmax = std::max(kbmax, nk[s * 2 + j] * 16);
      }
    }
    if (kw <= 256) break;
  }
  p.kw = (kw + 63) & ~63, p.kb = (kbmax + 63) & ~63;
  p.ru = std::min(40, kRingRows - ty->max_taps + 1) & ~7;  // multiple of 8: a colour plane is a whole number of 8-row operand groups
  p.y_begin = ty->src_begin & ~1;
  p.n_units = p.ru > 0 ? (ty->src_end - p.y_begin + p.ru - 1) / p.ru : 0;
  const int b_tile = (p.kb / 64) * 4096;
  const size_t smem = 1024 + (size_t)p.kw * 256 + 2 * (size_t)b_tile + ((((size_t)(p.ru + p.ru / 2) * p.kw) + 127) & ~(size_t)127) + (kRingRows * kRingStride + kVRows * kVTaps + 2 * kVRows + kMaxUnits) * 4 + 64;
  p.ok = p.ru >= 16 && p.kw <= 256 && p.n_units <= kMaxUnits && smem <= 227 * 1024;  // TMA box <= 256 columns
  if (p.ok) {
    std::vector<uint16_t> w((size_t)p.n_slabs * 2 * b_tile / 2, 0);
    for (int s = 0; s < p.n_slabs; ++s)
      for (int j = 0; j < 2; ++j)
        for (int nrow = 0; nrow < 16; ++nrow) {
          const int c = s * p.nc + 16 * j + nrow;
          if (c >= res || nk[s * 2 + j] == 0) continue;
          for (int k = 0; k < nk[s * 2 + j] * 16; ++k) {
            const int t = x_lo[s] + k0[s * 2 + j] * 16 + k - tx->h_min[c];
            if (t < 0 || t >= tx->h_size[c]) continue;
            const float wv = tx->h_w[(size_t)c * tx->max_taps + t];
            const uint16_t hb = f32_to_f16_bits(wv), lb = f32_to_f16_bits(wv - f16_bits_to_f32(hb));
            for (int hl = 0; hl < 2; ++hl) {
              const int nr = hl * 16 + nrow;  // row of the 32-row B tile
              const size_t off = (size_t)(k >> 6) * 4096 + (size_t)(nr >> 3) * 1024 + (size_t)(nr & 7) * 128 + (size_t)((((k & 63) >> 3) ^ (nr & 7)) << 4) + (size_t)((k & 7) << 1);
              w[((size_t)(s * 2 + j) * b_tile + off) / 2] = hl ? lb : hb;
            }
          }
        }
    std::vector<int> unit_last(p.n_units);
    for (int u = 0, last = 0; u < p.n_units; ++u) {
      const int rows_end = p.y_begin + (u + 1) * p.ru;
      while (last < res && ty->h_min[last] + ty->h_size[last] <= rows_end) ++last;
      unit_last[u] = last;
    }
    if (p.n_units > 0) unit_last[p.n_units - 1] = res;
    const size_t ib = p.n_slabs * sizeof(int);
    if (cudaMalloc(&p.d_unit_last, p.n_units * sizeof(int)) != cudaSuccess) return nullptr;
    cudaMemcpy(p.d_unit_last, unit_last.data(), p.n_units * sizeof(int), cudaMemcpyHostToDevice);
    if (cudaMalloc(&p.d_x_lo, ib) != cudaSuccess || cudaMalloc(&p.d_k0, 2 * ib) != cudaSuccess || cudaMalloc(&p.d_nk, 2 * ib) != cudaSuccess ||
        cudaMalloc(&p.d_w, w.size() * 2) != cudaSuccess)
      return nullptr;
    cudaMemcpy(p.d_x_lo, x_lo.data(), ib, cudaMemcpyHostToDevice);
    cudaMemcpy(p.d_k0, k0.data(), 2 * ib, cudaMemcpyHostToDevice);
    cudaMemcpy(p.d_nk, nk.data(), 2 * ib, cudaMemcpyHostToDevice);
    cudaMemcpy(p.d_w, w.data(), w.size() * 2, cudaMemcpyHostToDevice);
  }
  return &(cache[key] = p);
}

void release_tc_plans(cb_ctx* ctx) {
  for (auto& kv : plans(ctx)) {
    cudaFree(kv.second.d_x_lo), cudaFree(kv.second.d_k0), cudaFree(kv.second.d_nk), cudaFree(kv.second.d_w), cudaFree(kv.second.d_unit_last);
  }
  plans(ctx).clear();
}

// Returns CB_OK when the tensor-pipe kernel ran; 1 when this configuration is not served by it (the caller falls back to v2).
int run_clip_preprocess_tc(cb_ctx* ctx, const cb_surface_pool* pool, const int* d_slots, int n, int max_slot, int res, int out_mode, int patch, int k_pad,
                           int dtype, const TapTable* tx, const TapTable* ty, void* out, cudaStream_t stream) {
  if (pool->format != CB_FMT_NV12 && pool->format != CB_FMT_NV12_SWS) return 1;
  if (ty->max_taps > 40) return 1;
  const TcPlan* p = get_plan(ctx, tx, ty, res);
  if (!p) return fail(ctx, CB_ERR_CUDA, "preprocess plan allocation failed");
  if (!p->ok) return 1;
  uint8_t* u8 = (uint8_t*)out;
  const size_t u8_bytes = (size_t)n * 3 * res * res;
  if (out_mode != 0) {
    if (ctx->tmp_u8_cap < u8_bytes) {
      if (ctx->d_tmp_u8) {
        CB_CUDA(ctx, cudaStreamSynchronize(stream));
        cudaFree(ctx->d_tmp_u8);
      }
      ctx->tmp_u8_cap = std::max(u8_bytes, (size_t)64 << 20);
      CB_CUDA(ctx, cudaMalloc(&ctx->d_tmp_u8, ctx->tmp_u8_cap));
    }
    u8 = ctx->d_tmp_u8;
  }
  const int W = pool->width, H = pool->height;
  CUtensorMap map_y, map_uv;
  uint64_t dims[3] = {(uint64_t)W, (uint64_t)H, (uint64_t)max_slot + 1};
  uint64_t strides[2] = {(uint64_t)pool->pitch, (uint64_t)pool->slot_stride};
  uint32_t box[3] = {(uint32_t)p->kw, (uint32_t)p->ru, 1};
  int rc = make_tensor_map(ctx, &map_y, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, pool->base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE);
  if (rc) return rc;
  uint64_t dims_uv[3] = {(uint64_t)W, (uint64_t)(H / 2), (uint64_t)max_slot + 1};
  uint32_t box_uv[3] = {(uint32_t)p->kw, (uint32_t)(p->ru / 2), 1};
  rc = make_tensor_map(ctx, &map_uv, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (const uint8_t*)pool->base + (size_t)pool->luma_rows * pool->pitch, dims_uv,
                       strides, box_uv, CU_TENSOR_MAP_SWIZZLE_NONE);
  if (rc) return rc;
  TcArgs a{};
  a.nc = p->nc;
  a.slots = d_slots, a.n = n, a.res = res, a.ru = p->ru, a.n_units = p->n_units, a.y_begin = p->y_begin, a.kw = p->kw, a.kb = p->kb;
  a.colour = pool->format;
  a.x_lo = p->d_x_lo, a.tile_k0 = p->d_k0, a.tile_nk = p->d_nk, a.wtiles = p->d_w;
  a.ymin = ty->d_min, a.ysize = ty->d_size, a.unit_last = p->d_unit_last, a.wy = ty->d_w, a.ty = ty->max_taps, a.out = u8;
  const int b_tile = (p->kb / 64) * 4096;
  const size_t smem = 1024 + (size_t)p->kw * 256 + 2 * (size_t)b_tile + ((((size_t)(p->ru + p->ru / 2) * p->kw) + 127) & ~(size_t)127) + (kRingRows * kRingStride + kVRows * kVTaps + 2 * kVRows + kMaxUnits) * 4 + 64;
  CB_CUDA(ctx, cudaFuncSetAttribute(clip_preprocess_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mark_launch(ctx, CB_PROF_PREPROCESS, stream);
  clip_preprocess_tc_kernel<<<dim3(p->n_slabs, n), kTcThreads, smem, stream>>>(map_y, map_uv, a);
  CB_CUDA(ctx, cudaGetLastError());
  if (out_mode != 0) {
    PackArgs q{};
    q.src = u8, q.lut = ctx->d_norm_lut, q.n = n, q.res = res, q.mode = out_mode, q.dtype = dtype, q.patch = patch, q.k_pad = k_pad, q.out = out;
    mark_launch(ctx, CB_PROF_PREPROCESS, stream);
    if (out_mode == 1) {
      const size_t total = (size_t)n * 3 * res * res;
      normalize_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(q);
    } else {
      const int g = res / patch;
      pack_patches_kernel<<<dim3(g, n), 256, k_pad * sizeof(int), stream>>>(q);
    }
    CB_CUDA(ctx, cudaGetLastError());
  }
  return CB_OK;
}

}  // namespace cb
