// Non-GEMM kernels of the image tower (sm_100a): LayerNorm, token assembly, attention, pooled tail.
//   layernorm_kernel       fp32 residual stream -> fp16 normalised activations (HBM-bound: 6 B/element)
//   assemble_kernel        patch-embed output + [CLS] + position embedding (+ CLIP pre_layrnorm) -> residual stream
//   attention_kernel       softmax(Q K^T / sqrt(d)) V per (image, head); K/V resident in shared memory,
//                          mma.sync m16n8k16 with fp32 online softmax (4 % of the tower's FLOPs; the dense
//                          Linear layers are the tcgen05 kernel in gemm.cu)
//   clip_tail_kernel       post_layernorm(CLS) -> visual_projection -> L2 normalise -> aesthetic affine head
#include <cuda_fp16.h>

#include <type_traits>

#include "common.h"
#include "ptx.cuh"

namespace cb {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------------------------------- LayerNorm
// One warp per row; D <= 32*4*kMaxChunks.  Two-pass statistics in registers (mean, then centred variance).
constexpr int kLnMaxChunks = 12;  // D <= 1536

// CHUNKS > 0: the row length is the compile-time constant 128 * CHUNKS (the towers' widths get their own instantiation: the
// register array is exactly the row, 46 instead of 78 registers at 1024, so more rows are in flight per SM); CHUNKS == 0: any
// multiple of 128 up to 128 * kLnMaxChunks.  Same operations in the same order either way.
template <bool OUT_F16, int CHUNKS = 0>
__device__ __forceinline__ void ln_row(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                       void* __restrict__ y, int d, float eps, int lane, const float* __restrict__ add = nullptr) {
  constexpr int kMax = CHUNKS > 0 ? CHUNKS : kLnMaxChunks;
  float4 v[kMax];
  const int chunks = CHUNKS > 0 ? CHUNKS : d >> 7;  // 128 floats per warp pass
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kMax; ++i)
    if (i < chunks) {
      v[i] = ((const float4*)x)[lane + 32 * i];
      if (add) {
        const float4 a = __ldg((const float4*)add + lane + 32 * i);
        v[i].x += a.x, v[i].y += a.y, v[i].z += a.z, v[i].w += a.w;
      }
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  const float mean = warp_sum(s) / (float)d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < kMax; ++i)
    if (i < chunks) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, e = v[i].w - mean;
      q += (a * a + b * b) + (c * c + e * e);
    }
  const float rstd = rsqrtf(warp_sum(q) / (float)d + eps);
#pragma unroll
  for (int i = 0; i < kMax; ++i)
    if (i < chunks) {
      const float4 g = __ldg((const float4*)gamma + lane + 32 * i), b = __ldg((const float4*)beta + lane + 32 * i);
      const float o0 = (v[i].x - mean) * rstd * g.x + b.x, o1 = (v[i].y - mean) * rstd * g.y + b.y;
      const float o2 = (v[i].z - mean) * rstd * g.z + b.z, o3 = (v[i].w - mean) * rstd * g.w + b.w;
      if (OUT_F16) {
        const __half2 h0 = __floats2half2_rn(o0, o1), h1 = __floats2half2_rn(o2, o3);
        uint2 o;
        o.x = *(const uint32_t*)&h0, o.y = *(const uint32_t*)&h1;
        ((uint2*)y)[lane + 32 * i] = o;
      } else {
        ((float4*)y)[lane + 32 * i] = make_float4(o0, o1, o2, o3);
      }
    }
}

template <int CHUNKS, int MINB>
__global__ void __launch_bounds__(256, MINB) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, __half* __restrict__ y, int rows, int d, float eps) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  ln_row<true, CHUNKS>(x + (size_t)row * d, gamma, beta, y + (size_t)row * d, d, eps, threadIdx.x & 31);
}

// ------------------------------------------------------------------------------- token assembly
// CLIP  : h[n][0] = LN(cls + pos[0]); h[n][1+i] = LN(patch[n][i] + pos[1+i])     (pre_layrnorm)
// SigLIP: h[n][i] = patch[n][i] + pos[i]                                          (patch bias is in the GEMM)
__global__ void __launch_bounds__(256) assemble_kernel(const float* __restrict__ patch, const float* __restrict__ cls,
                                                       const float* __restrict__ pos, const float* __restrict__ gamma,
                                                       const float* __restrict__ beta, float* __restrict__ h, int n, int tokens, int grid2,
                                                       int d, float eps) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n * tokens) return;
  const int img = row / tokens, t = row - img * tokens;
  const bool has_cls = tokens != grid2;
  const float* src = (has_cls && t == 0) ? cls : patch + ((size_t)img * grid2 + (t - (has_cls ? 1 : 0))) * d;
  const float* p = pos + (size_t)t * d;
  float* dst = h + (size_t)row * d;
  if (gamma) {
    ln_row<false>(src, gamma, beta, dst, d, eps, lane, p);
  } else {
    for (int i = lane; i < (d >> 2); i += 32) {
      float4 a = ((const float4*)src)[i];
      const float4 b = __ldg((const float4*)p + i);
      a.x += b.x, a.y += b.y, a.z += b.z, a.w += b.w;
      ((float4*)dst)[i] = a;
    }
  }
}

// ------------------------------------------------------------------------------------ attention
__device__ __forceinline__ void mma_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t* r, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t* r, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ float fast_exp2(float x) {  // MUFU.EX2, inputs <= 0 here; flush-to-zero is what softmax wants
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *(const uint32_t*)&h;
}

constexpr int kAttnWarps = 9;
constexpr int kAttnThreads = kAttnWarps * 32;

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// HD: head dim padded to a multiple of 16 (64 -> 64, 72 -> 80).  Each warp owns 16-query tiles; K and V live in shared
// memory (cp.async fill) and are consumed with ldmatrix / mma.sync.m16n8k16 in 32-key chunks whose shape is a compile-time
// constant (no convergence barriers around the .sync instructions); MMAs are issued over independent accumulators back to
// back; softmax is online in fp32 with LAZY rescaling (O and the row sums are rescaled only when a row of the warp sees a new
// maximum - rare after the first chunks).
//   STREAM = false: one CTA per (image, head), all keys resident, warps loop over the query tiles      (T = 50, 257, ...)
//   STREAM = true : grid.y splits the query tiles (one per warp), keys stream through shared memory in
//                   blocks of kStreamKeys, the softmax state stays in registers across blocks             (T = 729, ...)
constexpr int kStreamKeys = 256;

template <int HD, bool STREAM>
__global__ void __launch_bounds__(kAttnThreads, 2) attention_kernel(const __half* __restrict__ qkv, __half* __restrict__ out, int tokens,
                                                                     int heads, int head_dim, float scale_log2e) {
  constexpr int PITCH = HD + 8;  // halves; 16-byte row skew keeps ldmatrix conflict-free
  constexpr int KS = HD / 16;    // k-steps over the head dimension
  extern __shared__ __align__(16) uint8_t smem_attn[];
  const int t_pad = (tokens + 15) & ~15;
  const int blk = STREAM ? kStreamKeys : t_pad;  // keys resident at a time
  __half* sK = (__half*)smem_attn;
  __half* sV = sK + (size_t)blk * PITCH;
  const int img = blockIdx.x / heads, head = blockIdx.x - img * heads;
  const int hidden = heads * head_dim;
  const size_t row_stride = (size_t)3 * hidden;
  const __half* base = qkv + (size_t)img * tokens * row_stride + (size_t)head * head_dim;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;

  // keys [k0, k0 + blk) (zero padded in both directions) -> shared memory, all copies in flight at once
  constexpr int VEC = HD / 8;
  const int vec_valid = head_dim / 8;  // head_dim % 8 == 0 is checked on the host
  auto load_block = [&](int k0) {
    const int rows = min(blk, t_pad - k0);
    for (int i = threadIdx.x; i < rows * VEC; i += kAttnThreads) {
      const int r = i / VEC, c = i - r * VEC;
      __half* dk = sK + (size_t)r * PITCH + c * 8;
      __half* dv = sV + (size_t)r * PITCH + c * 8;
      if (k0 + r < tokens && c < vec_valid) {
        const __half* p = base + (size_t)(k0 + r) * row_stride + c * 8;
        cp_async_16(dk, p + hidden);
        cp_async_16(dv, p + 2 * hidden);
      } else {
        *(uint4*)dk = make_uint4(0, 0, 0, 0);
        *(uint4*)dv = make_uint4(0, 0, 0, 0);
      }
    }
  };
  if (!STREAM) load_block(0);

  // per-lane shared-memory offsets of the ldmatrix rows (bytes)
  const uint32_t k_lane = smem_u32(sK) + (uint32_t)(((lane & 7) * PITCH + (lane >> 3) * 8) * 2);
  const uint32_t k_lane_tail = smem_u32(sK) + (uint32_t)(((lane & 7) * PITCH + (HD - 16) + ((lane >> 3) & 1) * 8) * 2);
  const uint32_t v_lane = smem_u32(sV) + (uint32_t)(((((lane >> 3) & 1) * 8 + (lane & 7)) * PITCH + (lane >> 4) * 8) * 2);
  using Full = std::integral_constant<int, 4>;
  using Tail = std::integral_constant<int, 2>;

  const int q_tiles = t_pad >> 4;
  const int qt_first = STREAM ? (int)blockIdx.y * kAttnWarps + warp : warp;
  const int qt_step = STREAM ? q_tiles : kAttnWarps;  // STREAM: exactly one tile per warp (maybe none)
  bool first = true;
  for (int qt = qt_first; qt < q_tiles || (STREAM && first); qt += qt_step) {
    const bool active = qt < q_tiles;  // STREAM: a warp without a tile still takes part in the block barriers
    // Q fragments straight from global memory (rows clamped; padded columns read as zero)
    uint32_t qa[KS][4];
    const int qrow = active ? qt * 16 : 0;
    const int r0 = min(qrow + g, tokens - 1), r1 = min(qrow + g + 8, tokens - 1);
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      const int c0 = ks * 16 + t4 * 2, c1 = c0 + 8;
      qa[ks][0] = c0 < head_dim ? __ldg((const uint32_t*)(base + (size_t)r0 * row_stride + c0)) : 0u;
      qa[ks][1] = c0 < head_dim ? __ldg((const uint32_t*)(base + (size_t)r1 * row_stride + c0)) : 0u;
      qa[ks][2] = c1 < head_dim ? __ldg((const uint32_t*)(base + (size_t)r0 * row_stride + c1)) : 0u;
      qa[ks][3] = c1 < head_dim ? __ldg((const uint32_t*)(base + (size_t)r1 * row_stride + c1)) : 0u;
    }
    if (!STREAM && qt + kAttnWarps < q_tiles) {  // pull the next tile's Q rows towards L2 while this tile computes
      const int rn = min((qt + kAttnWarps) * 16 + (lane & 15), tokens - 1);
      prefetch_l2(base + (size_t)rn * row_stride);
    }
    if (!STREAM && first) {  // the Q loads above overlap the K/V fill
      cp_async_wait_all();
      __syncthreads();
    }
    first = false;

    // S = Q K^T for NKT 8-key tiles; `srow` = row of the chunk's first key inside the resident block
    auto qk_chunk = [&](int srow, auto nkt_c, float (&sc)[4][4]) {
      constexpr int NKT = decltype(nkt_c)::value;
#pragma unroll
      for (int i = 0; i < 4; ++i) sc[i][0] = sc[i][1] = sc[i][2] = sc[i][3] = 0.f;
      const uint32_t kbase = k_lane + (uint32_t)(srow * PITCH * 2);
#pragma unroll
      for (int kp = 0; kp < HD / 32; ++kp) {  // two k-steps per ldmatrix.x4
        uint32_t kb[NKT][4];
#pragma unroll
        for (int i = 0; i < NKT; ++i) ldmatrix_x4(kb[i], kbase + (uint32_t)((i * 8 * PITCH + kp * 32) * 2));
#pragma unroll
        for (int i = 0; i < NKT; ++i) mma_16816(sc[i], qa[2 * kp], kb[i][0], kb[i][1]);
#pragma unroll
        for (int i = 0; i < NKT; ++i) mma_16816(sc[i], qa[2 * kp + 1], kb[i][2], kb[i][3]);
      }
      if (HD % 32) {  // odd number of k-steps (HD = 80): last 16 columns
        uint32_t kb[NKT][4];
#pragma unroll
        for (int i = 0; i < NKT; ++i) ldmatrix_x4(kb[i], k_lane_tail + (uint32_t)((srow + i * 8) * PITCH * 2));
#pragma unroll
        for (int i = 0; i < NKT; ++i) mma_16816(sc[i], qa[KS - 1], kb[i][0], kb[i][1]);
      }
    };

    float m0 = -INFINITY, m1 = -INFINITY;  // running maxima of rows g and g+8 (quad-uniform)
    float o[HD / 8][4];
#pragma unroll
    for (int d = 0; d < HD / 8; ++d) o[d][0] = o[d][1] = o[d][2] = o[d][3] = 0.f;
    float l0 = 0.f, l1 = 0.f;
    auto pv_chunk = [&](int kc, int srow, auto nkt_c) {  // kc: absolute key index of the chunk (masking)
      constexpr int NKT = decltype(nkt_c)::value;
      float sc[4][4];
      qk_chunk(srow, nkt_c, sc);
      if (kc + NKT * 8 > tokens) {  // padded keys only live in the last chunk(s)
#pragma unroll
        for (int i = 0; i < NKT; ++i) {
          const int key = kc + i * 8 + t4 * 2;
          if (key >= tokens) sc[i][0] = sc[i][2] = -INFINITY;
          if (key + 1 >= tokens) sc[i][1] = sc[i][3] = -INFINITY;
        }
      }
      float mx0 = m0, mx1 = m1;
#pragma unroll
      for (int i = 0; i < NKT; ++i) {
        mx0 = fmaxf(mx0, fmaxf(sc[i][0], sc[i][1]));
        mx1 = fmaxf(mx1, fmaxf(sc[i][2], sc[i][3]));
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      if (__any_sync(0xffffffffu, mx0 > m0 || mx1 > m1)) {  // warp-uniform: rescale the accumulators to the new maxima
        const float c0 = fast_exp2((m0 - mx0) * scale_log2e), c1 = fast_exp2((m1 - mx1) * scale_log2e);  // exp2(-inf) = 0 at the start
        m0 = mx0, m1 = mx1;
        l0 *= c0, l1 *= c1;
#pragma unroll
        for (int d = 0; d < HD / 8; ++d) o[d][0] *= c0, o[d][1] *= c0, o[d][2] *= c1, o[d][3] *= c1;
      }
      const float b0 = m0 * scale_log2e, b1 = m1 * scale_log2e;
      uint32_t pa[2][4];  // P as A fragments: k-step j covers key tiles 2j, 2j+1
#pragma unroll
      for (int i = 0; i < NKT; ++i) {  // masked keys: exp2(-inf) = 0
        const float p0 = fast_exp2(fmaf(sc[i][0], scale_log2e, -b0)), p1 = fast_exp2(fmaf(sc[i][1], scale_log2e, -b0));
        const float p2 = fast_exp2(fmaf(sc[i][2], scale_log2e, -b1)), p3 = fast_exp2(fmaf(sc[i][3], scale_log2e, -b1));
        l0 += p0 + p1, l1 += p2 + p3;
        pa[i >> 1][(i & 1) * 2 + 0] = pack_half2(p0, p1);
        pa[i >> 1][(i & 1) * 2 + 1] = pack_half2(p2, p3);
      }
      constexpr int DP = HD / 16;  // pairs of 8-wide dim tiles
#pragma unroll
      for (int j = 0; j < NKT / 2; ++j) {
        uint32_t vb[DP][4];
        const uint32_t vbase = v_lane + (uint32_t)((srow + j * 16) * PITCH * 2);
#pragma unroll
        for (int dp = 0; dp < DP; ++dp) ldmatrix_x4_trans(vb[dp], vbase + (uint32_t)(dp * 32));
#pragma unroll
        for (int dp = 0; dp < DP; ++dp) {
          mma_16816(o[2 * dp], pa[j], vb[dp][0], vb[dp][1]);
          mma_16816(o[2 * dp + 1], pa[j], vb[dp][2], vb[dp][3]);
        }
      }
    };

    for (int k0 = 0; k0 < t_pad; k0 += blk) {  // one iteration when the keys are resident
      if (STREAM) {
        __syncthreads();  // every warp is done with the previous block
        load_block(k0);
        cp_async_wait_all();
        __syncthreads();
      }
      if (active) {
        const int rows = min(blk, t_pad - k0), full_end = rows & ~31;
        for (int r = 0; r < full_end; r += 32) pv_chunk(k0 + r, r, Full{});
        if (full_end < rows) pv_chunk(k0 + full_end, full_end, Tail{});
      }
    }
    if (!active) break;

    // quad-reduce the row sums, normalise, store
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float inv0 = 1.f / l0, inv1 = 1.f / l1;
    const int row0 = qt * 16 + g, row1 = row0 + 8;
    __half* ob = out + (size_t)img * tokens * hidden + (size_t)head * head_dim;
#pragma unroll
    for (int d = 0; d < HD / 8; ++d) {
      const int c = d * 8 + t4 * 2;
      if (c < head_dim) {
        if (row0 < tokens) *(uint32_t*)(ob + (size_t)row0 * hidden + c) = pack_half2(o[d][0] * inv0, o[d][1] * inv0);
        if (row1 < tokens) *(uint32_t*)(ob + (size_t)row1 * hidden + c) = pack_half2(o[d][2] * inv1, o[d][3] * inv1);
      }
    }
  }
  if (!STREAM && first) {  // a warp without a tile (q_tiles < warps) still has to meet the fill barrier
    cp_async_wait_all();
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------- CLIP tail
// One CTA per image: post_layernorm on the CLS row, projection (fp32 weights), L2 normalise, aesthetic affine head.
__global__ void __launch_bounds__(256) clip_tail_kernel(const float* __restrict__ h, size_t img_stride, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, const float* __restrict__ proj, int d, int proj_dim,
                                                        float eps, const float* __restrict__ aes_w, float aes_b, float* __restrict__ emb_out,
                                                        float* __restrict__ feat_out, float* __restrict__ score_out) {
  extern __shared__ float sm_tail[];
  float* pooled = sm_tail;          // [d]
  float* feat = sm_tail + d;        // [out_dim]
  __shared__ float red[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const float* x = h + (size_t)blockIdx.x * img_stride;
  auto block_sum = [&](float v) {
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = (tid < nw) ? red[tid] : 0.f;
    if (warp == 0) {
      t = warp_sum(t);
      if (lane == 0) red[0] = t;
    }
    __syncthreads();
    return red[0];
  };
  float s = 0.f;
  for (int i = tid; i < d; i += blockDim.x) s += x[i];
  const float mean = block_sum(s) / (float)d;
  float q = 0.f;
  for (int i = tid; i < d; i += blockDim.x) {
    const float c = x[i] - mean;
    q += c * c;
  }
  const float rstd = rsqrtf(block_sum(q) / (float)d + eps);
  for (int i = tid; i < d; i += blockDim.x) pooled[i] = (x[i] - mean) * rstd * gamma[i] + beta[i];
  __syncthreads();
  const int out_dim = proj ? proj_dim : d;
  if (proj) {
    for (int o = warp; o < proj_dim; o += nw) {
      const float* w = proj + (size_t)o * d;
      float acc = 0.f;
      for (int i = lane * 4; i < d; i += 128) {
        const float4 a = __ldg((const float4*)(w + i));
        acc += a.x * pooled[i] + a.y * pooled[i + 1] + a.z * pooled[i + 2] + a.w * pooled[i + 3];
      }
      acc = warp_sum(acc);
      if (lane == 0) feat[o] = acc;
    }
  } else {
    for (int i = tid; i < d; i += blockDim.x) feat[i] = pooled[i];
  }
  __syncthreads();
  float n2 = 0.f;
  for (int i = tid; i < out_dim; i += blockDim.x) n2 += feat[i] * feat[i];
  const float inv = 1.f / sqrtf(block_sum(n2));
  float sc = 0.f;
  for (int i = tid; i < out_dim; i += blockDim.x) {
    const float e = feat[i] * inv;
    emb_out[(size_t)blockIdx.x * out_dim + i] = e;
    if (feat_out) feat_out[(size_t)blockIdx.x * out_dim + i] = feat[i];
    if (aes_w) sc += e * aes_w[i];
  }
  if (score_out && aes_w) {
    const float tot = block_sum(sc);
    if (tid == 0) score_out[blockIdx.x] = tot + aes_b;
  }
}

// ------------------------------------------------------------------------------------ SigLIP MAP head
// Multi-head attention pooling with ONE learned query (HF SiglipMultiheadAttentionPoolingHead): per (image, head)
// softmax_t(q_h . k_t) applied to v_t.  kv: fp16 [n][tokens][2*hidden] (k | v), q: fp32 [hidden] already scaled by
// head_dim^-1/2, out: fp16 [n][hidden].
__global__ void __launch_bounds__(256) map_pool_kernel(const __half* __restrict__ kv, const float* __restrict__ q, __half* __restrict__ out,
                                                       int tokens, int heads, int head_dim) {
  extern __shared__ float sm_map[];  // [tokens] probabilities, then [head_dim] query
  float* prob = sm_map;
  float* qh = sm_map + tokens;
  __shared__ float red[32];
  const int img = blockIdx.x / heads, head = blockIdx.x - img * heads;
  const int hidden = heads * head_dim, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const __half* base = kv + (size_t)img * tokens * 2 * hidden + (size_t)head * head_dim;
  for (int d = tid; d < head_dim; d += blockDim.x) qh[d] = q[head * head_dim + d];
  __syncthreads();
  float mx = -INFINITY;
  for (int t = tid; t < tokens; t += blockDim.x) {
    const __half* k = base + (size_t)t * 2 * hidden;
    float s = 0.f;
    for (int d = 0; d < head_dim; d += 2) {
      const float2 kk = __half22float2(*(const __half2*)(k + d));
      s = fmaf(kk.x, qh[d], fmaf(kk.y, qh[d + 1], s));
    }
    prob[t] = s;
    mx = fmaxf(mx, s);
  }
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
  for (int i = 1; i < nw; ++i) mx = fmaxf(mx, red[i]);
  __syncthreads();
  float sum = 0.f;
  for (int t = tid; t < tokens; t += blockDim.x) {
    const float e = __expf(prob[t] - mx);
    prob[t] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  float tot = 0.f;
  for (int i = 0; i < nw; ++i) tot += red[i];
  const float inv = 1.f / tot;
  // o_d = sum_t p_t v[t][d]: threads over (d, token slice) then a shared-memory reduction over slices
  const int slices = blockDim.x / head_dim > 0 ? blockDim.x / head_dim : 1;
  __syncthreads();
  float* part = qh;  // reuse: needs slices*head_dim floats (allocated by the host)
  if (tid < slices * head_dim) {
    const int d = tid % head_dim, sl = tid / head_dim;
    const __half* v = base + hidden + d;
    float acc = 0.f;
    for (int t = sl; t < tokens; t += slices) acc = fmaf(prob[t], __half2float(v[(size_t)t * 2 * hidden]), acc);
    part[sl * head_dim + d] = acc;
  }
  __syncthreads();
  if (tid < head_dim) {
    float acc = 0.f;
    for (int sl = 0; sl < slices; ++sl) acc += part[sl * head_dim + tid];
    out[(size_t)img * hidden + head * head_dim + tid] = __float2half_rn(acc * inv);
  }
}

// emb = feat / ||feat||, optional score = w . emb + b; one warp per row
__global__ void __launch_bounds__(256) l2norm_score_kernel(const float* __restrict__ feat, int d, const float* __restrict__ aes_w, float aes_b,
                                                           float* __restrict__ emb_out, float* __restrict__ feat_out, float* __restrict__ score_out,
                                                           int n) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  const float* x = feat + (size_t)row * d;
  float n2 = 0.f;
  for (int i = lane; i < d; i += 32) n2 = fmaf(x[i], x[i], n2);
  const float inv = 1.f / sqrtf(warp_sum(n2));
  float sc = 0.f;
  for (int i = lane; i < d; i += 32) {
    const float e = x[i] * inv;
    emb_out[(size_t)row * d + i] = e;
    if (feat_out) feat_out[(size_t)row * d + i] = x[i];
    if (aes_w) sc = fmaf(e, aes_w[i], sc);
  }
  if (score_out && aes_w) {
    sc = warp_sum(sc);
    if (lane == 0) score_out[row] = sc + aes_b;
  }
}

// score[i] = w . emb[i] + b : the reference's aesthetic MLP (aesthetics.py:44-53) folded to its affine map
__global__ void __launch_bounds__(256) affine_score_kernel(const float* __restrict__ emb, const float* __restrict__ w, float b,
                                                           float* __restrict__ out, int n, int d) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n) return;
  float acc = 0.f;
  for (int i = lane; i < d; i += 32) acc += emb[(size_t)row * d + i] * __ldg(w + i);
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc + b;
}

// ------------------------------------------------------------------------------------------ host
int affine_score(cb_ctx* ctx, const float* emb, const float* w, float b, float* out, int n, int d, cudaStream_t stream) {
  if (!emb || !w || !out) return fail(ctx, CB_ERR_ARG, "affine_score: null operand");
  if (n <= 0) return CB_OK;
  mark_launch(ctx, CB_PROF_OTHER, stream);
  affine_score_kernel<<<(n + 7) / 8, 256, 0, stream>>>(emb, w, b, out, n, d);
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

int layernorm_f16(cb_ctx* ctx, const float* x, const float* gamma, const float* beta, void* y, int rows, int d, float eps, cudaStream_t stream) {
  if (!x || !gamma || !beta || !y) return fail(ctx, CB_ERR_ARG, "layernorm: null operand");
  if (rows <= 0) return CB_OK;
  if (d % 128 || d > 128 * kLnMaxChunks) return fail(ctx, CB_ERR_UNSUPPORTED, "layernorm: d=%d must be a multiple of 128 and <= %d", d, 128 * kLnMaxChunks);
  mark_launch(ctx, CB_PROF_LAYERNORM, stream);
  const unsigned grid = (unsigned)((rows + 7) / 8);
  // one instantiation per tower width reaches copy bandwidth, the generic one 81-88 % of it (profiles/r02_layernorm_ab.jsonl)
  switch (d >> 7) {  // ViT-B 768, ViT-L 1024, SoViT-400m 1152
    case 6: layernorm_kernel<6, 4><<<grid, 256, 0, stream>>>(x, gamma, beta, (__half*)y, rows, d, eps); break;
    case 8: layernorm_kernel<8, 3><<<grid, 256, 0, stream>>>(x, gamma, beta, (__half*)y, rows, d, eps); break;
    case 9: layernorm_kernel<9, 3><<<grid, 256, 0, stream>>>(x, gamma, beta, (__half*)y, rows, d, eps); break;
    default: layernorm_kernel<0, 3><<<grid, 256, 0, stream>>>(x, gamma, beta, (__half*)y, rows, d, eps); break;
  }
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

int assemble_tokens(cb_ctx* ctx, const float* patch, const float* cls, const float* pos, const float* gamma, const float* beta, float* h, int n,
                    int tokens, int grid2, int d, float eps, cudaStream_t stream) {
  if (d % 128 || d > 128 * kLnMaxChunks) return fail(ctx, CB_ERR_UNSUPPORTED, "assemble: d=%d unsupported", d);
  const int rows = n * tokens;
  mark_launch(ctx, CB_PROF_OTHER, stream);
  assemble_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(patch, cls, pos, gamma, beta, h, n, tokens, grid2, d, eps);
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

int attention_tc2(cb_ctx* ctx, const void* qkv, void* out, int n, int tokens, int heads, int head_dim, cudaStream_t stream, bool* launched);

int attention_f16(cb_ctx* ctx, const void* qkv, void* out, int n, int tokens, int heads, int head_dim, cudaStream_t stream) {
  if (!qkv || !out) return fail(ctx, CB_ERR_ARG, "attention: null operand");
  if (n <= 0) return CB_OK;
  {  // head_dim 64, 129..257 tokens (ViT-L/14): tcgen05 kernel (attention_tc2.cu; CB_ATTN_KERNEL=mma skips it); everything else: mma.sync kernel below
    bool launched = false;
    const int rc = attention_tc2(ctx, qkv, out, n, tokens, heads, head_dim, stream, &launched);
    if (rc || launched) return rc;
  }
  if (tokens <= 0 || heads <= 0 || head_dim % 8 || head_dim > 80 || head_dim < 16)
    return fail(ctx, CB_ERR_UNSUPPORTED, "attention: tokens=%d heads=%d head_dim=%d unsupported", tokens, heads, head_dim);
  const int hd = head_dim <= 64 ? 64 : 80;
  const int t_pad = (tokens + 15) & ~15;
  const size_t resident = (size_t)2 * t_pad * (hd + 8) * 2;
  const bool stream_keys = resident > 100 * 1024;  // keep two CTAs per SM; longer sequences stream their keys
  const size_t smem = stream_keys ? (size_t)2 * kStreamKeys * (hd + 8) * 2 : resident;
  const float scale_log2e = 1.4426950408889634f / sqrtf((float)head_dim);
  const dim3 grid(n * heads, stream_keys ? ((t_pad >> 4) + kAttnWarps - 1) / kAttnWarps : 1);
  mark_launch(ctx, CB_PROF_ATTENTION, stream);
#define CB_ATTN_LAUNCH(HD_, ST_)                                                                                               \
  do {                                                                                                                         \
    CB_CUDA(ctx, cudaFuncSetAttribute(attention_kernel<HD_, ST_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));    \
    attention_kernel<HD_, ST_><<<grid, kAttnThreads, smem, stream>>>((const __half*)qkv, (__half*)out, tokens, heads, head_dim, scale_log2e); \
  } while (0)
  if (hd == 64 && !stream_keys) CB_ATTN_LAUNCH(64, false);
  else if (hd == 64) CB_ATTN_LAUNCH(64, true);
  else if (!stream_keys) CB_ATTN_LAUNCH(80, false);
  else CB_ATTN_LAUNCH(80, true);
#undef CB_ATTN_LAUNCH
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

int map_pool(cb_ctx* ctx, const void* kv, const float* q, void* out, int n, int tokens, int heads, int head_dim, cudaStream_t stream) {
  const int threads = 256;
  const int slices = threads / head_dim > 0 ? threads / head_dim : 1;
  const size_t smem = (size_t)(tokens + slices * head_dim) * sizeof(float);
  if (smem > 48 * 1024) CB_CUDA(ctx, cudaFuncSetAttribute(map_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mark_launch(ctx, CB_PROF_OTHER, stream);
  map_pool_kernel<<<n * heads, threads, smem, stream>>>((const __half*)kv, q, (__half*)out, tokens, heads, head_dim);
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

int l2norm_score(cb_ctx* ctx, const float* feat, int d, const float* aes_w, float aes_b, float* emb, float* feat_out, float* score, int n,
                 cudaStream_t stream) {
  mark_launch(ctx, CB_PROF_OTHER, stream);
  l2norm_score_kernel<<<(n + 7) / 8, 256, 0, stream>>>(feat, d, aes_w, aes_b, emb, feat_out, score, n);
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

int clip_tail(cb_ctx* ctx, const float* h, size_t img_stride, const float* gamma, const float* beta, const float* proj, int d, int proj_dim,
              float eps, const float* aes_w, float aes_b, float* emb_out, float* feat_out, float* score_out, int n, cudaStream_t stream) {
  const int out_dim = proj ? proj_dim : d;
  const size_t smem = (size_t)(d + out_dim) * sizeof(float);
  mark_launch(ctx, CB_PROF_OTHER, stream);
  clip_tail_kernel<<<n, 256, smem, stream>>>(h, img_stride, gamma, beta, proj, d, proj_dim, eps, aes_w, aes_b, emb_out, feat_out, score_out);
  CB_CUDA(ctx, cudaGetLastError());
  return CB_OK;
}

}  // namespace cb

extern "C" {
int cb_affine_score(cb_ctx* ctx, const float* emb, const float* w, float b, float* out, int n, int d, void* stream) {
  if (!ctx) return CB_ERR_ARG;
  return cb::affine_score(ctx, emb, w, b, out, n, d, (cudaStream_t)stream);
}
int cb_layernorm_f16(cb_ctx* ctx, const float* x, const float* gamma, const float* beta, void* y, int rows, int d, float eps, void* stream) {
  if (!ctx) return CB_ERR_ARG;
  return cb::layernorm_f16(ctx, x, gamma, beta, y, rows, d, eps, (cudaStream_t)stream);
}
int cb_attention_f16(cb_ctx* ctx, const void* qkv, void* out, int n, int tokens, int heads, int head_dim, void* stream) {
  if (!ctx) return CB_ERR_ARG;
  return cb::attention_f16(ctx, qkv, out, n, tokens, heads, head_dim, (cudaStream_t)stream);
}
}
