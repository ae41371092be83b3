// Round-2 rewrites of the DaViT / BART SIMT kernels for the 64x64-crop mode (416 crops per batch, maps 16x16 .. 2x2).
// The first versions (florence_ops.cu) spent 3.5 ms of the 9.2 ms caption encode in these kernels at 0.5-1 TB/s: every
// token re-read its nine depthwise taps and weights through L1, every (crop, head) was a one-warp CTA, the channel attention
// ran its softmax as 64 butterfly reductions per group.  Here a CTA owns a tile that fits shared memory, loads it once with
// coalesced 16-byte accesses, keeps per-thread constants (depthwise weights, probability rows) in registers, and writes
// whole rows back.  Selected by split bit 2 (value 4) of the C-ABI entry points; without it, and for shapes these do not
// cover (768-mode maps), the entry points run the first versions, which also serve as the checkers (tests/test_ops_gpu.py
// compares both).
// Reference math: hf:models/florence2/modeling_florence2.py (ConvPosEnc 281-293, WindowAttention 346-383,
// ChannelAttention 228-264), hf:models/bart/modeling_bart.py:143-258.
#include "ptx.cuh"
#include "b2p_internal.h"
#include <atomic>
#include <cuda_fp16.h>
#include <math.h>

namespace b2p {

// Bulk asynchronous copy global -> shared (the non-tensor TMA path): ONE instruction moves a contiguous block (16-byte
// aligned, size % 16 == 0) and signals an mbarrier with its byte count.  The first versions of these kernels staged their
// tiles with per-thread load/store loops whose iterations serialised on the L2 round trip (time_ops: ~24 us per launch for
// 40 MB that sits in L2); with bulk copies the whole tile is in flight at once and the threads prefetch their constants
// meanwhile.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

__device__ __forceinline__ float wsum(float v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// fp16 store of 4 consecutive channels (c % 4 == 0); split > 0: [hi | lo] pair, lo `split` elements after hi
__device__ __forceinline__ void put4(__half* row, int c, int split, const float4& v) {
  __align__(8) __half2 h[2] = {__floats2half2_rn(v.x, v.y), __floats2half2_rn(v.z, v.w)};
  *reinterpret_cast<uint2*>(row + c) = *reinterpret_cast<const uint2*>(h);
  if (split) {
    const float2 a = __half22float2(h[0]), b = __half22float2(h[1]);
    __align__(8) __half2 l[2] = {__floats2half2_rn(v.x - a.x, v.y - a.y), __floats2half2_rn(v.z - b.x, v.w - b.y)};
    *reinterpret_cast<uint2*>(row + split + c) = *reinterpret_cast<const uint2*>(l);
  }
}

// ------------------------------------------------------------------------------ depthwise 3x3 + residual + LayerNorm
// y = dwconv3x3(x) + bias + x (fp32 residual stream), h = LayerNorm(y) (fp16 [hi | lo] GEMM operand).
// CTA = (image, strip of R rows): the strip + its halo rows sit in shared memory (one coalesced load).  256 threads =
// C/4 channel quads x G token groups; a thread keeps its 9 weights in registers and produces <= NT tokens, so the taps are
// 9 conflict-free LDS.128 per token instead of 18 global loads.  LayerNorm statistics: warp butterfly + one partial per
// 128-channel block through shared memory (two passes: mean, then variance about the mean, as nn.LayerNorm).
// The convolution sums in the order of dwconv_ln_kernel (y is bit-identical); the LayerNorm sums associate differently.
constexpr int kDwThreads = 256, kDwNT = 8;

// shared memory: [input tile: the strip's rows + existing halo rows, W x C each][one zero pixel][conv results R x W x C]
// [partials 2 x R*W*wpt][mbarrier].  Out-of-image taps read the zero pixel (a select on the address instead of a branch; a
// zero tap leaves the fp32 sum unchanged, so y stays bit-identical with the first versions); W is a power of two (shift / mask
// instead of divisions); the token loops stay ROLLED: fully unrolled the kernel was 4096 instructions and its warps stalled
// on instruction fetch (ncu: "no instruction" was the top stall reason).
__global__ void __launch_bounds__(kDwThreads, 3) dwconv_ln_v3_kernel(const float* __restrict__ x, int H, int W, int lw, int C, int R,
                                                                     const float* __restrict__ w9c, const float* __restrict__ bias,
                                                                     float* __restrict__ y, const float* __restrict__ g,
                                                                     const float* __restrict__ bt, float eps, __half* __restrict__ o16,
                                                                     int split) {
  pdl_wait();
  extern __shared__ float4 dsm4[];
  const int C4 = C >> 2, G = kDwThreads / C4, wpt = C4 >> 5;   // wpt: warps (128-channel blocks) per token
  const int strips = (H + R - 1) / R;
  const int b = blockIdx.x / strips, s = blockIdx.x - b * strips;
  const int y0 = s * R, y1 = min(H, y0 + R);
  const int ya = max(0, y0 - 1), yb = min(H, y1 + 1);
  const int rs = W * C4;                                       // float4 per tile row
  const int zoff = (R + 2) * rs;                               // the zero pixel
  float4* ys4 = dsm4 + zoff + C4;                              // this thread re-reads only what it wrote: no barrier needed
  float* part = reinterpret_cast<float*>(ys4 + R * rs);       // [2][R*W*wpt]
  const int pstride = R * W * wpt;
  const uint32_t bar = smem_u32(part + 2 * pstride);           // 2 * pstride is even: 8-byte aligned
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  for (int i = threadIdx.x; i < C4; i += kDwThreads) dsm4[zoff + i] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t bytes = uint32_t(yb - ya) * uint32_t(rs) * 16u;
    mbar_expect_tx(bar, bytes);
    bulk_g2s(smem_u32(dsm4), x + ((long long)b * H + ya) * W * C, bytes, bar);
  }
  const int c4 = threadIdx.x % C4, grp = threadIdx.x / C4, wc = c4 >> 5, lane = threadIdx.x & 31;
  float4 wv[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) wv[k] = reinterpret_cast<const float4*>(w9c + k * C)[c4];
  const float4 bv = reinterpret_cast<const float4*>(bias)[c4];
  const float4 gg = reinterpret_cast<const float4*>(g)[c4], bb = reinterpret_cast<const float4*>(bt)[c4];
  const int TT = (y1 - y0) << lw;        // output tokens of this strip
  const int wm = W - 1;
  const long long tok0 = ((long long)b * H + y0) << lw;
  mbar_wait(bar, 0);
  // ---- convolution + residual, row sums
#pragma unroll 1
  for (int t = grp; t < TT; t += G) {    // warp-uniform
    const int ty = y0 + (t >> lw), tx = t & wm;
    const int base = ((ty - ya) * W + tx) * C4 + c4;           // centre tap
    float4 acc = bv;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const bool rv = (ty + ky - 1 >= 0) && (ty + ky - 1 < H);
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const bool ok = rv && (tx + kx - 1 >= 0) && (tx + kx - 1 < W);
        const float4 xv = dsm4[ok ? base + (ky - 1) * rs + (kx - 1) * C4 : zoff + c4];
        const float4 ww = wv[ky * 3 + kx];
        acc.x += xv.x * ww.x; acc.y += xv.y * ww.y; acc.z += xv.z * ww.z; acc.w += xv.w * ww.w;
      }
    }
    const float4 xc = dsm4[base];
    acc.x += xc.x; acc.y += xc.y; acc.z += xc.z; acc.w += xc.w;
    reinterpret_cast<float4*>(y + (tok0 + t) * C)[c4] = acc;
    ys4[t * C4 + c4] = acc;
    const float r = wsum((acc.x + acc.y) + (acc.z + acc.w));
    if (lane == 0) part[t * wpt + wc] = r;
  }
  __syncthreads();
  // ---- variance about the mean
  const float invC = 1.f / float(C);
#pragma unroll 1
  for (int t = grp; t < TT; t += G) {
    float m = 0.f;
    for (int k = 0; k < wpt; ++k) m += part[t * wpt + k];
    m *= invC;
    const float4 v = ys4[t * C4 + c4];
    const float dx = v.x - m, dy = v.y - m, dz = v.z - m, dw = v.w - m;
    const float r = wsum((dx * dx + dy * dy) + (dz * dz + dw * dw));
    if (lane == 0) part[pstride + t * wpt + wc] = r;
  }
  __syncthreads();
  const int ld16 = split ? 2 * C : C;
#pragma unroll 1
  for (int t = grp; t < TT; t += G) {
    float m = 0.f, q = 0.f;
    for (int k = 0; k < wpt; ++k) { m += part[t * wpt + k]; q += part[pstride + t * wpt + k]; }
    m *= invC;
    const float rstd = rsqrtf(q * invC + eps);
    const float4 v = ys4[t * C4 + c4];
    float4 o;
    o.x = (v.x - m) * rstd * gg.x + bb.x; o.y = (v.y - m) * rstd * gg.y + bb.y;
    o.z = (v.z - m) * rstd * gg.z + bb.z; o.w = (v.w - m) * rstd * gg.w + bb.w;
    put4(o16 + (tok0 + t) * ld16, 4 * c4, split, o);
  }
}

// -> 0 launched, 1 shape not covered (caller falls back to the first-version kernels), < 0 error
int dwconv_ln_v3_launch(const float* x, int B, int H, int W, int C, const float* w9c, const float* bias, float* y,
                        const float* gamma, const float* beta, float eps, void* out16, int split, cudaStream_t st) {
  const int C4 = C / 4;
  if (C % 128 || C4 > kDwThreads || kDwThreads % C4 || B <= 0 || W < 1 || (W & (W - 1))) return 1;
  int lw = 0;
  while ((1 << lw) < W) ++lw;
  const int G = kDwThreads / C4;
  if (W > kDwNT * G) return 1;
  int R = (kDwNT * G) / W;
  if (R > H) R = H;
  const size_t smem = (size_t(2 * R + 2) * W + 1) * C * sizeof(float) + (2 * size_t(R) * W * (C4 / 32) + 4) * sizeof(float);
  if (smem > 100 * 1024) return 1;
  static std::atomic<bool> attr{false};
  if (!attr) {
    if (cudaFuncSetAttribute(dwconv_ln_v3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024) != cudaSuccess)
      return set_error("dwconv_ln: cudaFuncSetAttribute failed");
    attr = true;
  }
  const int strips = (H + R - 1) / R;
  launch_pdl(dwconv_ln_v3_kernel, dim3(B * strips), dim3(kDwThreads), smem, st, x, H, W, lw, C, R, w9c, bias, y, gamma, beta, eps,
             (__half*)out16, split ? C : 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(cudaGetErrorString(e));
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------ window attention, one window per image
// Maps no larger than the 12x12 window (the 8x8 / 4x4 / 2x2 maps of the 64x64-crop mode): the map is ONE window of nreal =
// H*W real tokens + (144 - nreal) zero-padded tokens whose k, v are the bias vectors (see window_attn_kernel).  CTA =
// (image, group of HPC heads): K and V of those heads for all tokens are staged once (coalesced float4 rows), thread =
// (head, query) runs the same online-softmax recurrence as window_attn_kernel (bit-identical results), and the outputs
// leave through a shared-memory transpose as whole [hi | lo] row segments.
// shared memory: [token][K seg (HPC*32) | V seg (HPC*32)] fp32 (re-used as the output stage), then the mbarrier.
// QB queries per thread (t, t + nreal / QB, ...): every K / V row read from shared memory feeds QB independent online-softmax
// chains (the one-query loop was bound by the latency of its LDS -> FMA -> MUFU chain at 30 % occupancy, ncu short_scoreboard).
template <int QB>
__global__ void __launch_bounds__(256 / QB, 3) window_attn_crop_kernel(const float* __restrict__ qkv, const float* __restrict__ qkv_bias,
                                                                       int nreal, int npad, int C, int heads, int HPC,
                                                                       __half* __restrict__ out, int split) {
  pdl_wait();
  extern __shared__ float4 wsm4[];
  constexpr int D = 32, D4 = 8;
  const int groups = heads / HPC;
  const int b = blockIdx.x / groups, hg = blockIdx.x - b * groups;
  const int h0 = hg * HPC;
  const int row4 = 2 * HPC * D4;                   // float4 per staged token row [K seg | V seg]
  const long long tok0 = (long long)b * nreal;
  const uint32_t bar = smem_u32(wsm4 + nreal * row4);
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  __syncthreads();
  if (threadIdx.x < 32) {
    const uint32_t seg_bytes = uint32_t(HPC) * D * 4u;
    if (threadIdx.x == 0) mbar_expect_tx(bar, uint32_t(nreal) * 2u * seg_bytes);
    __syncwarp();
    for (int t = threadIdx.x; t < nreal; t += 32) {
      const float* rowp = qkv + (tok0 + t) * 3 * C + h0 * D;
      const uint32_t dst = smem_u32(wsm4 + t * row4);
      if (HPC == heads) {
        bulk_g2s(dst, rowp + C, 2u * seg_bytes, bar);               // K and V of all heads are adjacent in the row
      } else {
        bulk_g2s(dst, rowp + C, seg_bytes, bar);
        bulk_g2s(dst + seg_bytes, rowp + 2 * C, seg_bytes, bar);
      }
    }
  }
  const int nq = nreal / QB;                                         // queries per (head, thread slot); nreal % QB == 0
  const int hh = threadIdx.x / nq, t0 = threadIdx.x - hh * nq;       // blockDim.x == HPC * nq
  const int head = h0 + hh;
  float4 q[QB][D4], acc[QB][D4];
  float m[QB], l[QB];
  const float scale = rsqrtf(float(D));
#pragma unroll
  for (int u = 0; u < QB; ++u) {
    const float4* qp = reinterpret_cast<const float4*>(qkv + (tok0 + t0 + u * nq) * 3 * C + head * D);
#pragma unroll
    for (int d = 0; d < D4; ++d) q[u][d] = qp[d];
  }
#pragma unroll
  for (int u = 0; u < QB; ++u) {
#pragma unroll
    for (int d = 0; d < D4; ++d) {
      q[u][d].x *= scale; q[u][d].y *= scale; q[u][d].z *= scale; q[u][d].w *= scale;
      acc[u][d] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    m[u] = -INFINITY; l[u] = 0.f;
  }
  if (npad > 0) {
#pragma unroll
    for (int u = 0; u < QB; ++u) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < D4; ++d) {
        const float4 kb = reinterpret_cast<const float4*>(qkv_bias + C + head * D)[d];
        s += (q[u][d].x * kb.x + q[u][d].y * kb.y) + (q[u][d].z * kb.z + q[u][d].w * kb.w);
      }
      m[u] = s;
      l[u] = float(npad);
#pragma unroll
      for (int d = 0; d < D4; ++d) {
        const float4 vb = reinterpret_cast<const float4*>(qkv_bias + 2 * C + head * D)[d];
        acc[u][d] = make_float4(l[u] * vb.x, l[u] * vb.y, l[u] * vb.z, l[u] * vb.w);
      }
    }
  }
  mbar_wait(bar, 0);
  for (int j = 0; j < nreal; ++j) {
    const float4* kr = wsm4 + j * row4 + hh * D4;
    float s[QB], p[QB];
#pragma unroll
    for (int u = 0; u < QB; ++u) s[u] = 0.f;
#pragma unroll
    for (int d = 0; d < D4; ++d) {
      const float4 kk = kr[d];
#pragma unroll
      for (int u = 0; u < QB; ++u) s[u] += (q[u][d].x * kk.x + q[u][d].y * kk.y) + (q[u][d].z * kk.z + q[u][d].w * kk.w);
    }
#pragma unroll
    for (int u = 0; u < QB; ++u) {
      if (s[u] > m[u]) {
        const float r = __expf(m[u] - s[u]);
        l[u] *= r;
#pragma unroll
        for (int d = 0; d < D4; ++d) { acc[u][d].x *= r; acc[u][d].y *= r; acc[u][d].z *= r; acc[u][d].w *= r; }
        m[u] = s[u];
      }
      p[u] = __expf(s[u] - m[u]);
      l[u] += p[u];
    }
    const float4* vr = kr + HPC * D4;
#pragma unroll
    for (int d = 0; d < D4; ++d) {
      const float4 vv = vr[d];
#pragma unroll
      for (int u = 0; u < QB; ++u) {
        acc[u][d].x += p[u] * vv.x; acc[u][d].y += p[u] * vv.y; acc[u][d].z += p[u] * vv.z; acc[u][d].w += p[u] * vv.w;
      }
    }
  }
  __syncthreads();                                  // everyone is done reading K / V: reuse the buffer as the output stage
  // stage: [plane (hi, lo)][token][HPC*32 halves]
  __half* stg = reinterpret_cast<__half*>(wsm4);
  const int seg = HPC * D;                          // halves per token per plane
#pragma unroll
  for (int u = 0; u < QB; ++u) {
    const float inv = 1.f / l[u];
    __half* rh = stg + (t0 + u * nq) * seg;
#pragma unroll
    for (int d = 0; d < D4; ++d)
      put4(rh, hh * D + 4 * d, split ? nreal * seg : 0,
           make_float4(acc[u][d].x * inv, acc[u][d].y * inv, acc[u][d].z * inv, acc[u][d].w * inv));
  }
  __syncthreads();
  const int planes = split ? 2 : 1;
  const int seg8 = seg >> 3;                        // 16-byte chunks per token per plane
  const int ld16 = split ? 2 * C : C;
  for (int i = threadIdx.x; i < planes * nreal * seg8; i += blockDim.x) {
    const int pl = i / (nreal * seg8), r = i - pl * nreal * seg8;
    const int tt = r / seg8, c8 = r - tt * seg8;
    const uint4 val = reinterpret_cast<const uint4*>(stg + (pl * nreal + tt) * seg)[c8];
    *reinterpret_cast<uint4*>(out + (tok0 + tt) * ld16 + pl * C + h0 * D + 8 * c8) = val;
  }
}

int window_attn_crop_launch(const float* qkv, const float* qkv_bias, int B, int H, int W, int C, int heads, int win, void* out,
                            int split, cudaStream_t st) {
  if (H > win || W > win || C != heads * 32 || B <= 0) return 1;
  const int nreal = H * W;
  if (nreal > 64) return 1;
  int HPC = 256 / nreal;
  if (HPC > heads) HPC = heads;
  while (HPC > 1 && heads % HPC) --HPC;
  const int QB = (nreal % 2 == 0) ? 2 : 1;          // two queries per thread whenever the token count is even
  const int threads = HPC * (nreal / QB);
  if (threads > 256 / QB || threads < 1) return 1;
  const size_t smem = size_t(2) * nreal * HPC * 32 * sizeof(float) + 16;
  static std::atomic<bool> attr{false};
  if (!attr) {
    if (cudaFuncSetAttribute(window_attn_crop_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(window_attn_crop_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65 * 1024) != cudaSuccess)
      return set_error("window_attn: cudaFuncSetAttribute failed");
    attr = true;
  }
  if (smem > 65 * 1024) return 1;
  if (QB == 2)
    launch_pdl(window_attn_crop_kernel<2>, dim3(B * (heads / HPC)), dim3(threads), smem, st, qkv, qkv_bias, nreal, win * win - nreal, C,
               heads, HPC, (__half*)out, split ? 1 : 0);
  else
    launch_pdl(window_attn_crop_kernel<1>, dim3(B * (heads / HPC)), dim3(threads), smem, st, qkv, qkv_bias, nreal, win * win - nreal, C,
               heads, HPC, (__half*)out, split ? 1 : 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(cudaGetErrorString(e));
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------ channel attention
// Per (image, group): S[i][j] = N^-0.5 sum_n q[n][i] k[n][j], P = softmax_j S, out[n][i] = sum_j P[i][j] v[n][j]  (d = 32).
// CTA = one (image, group), NW warps; q, k, v of the group are staged once.  Warp w owns tokens [w*Nw, (w+1)*Nw): lane j
// accumulates its column of S for all 32 rows in registers (one conflict-free LDS of k[n][j] + 8 broadcast LDS.128 of q[n][:]
// per token), partial S tiles are summed in warp order, lane i then runs the softmax of row i serially (no butterflies) and
// keeps P[i][:] in registers for the output pass (8 broadcast LDS.128 of v[n][:] per token).
template <int NW>
__global__ void __launch_bounds__(NW * 32) channel_attn_v3_kernel(const float* __restrict__ qkv, int N, int C, int groups,
                                                                  __half* __restrict__ out, int split) {
  pdl_wait();
  extern __shared__ float4 csm4[];
  constexpr int D = 32;
  float* qs = reinterpret_cast<float*>(csm4);      // [N][32]
  float* ks = qs + N * D;
  float* vs = ks + N * D;
  float* Sp = vs + N * D;                           // [NW][32][33] partial S, then P in slot 0
  const int g = blockIdx.x % groups, b = blockIdx.x / groups;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* base = qkv + (long long)b * N * 3 * C + g * D;
  // staging: 4 iterations (12 independent 16-byte loads) in flight per thread before the first store
  for (int i0 = threadIdx.x; i0 < N * 8; i0 += 4 * NW * 32) {
    float4 tq[4], tk[4], tv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * NW * 32;
      if (i < N * 8) {
        const float* rowp = base + (long long)(i >> 3) * 3 * C;
        tq[u] = reinterpret_cast<const float4*>(rowp)[i & 7];
        tk[u] = reinterpret_cast<const float4*>(rowp + C)[i & 7];
        tv[u] = reinterpret_cast<const float4*>(rowp + 2 * C)[i & 7];
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * NW * 32;
      if (i < N * 8) {
        reinterpret_cast<float4*>(qs)[i] = tq[u];
        reinterpret_cast<float4*>(ks)[i] = tk[u];
        reinterpret_cast<float4*>(vs)[i] = tv[u];
      }
    }
  }
  __syncthreads();
  const int Nw = (N + NW - 1) / NW;
  const int n0 = w * Nw, n1 = min(N, n0 + Nw);
  float s[D];
#pragma unroll
  for (int i = 0; i < D; ++i) s[i] = 0.f;
  for (int n = n0; n < n1; ++n) {
    const float kj = ks[n * D + lane];
    const float4* qr = reinterpret_cast<const float4*>(qs + n * D);
#pragma unroll
    for (int i4 = 0; i4 < 8; ++i4) {
      const float4 qq = qr[i4];
      s[4 * i4 + 0] += qq.x * kj; s[4 * i4 + 1] += qq.y * kj; s[4 * i4 + 2] += qq.z * kj; s[4 * i4 + 3] += qq.w * kj;
    }
  }
  float* mySp = Sp + w * (D * 33);
#pragma unroll
  for (int i = 0; i < D; ++i) mySp[i * 33 + lane] = s[i];
  __syncthreads();
  if (w == 0) {
    // lane = row i: sum the partial tiles in warp order, softmax over j, P[i][:] back into slot 0
    const float sc = rsqrtf(float(N));
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < D; ++j) {
      float a = Sp[lane * 33 + j];
      for (int ww = 1; ww < NW; ++ww) a += Sp[ww * (D * 33) + lane * 33 + j];
      a *= sc;
      s[j] = a;
      mx = fmaxf(mx, a);
    }
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < D; ++j) { s[j] = __expf(s[j] - mx); sum += s[j]; }
    const float inv = 1.f / sum;
#pragma unroll
    for (int j = 0; j < D; ++j) Sp[lane * 33 + j] = s[j] * inv;
  }
  __syncthreads();
  float pr[D];
#pragma unroll
  for (int j = 0; j < D; ++j) pr[j] = Sp[lane * 33 + j];
  const int ld16 = split ? 2 * C : C;
  for (int n = n0; n < n1; ++n) {
    const float4* vr = reinterpret_cast<const float4*>(vs + n * D);
    float acc = 0.f;
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
      const float4 vv = vr[j4];
      acc += pr[4 * j4 + 0] * vv.x; acc += pr[4 * j4 + 1] * vv.y; acc += pr[4 * j4 + 2] * vv.z; acc += pr[4 * j4 + 3] * vv.w;
    }
    __half* orow = out + ((long long)b * N + n) * ld16 + g * D + lane;
    const __half hv = __float2half_rn(acc);
    *orow = hv;
    if (split) orow[C] = __float2half_rn(acc - __half2float(hv));
  }
}

// Few tokens (N <= 32: the 4x4 / 2x2 maps, nine + one launches per encode): CTA = (image, chunk of GPC groups), one warp
// per group, the [q | k | v] segments of the chunk arrive by bulk copies.  Lane i owns ROW i of S: s[j] += q[n][i] * k[n][j]
// with k[n][:] broadcast, so the softmax over j and the probabilities P[i][:] stay in that lane's registers (no transpose,
// no inter-warp traffic); the output pass broadcasts v[n][:].
__global__ void __launch_bounds__(256) channel_attn_rows_kernel(const float* __restrict__ qkv, int N, int C, int groups, int GPC,
                                                                __half* __restrict__ out, int split) {
  pdl_wait();
  extern __shared__ float4 csm4[];
  constexpr int D = 32;
  const int chunks = groups / GPC;
  const int b = blockIdx.x / chunks, g0 = (blockIdx.x - b * chunks) * GPC;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rowf = 3 * GPC * D;                       // floats per staged token row [q seg | k seg | v seg]
  float* sm = reinterpret_cast<float*>(csm4);
  const uint32_t bar = smem_u32(sm + N * rowf);
  if (threadIdx.x == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  __syncthreads();
  if (threadIdx.x < 32) {
    const uint32_t seg_bytes = uint32_t(GPC) * D * 4u;
    if (threadIdx.x == 0) mbar_expect_tx(bar, uint32_t(N) * 3u * seg_bytes);
    __syncwarp();
    if (GPC == groups) {
      // whole rows, and the rows of one image are contiguous: one copy
      if (threadIdx.x == 0) bulk_g2s(smem_u32(sm), qkv + (long long)b * N * 3 * C, uint32_t(N) * 3u * seg_bytes, bar);
    } else {
      for (int i = threadIdx.x; i < 3 * N; i += 32) {
        const int n = i / 3, part = i - 3 * n;
        bulk_g2s(smem_u32(sm + n * rowf + part * GPC * D), qkv + ((long long)b * N + n) * 3 * C + part * C + g0 * D, seg_bytes, bar);
      }
    }
  }
  mbar_wait(bar, 0);
  const float* qs = sm + w * D;                       // + n * rowf
  const float* ks = sm + GPC * D + w * D;
  const float* vs = sm + 2 * GPC * D + w * D;
  float s[D];
#pragma unroll
  for (int j = 0; j < D; ++j) s[j] = 0.f;
  for (int n = 0; n < N; ++n) {
    const float qi = qs[n * rowf + lane];
    const float4* kr = reinterpret_cast<const float4*>(ks + n * rowf);
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
      const float4 kk = kr[j4];
      s[4 * j4 + 0] += qi * kk.x; s[4 * j4 + 1] += qi * kk.y; s[4 * j4 + 2] += qi * kk.z; s[4 * j4 + 3] += qi * kk.w;
    }
  }
  const float sc = rsqrtf(float(N));
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < D; ++j) { s[j] *= sc; mx = fmaxf(mx, s[j]); }
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < D; ++j) { s[j] = __expf(s[j] - mx); sum += s[j]; }
  const float inv = 1.f / sum;
#pragma unroll
  for (int j = 0; j < D; ++j) s[j] *= inv;
  const int ld16 = split ? 2 * C : C;
  const int g = g0 + w;
  for (int n = 0; n < N; ++n) {
    const float4* vr = reinterpret_cast<const float4*>(vs + n * rowf);
    float acc = 0.f;
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
      const float4 vv = vr[j4];
      acc += s[4 * j4 + 0] * vv.x; acc += s[4 * j4 + 1] * vv.y; acc += s[4 * j4 + 2] * vv.z; acc += s[4 * j4 + 3] * vv.w;
    }
    __half* orow = out + ((long long)b * N + n) * ld16 + g * D + lane;
    const __half hv = __float2half_rn(acc);
    *orow = hv;
    if (split) orow[C] = __float2half_rn(acc - __half2float(hv));
  }
}

static int channel_attn_rows_go(const float* qkv, int B, int N, int C, int groups, void* out, int split, cudaStream_t st) {
  int GPC = groups < 8 ? groups : 8;
  while (GPC > 1 && (groups % GPC || size_t(N) * 3 * GPC * 128 > 64 * 1024)) --GPC;
  const size_t smem = size_t(N) * 3 * GPC * 128 + 16;
  if (groups % GPC || smem > 65 * 1024) return 1;
  static std::atomic<bool> attr{false};
  if (!attr) {
    if (cudaFuncSetAttribute(channel_attn_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 65 * 1024) != cudaSuccess)
      return set_error("channel_attn: cudaFuncSetAttribute failed");
    attr = true;
  }
  launch_pdl(channel_attn_rows_kernel, dim3(B * (groups / GPC)), dim3(GPC * 32), smem, st, qkv, N, C, groups, GPC, (__half*)out, split ? 1 : 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(cudaGetErrorString(e));
  count_launch();
  return 0;
}

template <int NW>
static int channel_attn_v3_go(const float* qkv, int B, int N, int C, int groups, void* out, int split, cudaStream_t st) {
  const size_t smem = (size_t(3) * N * 32 + size_t(NW) * 32 * 33) * sizeof(float);
  static std::atomic<bool> attr{false};
  if (!attr) {
    if (cudaFuncSetAttribute(channel_attn_v3_kernel<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024) != cudaSuccess)
      return set_error("channel_attn: cudaFuncSetAttribute failed");
    attr = true;
  }
  if (smem > 160 * 1024) return 1;
  launch_pdl(channel_attn_v3_kernel<NW>, dim3(B * groups), dim3(NW * 32), smem, st, qkv, N, C, groups, (__half*)out, split ? 1 : 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(cudaGetErrorString(e));
  count_launch();
  return 0;
}

int channel_attn_v3_launch(const float* qkv, int B, int N, int C, int groups, void* out, int split, cudaStream_t st) {
  if (C != groups * 32 || B <= 0 || N <= 0 || N > 320) return 1;
  if (N <= 32) {
    const int r = channel_attn_rows_go(qkv, B, N, C, groups, out, split, st);
    if (r <= 0) return r;
    return channel_attn_v3_go<1>(qkv, B, N, C, groups, out, split, st);
  }
  if (N <= 96) return channel_attn_v3_go<2>(qkv, B, N, C, groups, out, split, st);
  return channel_attn_v3_go<8>(qkv, B, N, C, groups, out, split, st);
}

// ------------------------------------------------------------------------------ BART attention, short sequences
// Encoder self-attention of the 64x64-crop mode: Lq = Lk = 13.  mha_kernel runs one warp per (batch, head, QUERY) and every
// warp re-reads the head's K and V rows (430 MB of L2 -> SM traffic per launch).  Here one warp owns a (batch, head): K and V
// (<= 16 keys, 2 values per lane per key) stay in registers and the queries are processed in turn with exactly the
// arithmetic of mha_kernel (four keys per step, then the tail) => bit-identical outputs.
// (dealing the queries of one head to several warps measured slower: 4 warps, 48 us against 38)
constexpr int kMhaLmax = 16;
__global__ void __launch_bounds__(128) mha_short_kernel(const float* __restrict__ qp, long long ldq, const float* __restrict__ kp,
                                                        const float* __restrict__ vp, long long ldk, int B, int Lq, int Lk, int heads,
                                                        __half* __restrict__ out, long long ldo, int split) {
  pdl_wait();
  const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (wid >= B * heads) return;
  const int h = wid % heads, b = wid / heads;
  const float* kb = kp + (long long)b * Lk * ldk + h * 64;
  const float* vb = vp + (long long)b * Lk * ldk + h * 64;
  float2 kf[kMhaLmax], vf[kMhaLmax];
#pragma unroll
  for (int j = 0; j < kMhaLmax; ++j) {
    if (j < Lk) {
      kf[j] = *reinterpret_cast<const float2*>(kb + (long long)j * ldk + 2 * lane);
      vf[j] = *reinterpret_cast<const float2*>(vb + (long long)j * ldk + 2 * lane);
    } else {
      kf[j] = make_float2(0.f, 0.f); vf[j] = make_float2(0.f, 0.f);
    }
  }
  const int L4 = Lk & ~3;
  // the query loop stays ROLLED (fully unrolled it is ~11k instructions and thrashes the instruction cache: 112 us per launch
  // against 40); the next query's row is fetched one iteration ahead so its L2 round trip overlaps this query's arithmetic
  const float* qrow = qp + (long long)b * Lq * ldq + h * 64 + 2 * lane;
  float2 qn = *reinterpret_cast<const float2*>(qrow);
#pragma unroll 1
  for (int qi = 0; qi < Lq; ++qi) {
    float2 q = qn;
    if (qi + 1 < Lq) qn = *reinterpret_cast<const float2*>(qrow + (long long)(qi + 1) * ldq);
    q.x *= 0.125f; q.y *= 0.125f;
    float m = -INFINITY, l = 0.f;
    float2 acc = make_float2(0.f, 0.f);
#pragma unroll
    for (int jb = 0; jb < kMhaLmax; jb += 4) {
      if (jb + 4 <= Lk) {
        float s[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) s[u] = q.x * kf[jb + u].x + q.y * kf[jb + u].y;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int u = 0; u < 4; ++u) s[u] += __shfl_xor_sync(0xffffffffu, s[u], o);
        }
        const float mn = fmaxf(fmaxf(m, fmaxf(s[0], s[1])), fmaxf(s[2], s[3]));
        const float r = __expf(m - mn);
        l *= r; acc.x *= r; acc.y *= r;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float p = __expf(s[u] - mn);
          l += p;
          acc.x += p * vf[jb + u].x;
          acc.y += p * vf[jb + u].y;
        }
        m = mn;
      }
    }
#pragma unroll
    for (int j = 0; j < kMhaLmax; ++j) {
      if (j >= L4 && j < Lk) {
        const float s = wsum(q.x * kf[j].x + q.y * kf[j].y);
        const float mn = fmaxf(m, s);
        const float r = __expf(m - mn), p = __expf(s - mn);
        l = l * r + p;
        acc.x = acc.x * r + p * vf[j].x;
        acc.y = acc.y * r + p * vf[j].y;
        m = mn;
      }
    }
    const float inv = 1.f / l;
    __half* orow = out + ((long long)b * Lq + qi) * ldo + h * 64 + 2 * lane;
    const float o0 = acc.x * inv, o1 = acc.y * inv;
    const __half2 hv = __floats2half2_rn(o0, o1);
    *reinterpret_cast<__half2*>(orow) = hv;
    if (split) {
      const float2 hf = __half22float2(hv);
      *reinterpret_cast<__half2*>(orow + split) = __floats2half2_rn(o0 - hf.x, o1 - hf.y);
    }
  }
}

int mha_short_launch(const float* q, long long ldq, const float* k, const float* v, long long ldk, int B, int Lq, int Lk, int heads,
                     void* out, long long ldo, int split, cudaStream_t st) {
  if (Lk > kMhaLmax || Lq > kMhaLmax || Lq < 2 || B <= 0) return 1;
  const int total = B * heads;
  launch_pdl(mha_short_kernel, dim3((total + 3) / 4), dim3(128), 0, st, q, ldq, k, v, ldk, B, Lq, Lk, heads, (__half*)out, ldo,
             split ? heads * 64 : 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(cudaGetErrorString(e));
  count_launch();
  return 0;
}

}  // namespace b2p
