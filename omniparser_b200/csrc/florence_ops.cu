// Non-GEMM kernels of the Florence-2 caption path (ref:util/utils.py:125 -> HF generate): LayerNorm, DaViT
// depthwise conv / window attention / channel attention, BART multi-head attention with KV cache, embedding +
// position + LayerNorm, image-token projector prep, and the greedy token pick with HF logits processors.
// All are HBM/latency-bound SIMT kernels in fp32; the dense contractions run in gemm_tcgen05.cu.
// Residual streams are fp32, GEMM operands fp16.
#include "b2p_internal.h"
#include <atomic>
#include <cuda_fp16.h>
#include <math.h>

namespace b2p {

__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
  for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// fp16 activation store.  split == 0: plain.  split == K > 0: "fp16x3" operand layout [hi(K) | lo(K)] (row stride 2K):
// the GEMM loads both halves of A and of W = [W_hi | W_lo] once per k-block and accumulates hi*hi + hi*lo + lo*hi in
// fp32 (2^-22-class products instead of 2^-11): the parity-grade precision mode of the caption path.
__device__ __forceinline__ void store_act(__half* row, int c, int split, float v) {
  const __half h = __float2half_rn(v);
  row[c] = h;
  if (split) row[split + c] = __float2half_rn(v - __half2float(h));
}

// 4 consecutive channels (c % 4 == 0) as one 8-byte store per copy
__device__ __forceinline__ void store_act4(__half* row, int c, int split, const float4& v) {
  __align__(8) __half2 h[2] = {__floats2half2_rn(v.x, v.y), __floats2half2_rn(v.z, v.w)};
  *reinterpret_cast<uint2*>(row + c) = *reinterpret_cast<const uint2*>(h);
  if (split) {
    const float2 a = __half22float2(h[0]), b = __half22float2(h[1]);
    __align__(8) __half2 l[2] = {__floats2half2_rn(v.x - a.x, v.y - a.y), __floats2half2_rn(v.z - b.x, v.w - b.y)};
    *reinterpret_cast<uint2*>(row + split + c) = *reinterpret_cast<const uint2*>(l);
  }
}

// ---------------------------------------------------------------------------------------- LayerNorm
// one warp per row; x fp32 [T][ldx]; writes fp16 and/or fp32 (nn.LayerNorm, biased variance, eps inside sqrt)
__global__ void layernorm_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ g,
                                 const float* __restrict__ b, float eps, int T, int C, __half* __restrict__ o16,
                                 long long ld16, float* __restrict__ o32, long long ld32, int split) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= T) return;
  const float4* xr = reinterpret_cast<const float4*>(x + (long long)row * ldx);
  const int C4 = C >> 2;
  float4 v[8];   // C <= 1024
  float s = 0.f;
  int n = 0;
  for (int c = lane; c < C4; c += 32, ++n) { v[n] = xr[c]; s += (v[n].x + v[n].y) + (v[n].z + v[n].w); }
  const float mean = warp_sum(s) / float(C);
  float q = 0.f;
  for (int i = 0; i < n; ++i) {
    const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
    q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
  }
  const float rstd = rsqrtf(warp_sum(q) / float(C) + eps);
  n = 0;
  for (int c = lane; c < C4; c += 32, ++n) {
    const float4 gg = reinterpret_cast<const float4*>(g)[c], bb = reinterpret_cast<const float4*>(b)[c];
    float4 y;
    y.x = (v[n].x - mean) * rstd * gg.x + bb.x; y.y = (v[n].y - mean) * rstd * gg.y + bb.y;
    y.z = (v[n].z - mean) * rstd * gg.z + bb.z; y.w = (v[n].w - mean) * rstd * gg.w + bb.w;
    if (o16) store_act4(o16 + (long long)row * ld16, 4 * c, split, y);
    if (o32) reinterpret_cast<float4*>(o32 + (long long)row * ld32)[c] = y;
  }
}

// Fused DaViT pre-block: y = dwconv3x3(x) + bias + x (fp32, the new residual stream) and h = LayerNorm(y) as the next
// GEMM operand.  One warp per token; channels in float4 lanes (C <= 1024).
__global__ void dwconv_ln_kernel(const float* __restrict__ x, int B, int H, int W, int C, const float* __restrict__ w9c,
                                 const float* __restrict__ bias, float* __restrict__ y, const float* __restrict__ g,
                                 const float* __restrict__ bt, float eps, __half* __restrict__ o16, int split) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  const long long tok = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (tok >= (long long)B * H * W) return;
  const int xx = int(tok % W), yy = int((tok / W) % H);
  const int C4 = C >> 2;
  float4 v[8];
  float s = 0.f;
  int n = 0;
  for (int c = lane; c < C4; c += 32, ++n) {
    float4 acc = reinterpret_cast<const float4*>(bias)[c];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int sy = yy + ky - 1;
      if (sy < 0 || sy >= H) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int sx = xx + kx - 1;
        if (sx < 0 || sx >= W) continue;
        const float4 xv = reinterpret_cast<const float4*>(x + (tok + (long long)(ky - 1) * W + (kx - 1)) * C)[c];
        const float4 wv = reinterpret_cast<const float4*>(w9c + (ky * 3 + kx) * C)[c];
        acc.x += xv.x * wv.x; acc.y += xv.y * wv.y; acc.z += xv.z * wv.z; acc.w += xv.w * wv.w;
      }
    }
    const float4 xc = reinterpret_cast<const float4*>(x + tok * C)[c];
    acc.x += xc.x; acc.y += xc.y; acc.z += xc.z; acc.w += xc.w;
    reinterpret_cast<float4*>(y + tok * C)[c] = acc;
    v[n] = acc;
    s += (acc.x + acc.y) + (acc.z + acc.w);
  }
  const float mean = warp_sum(s) / float(C);
  float q = 0.f;
  for (int i = 0; i < n; ++i) {
    const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
    q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
  }
  const float rstd = rsqrtf(warp_sum(q) / float(C) + eps);
  n = 0;
  __half* orow = o16 + tok * (split ? 2 * C : C);
  for (int c = lane; c < C4; c += 32, ++n) {
    const float4 gg = reinterpret_cast<const float4*>(g)[c], bb = reinterpret_cast<const float4*>(bt)[c];
    float4 o;
    o.x = (v[n].x - mean) * rstd * gg.x + bb.x; o.y = (v[n].y - mean) * rstd * gg.y + bb.y;
    o.z = (v[n].z - mean) * rstd * gg.z + bb.z; o.w = (v[n].w - mean) * rstd * gg.w + bb.w;
    store_act4(orow, 4 * c, split, o);
  }
}

// ---------------------------------------------------------------------------------------- window attention
// qkv fp16 [B*H*W][3C] for REAL tokens only.  The reference zero-pads the normed map to a multiple of the 12x12
// window; padded tokens have qkv = bias and take part as keys/values unmasked
// (hf:models/florence2/modeling_florence2.py:346-350,377-383).  Exact shortcut: one "pad key" (k = bias_k,
// v = bias_v) with multiplicity n_pad = 144 - n_real.  One CTA per (batch, window, head); one thread per query.
__global__ void window_attn_kernel(const float* __restrict__ qkv, const float* __restrict__ qkv_bias, int B, int H, int W,
                                   int C, int heads, int win, __half* __restrict__ out, int split, int kv_cap) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  extern __shared__ float4 sm4[];
  constexpr int D = 32, D4 = D / 4;
  const int nwx = (W + win - 1) / win, nwy = (H + win - 1) / win;
  int bid = blockIdx.x;
  const int head = bid % heads; bid /= heads;
  const int wx = bid % nwx; bid /= nwx;
  const int wy = bid % nwy;
  const int b = bid / nwy;
  const int y0 = wy * win, x0 = wx * win;
  const int ny = min(win, H - y0), nx = min(win, W - x0);
  const int nreal = ny * nx, npad = win * win - nreal;
  float4* Ks = sm4;                       // [nreal][D4]
  float4* Vs = sm4 + kv_cap * D4;         // [nreal][D4]; kv_cap = most real tokens any window of this map holds
  for (int i = threadIdx.x; i < nreal * D4; i += blockDim.x) {
    const int t = i / D4, d = i - t * D4;
    const long long tok = ((long long)b * H + y0 + t / nx) * W + x0 + t % nx;
    Ks[i] = reinterpret_cast<const float4*>(qkv + tok * 3 * C + C + head * D)[d];
    Vs[i] = reinterpret_cast<const float4*>(qkv + tok * 3 * C + 2 * C + head * D)[d];
  }
  __syncthreads();
  const float scale = rsqrtf(float(D));
  for (int t = threadIdx.x; t < nreal; t += blockDim.x) {
    const long long tok = ((long long)b * H + y0 + t / nx) * W + x0 + t % nx;
    float4 q[D4], acc[D4];
#pragma unroll
    for (int d = 0; d < D4; ++d) {
      q[d] = reinterpret_cast<const float4*>(qkv + tok * 3 * C + head * D)[d];
      q[d].x *= scale; q[d].y *= scale; q[d].z *= scale; q[d].w *= scale;
      acc[d] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float m = -INFINITY, l = 0.f;
    if (npad > 0) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < D4; ++d) {
        const float4 kb = reinterpret_cast<const float4*>(qkv_bias + C + head * D)[d];
        s += (q[d].x * kb.x + q[d].y * kb.y) + (q[d].z * kb.z + q[d].w * kb.w);
      }
      m = s;
      l = float(npad);
#pragma unroll
      for (int d = 0; d < D4; ++d) {
        const float4 vb = reinterpret_cast<const float4*>(qkv_bias + 2 * C + head * D)[d];
        acc[d] = make_float4(l * vb.x, l * vb.y, l * vb.z, l * vb.w);
      }
    }
    for (int j = 0; j < nreal; ++j) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < D4; ++d) {
        const float4 kk = Ks[j * D4 + d];
        s += (q[d].x * kk.x + q[d].y * kk.y) + (q[d].z * kk.z + q[d].w * kk.w);
      }
      if (s > m) {
        const float r = __expf(m - s);
        l *= r;
#pragma unroll
        for (int d = 0; d < D4; ++d) { acc[d].x *= r; acc[d].y *= r; acc[d].z *= r; acc[d].w *= r; }
        m = s;
      }
      const float p = __expf(s - m);
      l += p;
#pragma unroll
      for (int d = 0; d < D4; ++d) {
        const float4 vv = Vs[j * D4 + d];
        acc[d].x += p * vv.x; acc[d].y += p * vv.y; acc[d].z += p * vv.z; acc[d].w += p * vv.w;
      }
    }
    const float inv = 1.f / l;
    __half* orow = out + tok * (split ? 2 * C : C);
#pragma unroll
    for (int d = 0; d < D4; ++d)
      store_act4(orow, head * D + 4 * d, split, make_float4(acc[d].x * inv, acc[d].y * inv, acc[d].z * inv, acc[d].w * inv));
  }
}

// ---------------------------------------------------------------------------------------- channel attention
// hf:models/florence2/modeling_florence2.py:228-264: per (batch, group) a d x d (d = 32) attention over channels:
// S[i][j] = N^-0.5 * sum_n q[n][i] k[n][j]; P = softmax_j(S); out[n][i] = sum_j P[i][j] v[n][j].
// One CTA (1024 threads = 32 x 32) per (batch, group); tokens streamed through shared memory in chunks.
__global__ void __launch_bounds__(256) channel_attn_kernel(const float* __restrict__ qkv, int N, int C, int groups,
                                                           __half* __restrict__ out, int split) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  constexpr int D = 32, CH = 64;
  __shared__ float qs[CH][D + 1], ks[CH][D + 1];
  __shared__ float P[D][D + 1];
  const int g = blockIdx.x % groups, b = blockIdx.x / groups;
  const int w = threadIdx.x >> 5, j = threadIdx.x & 31;   // warp w owns rows i = 4w .. 4w+3, lane = column j
  const float* base = qkv + (long long)b * N * 3 * C;
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  for (int n0 = 0; n0 < N; n0 += CH) {
    const int cn = min(CH, N - n0);
    for (int t = threadIdx.x; t < cn * D; t += blockDim.x) {
      const int n = t / D, d = t - n * D;
      qs[n][d] = base[(long long)(n0 + n) * 3 * C + g * D + d];
      ks[n][d] = base[(long long)(n0 + n) * 3 * C + C + g * D + d];
    }
    __syncthreads();
    for (int n = 0; n < cn; ++n) {
      const float kv = ks[n][j];
#pragma unroll
      for (int r = 0; r < 4; ++r) s[r] += qs[n][4 * w + r] * kv;
    }
    __syncthreads();
  }
  const float sc = rsqrtf(float(N));
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const float v = s[r] * sc;
    const float m = warp_max(v);
    const float e = __expf(v - m);
    P[4 * w + r][j] = e / warp_sum(e);
  }
  __syncthreads();
  // out[n][g*32 + j] = sum_jj P[j][jj] v[n][jj]: 8 tokens per pass (one per warp), lane = output channel j
  float pr[D];
#pragma unroll
  for (int jj = 0; jj < D; ++jj) pr[jj] = P[j][jj];
  for (int n = w; n < N; n += 8) {
    const float* vr = base + (long long)n * 3 * C + 2 * C + g * D;
    const float vj = vr[j];
    float acc = 0.f;
#pragma unroll
    for (int jj = 0; jj < D; ++jj) acc += pr[jj] * __shfl_sync(0xffffffffu, vj, jj);
    store_act(out + ((long long)b * N + n) * (split ? 2 * C : C), g * D + j, split, acc);
  }
}

// ---------------------------------------------------------------------------------------- BART attention
// One warp per (batch, head, query).  d_head = 64 (2 values per lane), scale applied to q (hf:models/bart/
// modeling_bart.py:143-258).  K/V row b*Lk + j at k + (b*Lk + j)*ldk + h*64.  Decoder self-attention: the current
// step's k, v (columns of the fused qkv GEMM output) are appended to the cache at position *step, and the
// attention covers cache[0..*step].
struct MhaArgs {
  const float* q; long long ldq;
  const float* k; const float* v; long long ldk;     // encoder / cross: [B*Lk][ldk]
  float* kcache; float* vcache; int tmax;             // decoder self: cache [B][tmax][heads*64]
  const float* knew; const float* vnew; long long ldnew;
  const int* step;
  int B, Lq, Lk, heads;
  __half* out; long long ldo; int split;
};

__global__ void mha_kernel(MhaArgs a) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int total = a.B * a.heads * a.Lq;
  if (wid >= total) return;
  const int qi = wid % a.Lq;
  const int h = (wid / a.Lq) % a.heads;
  const int b = wid / (a.Lq * a.heads);
  const int HD = a.heads * 64;
  float2 q = *reinterpret_cast<const float2*>(a.q + ((long long)b * a.Lq + qi) * a.ldq + h * 64 + 2 * lane);
  q.x *= 0.125f; q.y *= 0.125f;
  int Lk = a.Lk;
  const float *kb, *vb;
  long long ldk;
  if (a.kcache) {
    const int t = *a.step;
    // append this step's k, v
    const float2 kn = *reinterpret_cast<const float2*>(a.knew + (long long)b * a.ldnew + h * 64 + 2 * lane);
    const float2 vn = *reinterpret_cast<const float2*>(a.vnew + (long long)b * a.ldnew + h * 64 + 2 * lane);
    *reinterpret_cast<float2*>(a.kcache + ((long long)b * a.tmax + t) * HD + h * 64 + 2 * lane) = kn;
    *reinterpret_cast<float2*>(a.vcache + ((long long)b * a.tmax + t) * HD + h * 64 + 2 * lane) = vn;
    __syncwarp();
    Lk = t + 1;
    kb = a.kcache + (long long)b * a.tmax * HD + h * 64;
    vb = a.vcache + (long long)b * a.tmax * HD + h * 64;
    ldk = HD;
  } else {
    kb = a.k + (long long)b * a.Lk * a.ldk + h * 64;
    vb = a.v + (long long)b * a.Lk * a.ldk + h * 64;
    ldk = a.ldk;
  }
  float m = -INFINITY, l = 0.f;
  float2 acc = make_float2(0.f, 0.f);
  int j = 0;
  // four keys per iteration: 8 independent row loads in flight and four interleaved butterfly reductions (the one-key loop
  // below is a ~700-cycle dependent chain per key: at L = 13 the whole kernel was load-latency bound)
  for (; j + 4 <= Lk; j += 4) {
    float2 kf[4], vf[4];
    float s[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      kf[u] = *reinterpret_cast<const float2*>(kb + (long long)(j + u) * ldk + 2 * lane);
      vf[u] = *reinterpret_cast<const float2*>(vb + (long long)(j + u) * ldk + 2 * lane);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) s[u] = q.x * kf[u].x + q.y * kf[u].y;
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
      acc.x += p * vf[u].x;
      acc.y += p * vf[u].y;
    }
    m = mn;
  }
  for (; j < Lk; ++j) {
    const float2 kf = *reinterpret_cast<const float2*>(kb + j * ldk + 2 * lane);
    const float s = warp_sum(q.x * kf.x + q.y * kf.y);
    const float mn = fmaxf(m, s);
    const float r = __expf(m - mn), p = __expf(s - mn);
    const float2 vf = *reinterpret_cast<const float2*>(vb + j * ldk + 2 * lane);
    l = l * r + p;
    acc.x = acc.x * r + p * vf.x;
    acc.y = acc.y * r + p * vf.y;
    m = mn;
  }
  const float inv = 1.f / l;
  __half* orow = a.out + ((long long)b * a.Lq + qi) * a.ldo;
  store_act(orow, h * 64 + 2 * lane, a.split, acc.x * inv);
  store_act(orow, h * 64 + 2 * lane + 1, a.split, acc.y * inv);
}

// ---------------------------------------------------------------------------------------- embeddings
// Encoder input: row (b, i) = (i < n_img ? image_feat[b][i] : E[prompt[i - n_img]]) + P[i + 2]
// (hf:models/florence2/modeling_florence2.py:742-761; learned positions with offset 2, hf:models/bart/
// modeling_bart.py:74-98).  Decoder input: row b = E[token[b]] + P[*step + 2].  Output fp32 (LayerNorm follows).
__global__ void encoder_embed_kernel(const float* __restrict__ img, int n_img, const float* __restrict__ E,
                                     const int* __restrict__ prompt, int n_prompt, const float* __restrict__ P, int B,
                                     int C, float* __restrict__ out) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  const int L = n_img + n_prompt;
  const long long n = (long long)B * L * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % C);
    const int t = int((i / C) % L);
    const int b = int(i / ((long long)C * L));
    const float e = (t < n_img) ? img[((long long)b * n_img + t) * C + c] : E[(long long)prompt[t - n_img] * C + c];
    out[i] = e + P[(long long)(t + 2) * C + c];
  }
}

__global__ void decoder_embed_kernel(const float* __restrict__ E, const int* __restrict__ seq, int seq_ld,
                                     const int* __restrict__ step, const float* __restrict__ P, int B, int C,
                                     float* __restrict__ out) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  const int t = *step;
  const long long n = (long long)B * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % C);
    const int b = int(i / C);
    out[i] = E[(long long)seq[b * seq_ld + t] * C + c] + P[(long long)(t + 2) * C + c];
  }
}

// Projector prep (hf:models/florence2/modeling_florence2.py:573-595): tokens = x + pos2d + temporal(0);
// rows: [mean over HW] ++ [HW tokens]; fp16 out [B][1+HW][C] feeding the 1024->768 projection GEMM.
__global__ void projector_prep_kernel(const float* __restrict__ x /*[B][HW][C]*/, const float* __restrict__ pos /*[HW][C]*/,
                                      int B, int HW, int C, __half* __restrict__ out, int split) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  const long long n = (long long)B * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = int(i % C);
    const int b = int(i / C);
    float s = 0.f;
    for (int t = 0; t < HW; ++t) {
      const float v = x[((long long)b * HW + t) * C + c] + pos[(long long)t * C + c];
      s += v;
      store_act(out + ((long long)b * (HW + 1) + 1 + t) * (split ? 2 * C : C), c, split, v);
    }
    store_act(out + (long long)b * (HW + 1) * (split ? 2 * C : C), c, split, s / float(HW));
  }
}

// ---------------------------------------------------------------------------------------- greedy pick
// HF greedy step (hf:generation/utils.py:2727-2805) with the processors Florence-2 configures, in HF order:
// no_repeat_ngram (hf:generation/logits_process.py:1012-1079), forced BOS (:1552), forced EOS (:1597); then
// argmax (first maximum), pad for finished rows, EOS bookkeeping.  seq[b][0] = decoder_start; this kernel writes
// seq[b][*step + 1].  One CTA per row.
struct PickArgs {
  const float* logits; long long ld; int V;
  int* seq; int seq_ld;
  int* finished;        // [B]
  const int* step;      // current decoder length - 1
  int ngram, forced_bos, forced_eos, eos, pad, max_len;   // max_len = total sequence length incl. start token
  float* dump;          // optional [B][V] processed scores of this step (parity checks)
  int* n_unfinished;    // device counter, decremented when a row finishes
};

__global__ void __launch_bounds__(1024) greedy_pick_kernel(PickArgs a) {
  pdl_wait();   // PDL: inputs come from the previous kernel in the stream
  const int b = blockIdx.x;
  const int t = *a.step;            // tokens so far = t + 1
  const int cur_len = t + 1;
  const float* lg = a.logits + (long long)b * a.ld;
  int* seq = a.seq + (long long)b * a.seq_ld;
  __shared__ float bv[32];
  __shared__ int bi[32];
  __shared__ int banned[64];
  __shared__ int nbanned;
  if (threadIdx.x == 0) {
    int nb = 0;
    if (a.ngram > 0 && cur_len + 1 >= a.ngram) {
      // ban every token that would complete an n-gram already present in seq[0..cur_len)
      const int pre = a.ngram - 1;
      for (int s = 0; s + a.ngram <= cur_len; ++s) {
        bool eq = true;
        for (int k = 0; k < pre; ++k) eq = eq && (seq[s + k] == seq[cur_len - pre + k]);
        if (eq && nb < 64) banned[nb++] = seq[s + pre];
      }
    }
    nbanned = nb;
  }
  __syncthreads();
  int force = -1;
  if (cur_len == 1 && a.forced_bos >= 0) force = a.forced_bos;
  if (cur_len == a.max_len - 1 && a.forced_eos >= 0) force = a.forced_eos;
  float best = -INFINITY;
  int besti = 0x7fffffff;
  if (a.dump || force < 0) {
    const bool vec = !a.dump && force < 0 && (a.ld % 2 == 0) && ((reinterpret_cast<uintptr_t>(lg) & 7) == 0);
    if (vec) {
      // plain scan; the (<= 19-entry) ban list is only consulted when a value would become the running maximum
      const float2* lp = reinterpret_cast<const float2*>(lg);
      const int V2 = a.V >> 1;
      // four strided loads in flight per thread before the compares (one load per iteration left every thread waiting on an
      // L2 round trip 25 times per row); the compares stay in ascending index order
      for (int v0 = threadIdx.x; v0 < V2; v0 += 4 * blockDim.x) {
        float2 t4[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int v2 = v0 + u * blockDim.x;
          t4[u] = (v2 < V2) ? lp[v2] : make_float2(-INFINITY, -INFINITY);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int v2 = v0 + u * blockDim.x;
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const float sv = e ? t4[u].y : t4[u].x;
            const int v = 2 * v2 + e;
            if (sv > best) {   // ascending v within a thread: ties keep the earlier index
              bool ban = false;
              for (int k = 0; k < nbanned; ++k) ban = ban || (banned[k] == v);
              if (!ban) { best = sv; besti = v; }
            }
          }
        }
      }
      if ((a.V & 1) && threadIdx.x == 0) {
        const int v = a.V - 1;
        const float sv = lg[v];
        bool ban = false;
        for (int k = 0; k < nbanned; ++k) ban = ban || (banned[k] == v);
        if (!ban && sv > best) { best = sv; besti = v; }
      }
    } else {
      for (int v = threadIdx.x; v < a.V; v += blockDim.x) {
        float sv = lg[v];
        for (int k = 0; k < nbanned; ++k) if (banned[k] == v) sv = -INFINITY;
        if (force >= 0) sv = (v == force) ? 0.f : -INFINITY;
        if (a.dump) a.dump[(long long)b * a.V + v] = sv;
        if (sv > best || (sv == best && v < besti)) { best = sv; besti = v; }
      }
    }
  } else if (threadIdx.x == 0) {
    best = 0.f;          // forced token: every other score is -inf (hf:generation/logits_process.py:1552,1597)
    besti = force;
  }
  for (int o = 16; o; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
    if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
  }
  if ((threadIdx.x & 31) == 0) { bv[threadIdx.x >> 5] = best; bi[threadIdx.x >> 5] = besti; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
      if (bv[w] > best || (bv[w] == best && bi[w] < besti)) { best = bv[w]; besti = bi[w]; }
    int tok = besti;
    if (a.finished[b]) tok = a.pad;
    seq[cur_len] = tok;
    if (!a.finished[b] && tok == a.eos) {
      a.finished[b] = 1;
      if (a.n_unfinished) atomicSub(a.n_unfinished, 1);
    }
  }
}

__global__ void step_advance_kernel(int* step) {
  pdl_wait();
  *step += 1;
}

static inline int grid_for(long long n, int threads) {
  long long b = (n + threads - 1) / threads;
  const long long cap = 148LL * 16;
  return int(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace b2p

using namespace b2p;

extern "C" {

int b2p_layernorm(const float* x, long long ldx, const float* gamma, const float* beta, float eps, int T, int C,
                  void* out16, long long ld16, float* out32, long long ld32, int split, cudaStream_t st) {
  if (T <= 0) return 0;
  if (C % 4 || C > 1024 || (ldx % 4) || (ld32 % 4) || (ld16 % 4)) return set_error("layernorm: C, ld must be multiples of 4, C <= 1024");
  const int wpb = 8;
  launch_pdl(layernorm_kernel, dim3((T + wpb - 1) / wpb), dim3(wpb * 32), 0, st, x, ldx, gamma, beta, eps, T, C, (__half*)out16, ld16, out32, ld32, split ? C : 0);
  B2P_CHECK_LAUNCH();
  return 0;
}

int b2p_dwconv_ln(const float* x, int B, int H, int W, int C, const float* w9c, const float* bias, float* y,
                  const float* gamma, const float* beta, float eps, void* out16, int split, cudaStream_t st) {
  if (C % 4 || C > 1024) return set_error("dwconv_ln: C must be a multiple of 4 and <= 1024");
  const long long T = (long long)B * H * W;
  if (split & 4) {   // round-2 strip kernel (florence_simt.cu); shapes it does not cover fall through
    const int r = dwconv_ln_v3_launch(x, B, H, W, C, w9c, bias, y, gamma, beta, eps, out16, split & 1, st);
    if (r <= 0) return r;
  }
  const int wpb = 8;
  launch_pdl(dwconv_ln_kernel, dim3(int((T + wpb - 1) / wpb)), dim3(wpb * 32), 0, st, x, B, H, W, C, w9c, bias, y, gamma, beta, eps, (__half*)out16, (split & 1) ? C : 0);
  B2P_CHECK_LAUNCH();
  return 0;
}

int b2p_window_attn(const float* qkv, const float* qkv_bias, int B, int H, int W, int C, int heads, int win, void* out,
                    int split, cudaStream_t st) {
  if (C / heads != 32) return set_error("window_attn: head_dim must be 32");
  if (split & 4) {   // one-window maps: CTA per (image, head group), florence_simt.cu
    if (int e = bind_device()) return e;
    const int r = window_attn_crop_launch(qkv, qkv_bias, B, H, W, C, heads, win, out, split & 1, st);
    if (r <= 0) return r;
  }
  const int nw = ((W + win - 1) / win) * ((H + win - 1) / win);
  // K/V staging sized by the REAL tokens of a window: the 4x4 / 2x2 maps of the 64x64-crop mode need 4 KB / 1 KB, not the
  // 36.9 KB of a full 12x12 window (which capped those launches at 6 one-warp CTAs per SM: ~100 us each, r1 step table)
  const int kv_cap = (W < win ? W : win) * (H < win ? H : win);
  const size_t smem = size_t(2) * kv_cap * 32 * sizeof(float);
  if (int e = bind_device()) return e;
  static std::atomic<bool> attr{false};
  if (!attr) {
    cudaFuncSetAttribute(window_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    attr = true;
  }
  if (smem > 64 * 1024) return set_error("window_attn: window too large");
  // (two queries per thread measured slower on the 16x16 map, 479 us against 357: 168 registers leave 12 warps per SM)
  // one thread per query of the window: small maps (4x4, 8x8 in the 64x64-crop mode) get small CTAs so more of them fit per SM
  const int nq = kv_cap;
  const int threads = nq >= 160 ? 160 : ((nq + 31) / 32) * 32;
  launch_pdl(window_attn_kernel, dim3(B * nw * heads), dim3(threads), smem, st, qkv, qkv_bias, B, H, W, C, heads, win, (__half*)out, (split & 1) ? C : 0, kv_cap);
  B2P_CHECK_LAUNCH();
  return 0;
}

int b2p_channel_attn(const float* qkv, int B, int N, int C, int groups, void* out, int split, cudaStream_t st) {
  if (C / groups != 32) return set_error("channel_attn: channels per group must be 32");
  if (split & 4) {   // register-tiled kernel, florence_simt.cu
    const int r = channel_attn_v3_launch(qkv, B, N, C, groups, out, split & 1, st);
    if (r <= 0) return r;
  }
  launch_pdl(channel_attn_kernel, dim3(B * groups), dim3(256), 0, st, qkv, N, C, groups, (__half*)out, (split & 1) ? C : 0);
  B2P_CHECK_LAUNCH();
  return 0;
}

// Encoder self-attention / decoder cross-attention: explicit K, V.
int b2p_mha(const float* q, long long ldq, const float* k, const float* v, long long ldk, int B, int Lq, int Lk, int heads,
            void* out, long long ldo, int split, cudaStream_t st) {
  if (split & 4) {   // short sequences: warp per (batch, head) with K / V in registers, florence_simt.cu
    const int r = mha_short_launch(q, ldq, k, v, ldk, B, Lq, Lk, heads, out, ldo, split & 1, st);
    if (r <= 0) return r;
  }
  MhaArgs a{};
  a.q = q; a.ldq = ldq; a.k = k; a.v = v; a.ldk = ldk;
  a.B = B; a.Lq = Lq; a.Lk = Lk; a.heads = heads; a.out = (__half*)out; a.ldo = ldo; a.split = (split & 1) ? heads * 64 : 0;
  const int total = B * heads * Lq;
  // (a thread-per-query variant measured 2.3x slower here: its per-thread 256-B rows are uncoalesced,
  // profiles/r1_step_table_v3.txt, and was removed)
  launch_pdl(mha_kernel, dim3((total + 7) / 8), dim3(256), 0, st, a);
  B2P_CHECK_LAUNCH();
  return 0;
}

// Decoder self-attention step with KV-cache append at position *step.
int b2p_mha_cached(const float* q, long long ldq, const float* knew, const float* vnew, long long ldnew, float* kcache,
                   float* vcache, int tmax, const int* step, int B, int heads, void* out, long long ldo, int split,
                   cudaStream_t st) {
  MhaArgs a{};
  a.q = q; a.ldq = ldq; a.knew = knew; a.vnew = vnew; a.ldnew = ldnew;
  a.kcache = kcache; a.vcache = vcache; a.tmax = tmax; a.step = step;
  a.B = B; a.Lq = 1; a.Lk = 0; a.heads = heads; a.out = (__half*)out; a.ldo = ldo; a.split = split ? heads * 64 : 0;
  const int total = B * heads;
  launch_pdl(mha_kernel, dim3((total + 7) / 8), dim3(256), 0, st, a);
  B2P_CHECK_LAUNCH();
  return 0;
}

int b2p_encoder_embed(const float* img, int n_img, const float* E, const int* prompt, int n_prompt, const float* P,
                      int B, int C, float* out, cudaStream_t st) {
  launch_pdl(encoder_embed_kernel, dim3(grid_for((long long)B * (n_img + n_prompt) * C, 256)), dim3(256), 0, st, img, n_img, E, prompt,
                                                                                            n_prompt, P, B, C, out);
  B2P_CHECK_LAUNCH();
  return 0;
}

int b2p_decoder_embed(const float* E, const int* seq, int seq_ld, const int* step, const float* P, int B, int C,
                      float* out, cudaStream_t st) {
  launch_pdl(decoder_embed_kernel, dim3(grid_for((long long)B * C, 256)), dim3(256), 0, st, E, seq, seq_ld, step, P, B, C, out);
  B2P_CHECK_LAUNCH();
  return 0;
}

int b2p_projector_prep(const float* x, const float* pos, int B, int HW, int C, void* out, int split, cudaStream_t st) {
  launch_pdl(projector_prep_kernel, dim3(grid_for((long long)B * C, 256)), dim3(256), 0, st, x, pos, B, HW, C, (__half*)out, split ? C : 0);
  B2P_CHECK_LAUNCH();
  return 0;
}

int b2p_greedy_pick(const float* logits, long long ld, int V, int B, int* seq, int seq_ld, int* finished,
                    const int* step, int ngram, int forced_bos, int forced_eos, int eos, int pad, int max_len,
                    float* dump, int* n_unfinished, cudaStream_t st) {
  PickArgs a{};
  a.logits = logits; a.ld = ld; a.V = V; a.seq = seq; a.seq_ld = seq_ld; a.finished = finished; a.step = step;
  a.ngram = ngram; a.forced_bos = forced_bos; a.forced_eos = forced_eos; a.eos = eos; a.pad = pad; a.max_len = max_len;
  a.dump = dump; a.n_unfinished = n_unfinished;
  launch_pdl(greedy_pick_kernel, dim3(B), dim3(1024), 0, st, a);
  B2P_CHECK_LAUNCH();
  return 0;
}

int b2p_step_advance(int* step, cudaStream_t st) {
  launch_pdl(step_advance_kernel, dim3(1), dim3(1), 0, st, step);
  B2P_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
