// One persistent, warp-specialised tcgen05 kernel for every dense contraction on the parse hot path:
//   mode 0  C[M,N] = A[M,K] * B[N,K]^T                 (1x1 convs on NHWC, all transformer linears, LM head)
//   mode 1  3x3 stride-1 pad-1 convolution on NHWC      (implicit GEMM: 9 shifted TMA boxes per Cin block)
//   mode 2  3x3 stride-2 pad-1 convolution on NHWC      (implicit GEMM through a 5-D even/odd "parity" view)
// Operands fp16 (or bf16), accumulate fp32 in TMEM, fused epilogue: +bias, SiLU / exact GELU, +residual,
// store fp16 or fp32 into a channel slice (row stride ldc) of the destination so concats are never
// materialised.  Replaces the cuDNN/cuBLAS library kernels behind ref:util/yolov9.py:120-121 (TorchScript
// YOLOv9-E forward) and ref:util/utils.py:125 (Florence-2 generate).
//
// Roles (576 threads): warp 0 = TMA producer (one lane), warp 1 = MMA issuer (one lane), warp 2 also owns TMEM
// alloc/dealloc, warps 2..17 = epilogue (TMEM lane group = warp % 4; the four warps of a group interleave the
// 16-column chunks): the epilogue is latency-bound (dependent MUFU/FP32 chains), so it gets most of the warps.
// Pipelines: smem ring full/empty (TMA <-> MMA), TMEM accumulator double buffer full/empty (MMA <-> epilogue).
#include "ptx.cuh"
#include "b2p_internal.h"
#include <cuda_fp16.h>
#include <math.h>
#include <stdlib.h>
#include <mutex>
#include <atomic>

namespace b2p {

static constexpr int kThreads = 576;      // 2 control warps + 16 epilogue warps
static constexpr int kEpiWarps = 16;
static constexpr int kEpiThreads = kEpiWarps * 32;
static constexpr int kTileM = 128;
static constexpr int kASlot = 16384;    // 128 rows x 128 B
static constexpr int kMaxStages = 8;
static constexpr int kTmemCols = 512;

// q = n / d for 0 <= n < 2^31 by multiply-high + shift (d >= 1), precomputed on the host
struct FastDiv {
  uint32_t mul, shr;
  __host__ static FastDiv make(int d) {
    FastDiv f;
    if (d <= 1) { f.mul = 0; f.shr = 0; return f; }          // shr == 0 marks d == 1
    uint32_t l = 0;
    while ((1u << l) < uint32_t(d)) ++l;                     // ceil(log2 d)
    const unsigned long long m = ((1ull << (32 + l)) + uint32_t(d) - 1) / uint32_t(d);   // ceil(2^(32+l) / d)  (33 bits)
    f.mul = uint32_t(m - (1ull << 32));
    f.shr = l;
    return f;
  }
  __device__ __forceinline__ int div(int n) const {
    if (shr == 0) return n;
    const uint32_t t = __umulhi(uint32_t(n), mul);
    return int((((uint32_t(n) - t) >> 1) + t) >> (shr - 1));   // Granlund-Montgomery round-up method, d in [2, 2^31)
  }
};

struct GemmArgs {
  int mode, M, N, num_kb, bk, bn;
  FastDiv d_ksplit, d_ntiles, d_mtiles, d_perimg, d_tilesx, d_cinb;   // divisors of the item -> tile decode
  int cin_blocks, tw, th, tiles_x, tiles_y, Ho, Wo, batch;
  int m_tiles, n_tiles, stages, ldpar;
  int nb;                // images per tile (small maps: a TMA box spans nb consecutive images)
  int tw_valid;          // valid output columns per tile row (== tw except in halo mode, where tw is the halo pitch)
  int stagesA, cin;      // separate-pipeline modes: A ring depth; Cin
  uint32_t a_slot;       // separate-pipeline modes: bytes per A slot
  // sep: A and B move through SEPARATE pipelines (always in halo mode 3, where one A tile feeds nine weight taps).
  // bres (implies sep): the WHOLE weight matrix of this launch (n_tiles == 1) stays resident in shared memory -- every B
  // k-block is loaded once per CTA, on its first work item, and the persistent loop afterwards streams only A tiles.  For
  // the small-channel layers (N, Cin <= 64..256 on the 160x160 / 80x80 maps: 10+ tiles per CTA) the weight re-loads and
  // their barrier round trips were the per-tile critical path (3.5 us per 128-pixel tile, profiles/r2_notes.md).
  int sep, bres, taps;
  int ksplit, kb_per;    // split-K: work item = (m tile, n tile, k slice); the last CTA to arrive for a tile reduces + stores
  uint32_t a_bytes, b_bytes, b_slot;
  uint32_t idesc;
  uint64_t desc_hi;   // high 32 bits of the smem matrix descriptor (SBO, version, layout), shifted in place
  void* out;
  long long ldc;
  int out_f32;
  const float* bias;
  const void* res;
  long long ldr;
  int act, vec_ok;
  int vec32_ok;   // out / residual rows and the lo planes are 32-byte aligned: 256-bit accesses in the epilogue
  int split;   // > 0: fp16 output in the fp16x3 operand layout: hi at column n, lo at column split + n (lo-plane offset)
  int res_lo;  // > 0: the fp16 residual is a hi/lo pair too, lo at column res_lo + n
  // fp16x3 operands: A rows are [hi(K) | lo(K)] (conv: per pixel [hi(Cin) | lo(Cin)]), W rows [hi | lo] likewise.  Each
  // pipeline stage holds A_hi, A_lo, B_hi, B_lo of ONE logical k-block (each loaded once) and the MMA warp issues the
  // three products hi*hi + hi*lo + lo*hi into the same fp32 accumulator.
  int mt_fast;   // tile order: 1 = M tiles fastest (concurrent CTAs share a B tile: weights larger than activations, e.g. the LM head)
  int x3, lo_a, lo_b, b_tap;   // lo_a / lo_b: column offset of the lo half in A / B; b_tap: B columns per conv tap
  float* ws;   // split-K partial tiles [tile][slice][128][bn] fp32
  int* counters;   // split-K {arrived, finished} counters per output tile (self-resetting)
  int sk_last;     // split-K variant: 1 = last arriver reduces (wait-free, B2P_SPLITK_LAST=1), 0 = distributed reduction
  unsigned long long* trace;   // B2P_TRACE build of the kernel only: [CTA][16] globaltimer stamps (see trace_stamp)
};

// Shared-memory matrix descriptor (PTX ISA "tcgen05 matrix descriptor"), K-major operand, swizzled:
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (=1, unused for swizzled K-major) | [32,46) SBO >> 4
//   [46,48) version = 1 (sm_100) | [61,64) layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B.
// SBO = byte distance between consecutive 8-row groups (8 rows x row pitch).
__host__ __device__ inline uint64_t make_desc_hi(int bk) {
  const uint64_t sbo = (bk == 64) ? 1024 : 512;
  const uint64_t layout = (bk == 64) ? 2 : 4;
  return (uint64_t(1) << 16) | ((sbo >> 4) << 32) | (uint64_t(1) << 46) | (layout << 61);
}
// Instruction descriptor for kind::f16: [4,6) D fmt (1 = f32) | [7,10) A fmt | [10,13) B fmt (0 = f16, 1 = bf16)
//   | bit 15/16 A/B major (0 = K-major) | [17,23) N >> 3 | [24,29) M >> 4.
__host__ inline uint32_t make_idesc(int bn, int bf16, int m = kTileM) {
  uint32_t f = bf16 ? 1u : 0u;
  return (1u << 4) | (f << 7) | (f << 10) | (uint32_t(bn >> 3) << 17) | (uint32_t(m >> 4) << 24);
}

__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float silu_fn(float x) {
  return x * fast_rcp(1.0f + fast_ex2(x * -1.4426950408889634f));   // SiLU: 2 MUFU + 3 FP32, ~2 ulp
}
// exact (erf) GELU, Florence-2 parity: erf by Abramowitz-Stegun 7.1.26 (|err| < 1.5e-7) on MUFU rcp/ex2 instead
// of the ~25-instruction libdevice erff: the GELU epilogues were instruction-bound
__device__ __forceinline__ float gelu_fn(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  const float t = fast_rcp(fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float e = 1.0f - p * t * fast_ex2(z * z * -1.4426950408889634f);   // erf(|x|/sqrt2)
  return 0.5f * x + 0.5f * fabsf(x) * e;                                      // 0.5 x (1 + sign(x) erf)
}
__device__ __forceinline__ float act_fn(float x, int act) {
  if (act == 1) return silu_fn(x);
  if (act == 2) return gelu_fn(x);
  return x;
}
// Activation of 16 accumulator columns.  The switch on the (runtime) activation code sits OUTSIDE the element loop: with
// act_fn(x[j], act) inside it the compiler kept one basic block per element (uniform branch, then the dependent
// FMUL -> MUFU.EX2 -> FADD -> MUFU.RCP -> FMUL chain), so the 16 chains ran back to back at full MUFU latency instead of
// interleaved -- the SiLU / GELU epilogues measured ~2.9x their MUFU-throughput bound (profiles/r2_notes.md 6).
__device__ __forceinline__ void act16(float (&x)[16], int act) {
  if (act == 1) {
#pragma unroll
    for (int j = 0; j < 16; ++j) x[j] = silu_fn(x[j]);
  } else if (act == 2) {
#pragma unroll
    for (int j = 0; j < 16; ++j) x[j] = gelu_fn(x[j]);
  }
}

// 256-bit global accesses (sm_100: LDG/STG.E.ENL2.256): one full 32-byte sector per lane and instruction instead of two
// 16-byte halves -- the epilogue's lane-per-row pattern touches 32 different lines per instruction, so halving the
// instruction count halves its LSU / L2 transaction cost.  Addresses must be 32-byte aligned (GemmArgs::vec32_ok).
__device__ __forceinline__ void st256(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]),
               "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void ld256(const void* p, uint32_t (&v)[8]) {
  asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]),
               "=r"(v[6]), "=r"(v[7]) : "l"(p));
}

struct EpiCtx {
  __half* outh; float* outf; const __half* resh; const float* resf;
};

// bias + activation + residual + store of 16 consecutive output columns [nb, nb+16) of one row.
// pre: bias of the 16 columns already in registers (loaded before the accumulator wait), or nullptr
__device__ __forceinline__ void epi_store16(const GemmArgs& g, const EpiCtx& e, float (&x)[16], int nb, long long pix, bool valid,
                                            const float4* pre = nullptr) {
  const bool full = (nb + 16 <= g.N);
  if (full && g.vec_ok) {
    if (g.bias) {
      const float4* bp = reinterpret_cast<const float4*>(g.bias + nb);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 b = pre ? pre[q] : __ldg(bp + q);
        x[4 * q + 0] += b.x; x[4 * q + 1] += b.y; x[4 * q + 2] += b.z; x[4 * q + 3] += b.w;
      }
    }
    act16(x, g.act);
    if (!valid) return;
    if (g.res) {
      if (g.out_f32) {
        if (g.vec32_ok) {
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            uint32_t t[8];
            ld256(e.resf + pix * g.ldr + nb + 8 * q, t);
#pragma unroll
            for (int k = 0; k < 8; ++k) x[8 * q + k] += __uint_as_float(t[k]);
          }
        } else {
          const float4* rp = reinterpret_cast<const float4*>(e.resf + pix * g.ldr + nb);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 t = rp[q];
            x[4 * q] += t.x; x[4 * q + 1] += t.y; x[4 * q + 2] += t.z; x[4 * q + 3] += t.w;
          }
        }
      } else {
        uint4 rr_[2];
        if (g.vec32_ok) {
          ld256(e.resh + pix * g.ldr + nb, *reinterpret_cast<uint32_t(*)[8]>(rr_));
        } else {
          const uint4* rp = reinterpret_cast<const uint4*>(e.resh + pix * g.ldr + nb);
          rr_[0] = rp[0]; rr_[1] = rp[1];
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const __half2* hp = reinterpret_cast<const __half2*>(&rr_[q]);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float2 f = __half22float2(hp[k]);
            x[8 * q + 2 * k] += f.x;
            x[8 * q + 2 * k + 1] += f.y;
          }
        }
        if (g.res_lo) {
          if (g.vec32_ok) {
            ld256(e.resh + pix * g.ldr + g.res_lo + nb, *reinterpret_cast<uint32_t(*)[8]>(rr_));
          } else {
            const uint4* rl = reinterpret_cast<const uint4*>(e.resh + pix * g.ldr + g.res_lo + nb);
            rr_[0] = rl[0]; rr_[1] = rl[1];
          }
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const __half2* hp = reinterpret_cast<const __half2*>(&rr_[q]);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float2 f = __half22float2(hp[k]);
              x[8 * q + 2 * k] += f.x;
              x[8 * q + 2 * k + 1] += f.y;
            }
          }
        }
      }
    }
    if (g.out_f32) {
      if (g.vec32_ok) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          uint32_t t[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) t[k] = __float_as_uint(x[8 * q + k]);
          st256(e.outf + pix * g.ldc + nb + 8 * q, t);
        }
      } else {
        float4* op = reinterpret_cast<float4*>(e.outf + pix * g.ldc + nb);
#pragma unroll
        for (int q = 0; q < 4; ++q) op[q] = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
      }
    } else {
      uint4 pk[2];
      __half2* hp = reinterpret_cast<__half2*>(pk);
#pragma unroll
      for (int k = 0; k < 8; ++k) hp[k] = __floats2half2_rn(x[2 * k], x[2 * k + 1]);
      if (g.vec32_ok) {
        st256(e.outh + pix * g.ldc + nb, *reinterpret_cast<uint32_t(*)[8]>(pk));
      } else {
        uint4* op = reinterpret_cast<uint4*>(e.outh + pix * g.ldc + nb);
        op[0] = pk[0];
        op[1] = pk[1];
      }
      if (g.split) {
        uint4 lo[2];
        __half2* lp = reinterpret_cast<__half2*>(lo);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float2 hf = __half22float2(hp[k]);
          lp[k] = __floats2half2_rn(x[2 * k] - hf.x, x[2 * k + 1] - hf.y);
        }
        if (g.vec32_ok) {
          st256(e.outh + pix * g.ldc + g.split + nb, *reinterpret_cast<uint32_t(*)[8]>(lo));
        } else {
          uint4* o3 = reinterpret_cast<uint4*>(e.outh + pix * g.ldc + g.split + nb);
          o3[0] = lo[0];
          o3[1] = lo[1];
        }
      }
    }
  } else {
    // ragged tail / unaligned destination: scalar path
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int n = nb + j;
      if (n < g.N) {
        float t = x[j];
        if (g.bias) t += __ldg(g.bias + n);
        t = act_fn(t, g.act);
        if (valid) {
          if (g.res) {
            t += g.out_f32 ? e.resf[pix * g.ldr + n] : __half2float(e.resh[pix * g.ldr + n]);
            if (g.res_lo) t += __half2float(e.resh[pix * g.ldr + g.res_lo + n]);
          }
          if (g.out_f32) e.outf[pix * g.ldc + n] = t;
          else {
            const __half hh = __float2half_rn(t);
            e.outh[pix * g.ldc + n] = hh;
            if (g.split) e.outh[pix * g.ldc + g.split + n] = __float2half_rn(t - __half2float(hh));
          }
        }
      }
    }
  }
}

// Phase stamps of the traced instantiation (B2P_TRACE=1, tools/trace_gemm.py): where a launch's microseconds go.
enum { kTrEntry = 0, kTrPrologue, kTrDepWait, kTrFirstTma, kTrFirstFull, kTrFirstAccDone, kTrFirstEpiStart, kTrLastEpiEnd, kTrExit };
template <bool kTrace>
__device__ __forceinline__ void trace_stamp(const GemmArgs& g, int slot) {
  if constexpr (kTrace) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g.trace[blockIdx.x * 16 + slot] = t;
  }
}

template <bool kTrace>
__device__ __forceinline__ void gemm_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmArgs& g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t a_part = g.x3 ? 2u * kASlot : uint32_t(kASlot);                     // [A_hi][A_lo] | [A]
  const uint32_t stage_bytes = g.sep ? g.b_slot : a_part + (g.x3 ? 2u : 1u) * g.b_slot;
  const uint32_t a_region = g.sep ? uint32_t(g.stagesA) * g.a_slot : 0u;   // separate pipelines: [A slots][B slots]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + a_region + size_t(g.stages) * stage_bytes);
  const uint32_t bar_full = smem_u32(bars);
  const uint32_t bar_empty = bar_full + 8 * g.stages;
  const uint32_t bar_tfull = bar_empty + 8 * g.stages;
  const uint32_t bar_tempty = bar_tfull + 16;
  const uint32_t bar_afull = bar_tempty + 16;              // halo mode only
  const uint32_t bar_aempty = bar_afull + 8 * g.stagesA;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * g.stages + 4 + 2 * g.stagesA);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // Programmatic dependent launch: this grid is persistent (<= one CTA per SM, all resident), so the next kernel in
  // the stream may start launching right away; its CTAs run their prologue on SMs as they free up and then block in
  // griddepcontrol.wait until this grid has completed and flushed.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (threadIdx.x == 0) trace_stamp<kTrace>(g, kTrEntry);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < g.stages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, kEpiWarps);
    }
    for (int a = 0; a < g.stagesA; ++a) {
      mbar_init(bar_afull + 8 * a, 1);
      mbar_init(bar_aempty + 8 * a, 1);
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(tmem_slot), kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) trace_stamp<kTrace>(g, kTrPrologue);
  // everything above touched only this CTA's shared/tensor memory; global reads/writes start below
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (threadIdx.x == 0) trace_stamp<kTrace>(g, kTrDepWait);

  const int total_items = g.m_tiles * g.n_tiles * g.ksplit;   // item = (mt * n_tiles + nt) * ksplit + ks
  const uint32_t smem_base = smem_u32(smem);

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    // Warp-converged like the MMA issuer below: all lanes run the loop and wait on the "empty" barriers, one elected lane
    // issues the TMA instructions; loop state lives in registers, item -> tile coordinates by multiply-shift division.
    const int n_stages = g.stages, n_stagesA = g.stagesA, ksplit = g.ksplit, kb_per = g.kb_per, num_kb = g.num_kb;
    const int mode = g.mode, bk = g.bk, bn = g.bn, cin = g.cin, cin_blocks = g.cin_blocks, b_tap = g.b_tap, ldpar = g.ldpar;
    const int th = g.th, tw_valid = g.tw_valid, nb = g.nb, lo_a = g.lo_a, lo_b = g.lo_b, taps = g.taps;
    const bool sep = g.sep != 0, bres = g.bres != 0, x3 = g.x3 != 0, mt_fast = g.mt_fast != 0;
    const uint32_t a_bytes = g.a_bytes, b_bytes = g.b_bytes, a_slot = g.a_slot, b_slot = g.b_slot;
    const FastDiv d_ksplit = g.d_ksplit, d_ntiles = g.d_ntiles, d_mtiles = g.d_mtiles, d_perimg = g.d_perimg, d_tilesx = g.d_tilesx,
                  d_cinb = g.d_cinb;
    const uint32_t b_base = smem_base + a_region;
    int stage = 0, stageA = 0;
    uint32_t phase = 0, phaseA = 0;
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int tile = d_ksplit.div(item);
      const int ks = item - tile * ksplit;
      int nt, mt;
      if (mt_fast) { nt = d_mtiles.div(tile); mt = tile - nt * g.m_tiles; }
      else { mt = d_ntiles.div(tile); nt = tile - mt * g.n_tiles; }
      const int n0 = nt * bn;
      int img = 0, y0 = 0, x0 = 0;
      if (mode != 0) {
        img = d_perimg.div(mt);
        const int r = mt - img * g.tiles_x * g.tiles_y;
        const int ty = d_tilesx.div(r);
        y0 = ty * th;
        x0 = (r - ty * g.tiles_x) * tw_valid;
        img *= nb;   // nb > 1 only when one tile covers whole images (per_img == 1)
      }
      const int kb0 = ks * kb_per, kb1 = min(num_kb, kb0 + kb_per);
      if (sep) {
        // separate pipelines.  Halo mode (3): ONE (th+2) x (tw+2) input tile per channel block feeds all nine taps (the MMA
        // side shifts the smem descriptor start address by (ky*pitch + kx) rows); only the weights stream per tap.
        // Other modes: one A tile per k-block.  Resident weights (bres): B slot (unit*taps + tap) is filled on this CTA's
        // first item only and never released.
        const bool first_item = (item == int(blockIdx.x));
        for (int u = kb0; u < kb1; ++u) {
          mbar_wait(bar_aempty + 8 * stageA, phaseA ^ 1);
          const uint32_t fa = bar_afull + 8 * stageA;
          const uint32_t dstA = smem_base + uint32_t(stageA) * a_slot;
          mbar_expect_tx_elect(fa, a_bytes);
          int bcol0;
          if (mode == 3) {
            tma_load_4d_elect(dstA, &tmA, fa, u * bk, x0 - 1, y0 - 1, img);
            bcol0 = u * bk;                                   // + tap * cin below
          } else if (mode == 0) {
            tma_load_2d_elect(dstA, &tmA, fa, u * bk, mt * kTileM);
            bcol0 = u * bk;
          } else {
            const int tap = d_cinb.div(u);
            const int c0 = (u - tap * cin_blocks) * bk;
            const int ky = (tap * 11) >> 5, kx = tap - ky * 3;     // tap / 3 for tap in 0..8
            bcol0 = tap * b_tap + c0;
            if (mode == 1) {
              tma_load_4d_elect(dstA, &tmA, fa, c0, x0 + kx - 1, y0 + ky - 1, img);
            } else {
              const int py = (ky != 1), px = (kx != 1);
              const int yo = y0 - (ky == 0), xo = x0 - (kx == 0);
              tma_load_5d_elect(dstA, &tmA, fa, c0 + px * ldpar, xo, py, yo, img);
            }
          }
          if constexpr (kTrace) { if (item == blockIdx.x && u == kb0 && lane == 0) trace_stamp<kTrace>(g, kTrFirstTma); }
          if (++stageA == n_stagesA) { stageA = 0; phaseA ^= 1; }
          if (bres) {
            if (first_item) {
              for (int tap = 0; tap < taps; ++tap) {
                const int slot = (u - kb0) * taps + tap;
                const uint32_t fb = bar_full + 8 * slot;
                mbar_expect_tx_elect(fb, b_bytes);
                tma_load_2d_elect(b_base + uint32_t(slot) * b_slot, &tmB, fb, (mode == 3) ? tap * cin + bcol0 : bcol0, n0);
              }
            }
            continue;
          }
          for (int tap = 0; tap < taps; ++tap) {
            mbar_wait(bar_empty + 8 * stage, phase ^ 1);
            const uint32_t fb = bar_full + 8 * stage;
            mbar_expect_tx_elect(fb, b_bytes);
            tma_load_2d_elect(b_base + uint32_t(stage) * b_slot, &tmB, fb, (mode == 3) ? tap * cin + bcol0 : bcol0, n0);
            if (++stage == n_stages) { stage = 0; phase ^= 1; }
          }
        }
        continue;
      }
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
        const uint32_t fb = bar_full + 8 * stage;
        const uint32_t sa = smem_base + uint32_t(stage) * stage_bytes;
        const uint32_t sb = sa + a_part;
        mbar_expect_tx_elect(fb, x3 ? 2u * (a_bytes + b_bytes) : a_bytes + b_bytes);
        int bcol = kb * bk;
        int tap = 0, c0 = 0, ky = 0, kx = 0;
        if (mode != 0) {
          tap = d_cinb.div(kb);
          c0 = (kb - tap * cin_blocks) * bk;
          ky = (tap * 11) >> 5; kx = tap - ky * 3;
          bcol = tap * b_tap + c0;
        }
        for (int half = 0; half <= int(x3); ++half) {     // half 1 = the lo parts (fp16x3 operands only)
          const uint32_t dst = sa + uint32_t(half) * kASlot;
          const int ca = half * lo_a;
          if (mode == 0) {
            tma_load_2d_elect(dst, &tmA, fb, ca + kb * bk, mt * kTileM);
          } else if (mode == 1) {
            tma_load_4d_elect(dst, &tmA, fb, ca + c0, x0 + kx - 1, y0 + ky - 1, img);
          } else {
            // input row 2*oy + (ky-1): ky=0 -> (oy-1, odd), ky=1 -> (oy, even), ky=2 -> (oy, odd); same in x.
            const int py = (ky != 1), px = (kx != 1);
            const int yo = y0 - (ky == 0), xo = x0 - (kx == 0);
            tma_load_5d_elect(dst, &tmA, fb, ca + c0 + px * ldpar, xo, py, yo, img);
          }
        }
        tma_load_2d_elect(sb, &tmB, fb, bcol, n0);
        if (x3) tma_load_2d_elect(sb + b_slot, &tmB, fb, bcol + lo_b, n0);
        if constexpr (kTrace) { if (item == blockIdx.x && kb == kb0 && lane == 0) trace_stamp<kTrace>(g, kTrFirstTma); }
        if (++stage == n_stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    // The whole warp runs this (warp-uniform) loop and waits on the barriers; one elected lane issues the tensor-core
    // instructions from inside the asm blocks (ptx.cuh umma_*_stage).  Everything the loops need is copied out of the
    // kernel-parameter struct first: with the volatile asm statements in between, the compiler re-read every g.* field
    // from the constant bank on every tap otherwise (92 SASS instructions per tap, ~3.6 us per 128-pixel tile of the
    // 32-channel layers against 0.3 us of tensor work: profiles/r2_notes.md).
    const int n_stages = g.stages, n_stagesA = g.stagesA, ksplit = g.ksplit, kb_per = g.kb_per, num_kb = g.num_kb;
    const bool sep = g.sep != 0, bres = g.bres != 0, halo = (g.mode == 3), x3 = g.x3 != 0, k64 = (g.bk == 64);
    const uint32_t idesc = g.idesc, a_slot = g.a_slot, b_slot = g.b_slot;
    const uint32_t dhi = uint32_t(g.desc_hi >> 32), dlo = uint32_t(g.desc_hi);       // descriptor halves (dlo = the LBO field)
    const uint32_t row_shift = (uint32_t(g.tw) * uint32_t(2 * g.bk)) >> 4, col_shift = uint32_t(2 * g.bk) >> 4;   // halo taps
    const uint32_t b_base = smem_base + a_region;
    int stage = 0, stageA = 0;
    uint32_t phase = 0, phaseA = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    bool b_ready = false;   // resident weights: every slot has landed once the first item has been issued
    auto lo_of = [dlo](uint32_t addr) { return ((addr & 0x3FFFFu) >> 4) | dlo; };
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int ks = (ksplit == 1) ? 0 : item % ksplit;
      const int kb0 = ks * kb_per, kb1 = min(num_kb, kb0 + kb_per);
      mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + uint32_t(acc * 256);
      uint32_t accum = 0;   // the first MMA of an item overwrites the accumulator
      if (sep) {
        for (int u = kb0; u < kb1; ++u) {
          mbar_wait(bar_afull + 8 * stageA, phaseA);
          tc_fence_after();
          const uint32_t a0 = lo_of(smem_base + uint32_t(stageA) * a_slot);
          if constexpr (kTrace) { if (item == blockIdx.x && u == kb0 && lane == 0) trace_stamp<kTrace>(g, kTrFirstFull); }
          const int taps_y = halo ? 3 : 1;
          int slot = bres ? (u - kb0) * (halo ? 9 : 1) : stage;
          for (int ky = 0; ky < taps_y; ++ky) {
            for (int kx = 0; kx < taps_y; ++kx) {
              if (!b_ready) {
                // resident weights: slot (unit, tap) completes its one and only phase (parity 0) during the first item
                mbar_wait(bar_full + 8 * slot, bres ? 0u : phase);
                tc_fence_after();
              }
              // halo mode: shifted view of the halo tile.  The 128B/64B swizzle pattern is anchored at the 1024-B aligned slot
              // base (that is how TMA wrote it), so the "matrix base offset" field stays 0 even though the start address
              // points into the middle of an atom: the XOR phase is taken from the address bits, as for the K-advance.
              const uint32_t a_lo = a0 + uint32_t(ky) * row_shift + uint32_t(kx) * col_shift;
              const uint32_t b_lo = lo_of(b_base + uint32_t(slot) * b_slot);
              if (k64) umma_f16_stage<4>(d_tmem, a_lo, b_lo, dhi, idesc, accum);
              else umma_f16_stage<2>(d_tmem, a_lo, b_lo, dhi, idesc, accum);
              accum = 1;
              if (bres) {
                ++slot;
              } else {
                umma_commit_elect(bar_empty + 8 * stage);
                if (++stage == n_stages) { stage = 0; phase ^= 1; }
                slot = stage;
              }
            }
          }
          umma_commit_elect(bar_aempty + 8 * stageA);
          if (++stageA == n_stagesA) { stageA = 0; phaseA ^= 1; }
        }
        if (bres) b_ready = true;
      } else {
        const uint32_t stage_bytes_ = stage_bytes;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(bar_full + 8 * stage, phase);
          tc_fence_after();
          if constexpr (kTrace) { if (item == blockIdx.x && kb == kb0 && lane == 0) trace_stamp<kTrace>(g, kTrFirstFull); }
          const uint32_t sa = smem_base + uint32_t(stage) * stage_bytes_;
          const uint32_t sb = sa + a_part;
          if (x3) {
            // advancing K inside the swizzle span = +32 B on the start address (encoded >> 4)
            if (k64) umma_f16x3_stage<4>(d_tmem, lo_of(sa), lo_of(sa + kASlot), lo_of(sb), lo_of(sb + b_slot), dhi, idesc, accum);
            else umma_f16x3_stage<2>(d_tmem, lo_of(sa), lo_of(sa + kASlot), lo_of(sb), lo_of(sb + b_slot), dhi, idesc, accum);
          } else {
            if (k64) umma_f16_stage<4>(d_tmem, lo_of(sa), lo_of(sb), dhi, idesc, accum);
            else umma_f16_stage<2>(d_tmem, lo_of(sa), lo_of(sb), dhi, idesc, accum);
          }
          accum = 1;
          umma_commit_elect(bar_empty + 8 * stage);
          if (++stage == n_stages) { stage = 0; phase ^= 1; }
        }
      }
      umma_commit_elect(bar_tfull + 8 * acc);
      if constexpr (kTrace) { if (item == blockIdx.x && lane == 0) trace_stamp<kTrace>(g, kTrFirstAccDone); }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else {
    // -------------------------------------------------------------- epilogue (16 warps: 128 TMEM lanes x 4 column phases)
    const int grp = warp & 3;
    const int cq = (warp - 2) >> 2;      // this warp owns the 16-column chunks cq, cq + 4, cq + 8, ...
    int acc = 0;
    uint32_t acc_phase = 0;
    EpiCtx e;
    e.outh = reinterpret_cast<__half*>(g.out);
    e.outf = reinterpret_cast<float*>(g.out);
    e.resh = reinterpret_cast<const __half*>(g.res);
    e.resf = reinterpret_cast<const float*>(g.res);
    // this thread's row of the tile: its position inside the (tw x th [x nb images]) tile never changes
    const int r = grp * 32 + lane;
    const int e_mode = g.mode, e_ksplit = g.ksplit, e_bn = g.bn, e_th = g.th, e_twv = g.tw_valid, e_nb = g.nb;
    const int e_Ho = g.Ho, e_Wo = g.Wo, e_batch = g.batch, e_tiles_x = g.tiles_x, e_per_img = g.tiles_x * g.tiles_y;
    const bool e_mtfast = g.mt_fast != 0;
    const FastDiv e_dks = g.d_ksplit, e_dnt = g.d_ntiles, e_dmt = g.d_mtiles, e_dpi = g.d_perimg, e_dtx = g.d_tilesx;
    int r_sub = 0, r_ty = 0, r_tx = 0;
    if (e_mode != 0) {
      const int rows_img = g.tw * g.th;                  // rows of one image inside the tile
      r_sub = (e_nb > 1) ? r / rows_img : 0;
      const int rloc = r - r_sub * rows_img;
      r_ty = rloc / g.tw;
      r_tx = rloc - r_ty * g.tw;
    }
    const bool r_ok = (r_sub < e_nb) && (r_ty < e_th) && (r_tx < e_twv);
    for (int item = blockIdx.x; item < total_items; item += gridDim.x) {
      const int tile = e_dks.div(item);
      const int ks = item - tile * e_ksplit;
      int nt, mt;
      if (e_mtfast) { nt = e_dmt.div(tile); mt = tile - nt * g.m_tiles; }
      else { mt = e_dnt.div(tile); nt = tile - mt * g.n_tiles; }
      const int n0 = nt * e_bn;
      long long pix;
      bool valid;
      if (e_mode == 0) {
        pix = (long long)mt * kTileM + r;
        valid = pix < g.M;
      } else {
        const int img0 = e_dpi.div(mt);
        const int rr = mt - img0 * e_per_img;
        const int img = img0 * e_nb + r_sub;
        const int tyi = e_dtx.div(rr);
        const int oy = tyi * e_th + r_ty;
        const int ox = (rr - tyi * e_tiles_x) * e_twv + r_tx;
        valid = r_ok && (img < e_batch) && (oy < e_Ho) && (ox < e_Wo);
        pix = ((long long)img * e_Ho + oy) * e_Wo + ox;
      }
      mbar_wait(bar_tfull + 8 * acc, acc_phase);
      tc_fence_after();
      if constexpr (kTrace) { if (item == blockIdx.x && threadIdx.x == 64) trace_stamp<kTrace>(g, kTrFirstEpiStart); }
      const uint32_t t_row = tmem_base + (uint32_t(grp * 32) << 16) + uint32_t(acc * 256);
      if (e_ksplit == 1) {
        // the accumulator goes back to the MMA warp as soon as this warp's LAST 16-column chunk sits in registers (before it
        // is processed).  (A software-pipelined variant with two register buffers measured no faster and spilled.)
        bool released = false;
        for (int c = cq * 16; c < e_bn; c += 64) {
          uint32_t v[16];
          tmem_ld16(t_row + c, v);
          tmem_ld_wait(v);
          if (c + 64 >= e_bn) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
            released = true;
          }
          if (n0 + c >= g.N) continue;   // warp-uniform
          float x[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) x[j] = __uint_as_float(v[j]);
          // (loading the chunk's bias before the TMEM wait was measured: forward 4.77 -> 5.19 ms, the extra live registers spill)
          epi_store16(g, e, x, n0 + c, pix, valid);
        }
        if (!released) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
        }
      } else {
        // split-K: every slice stores its raw fp32 partial tile, then the partials are summed in slice order (deterministic) and
        // the epilogue runs -- by the last CTA to arrive (sk_last: nobody waits for anybody, so partially resident grids cannot
        // deadlock) or, by default, distributed over the tile's ksplit CTAs (faster, see below).
        float* wsp = g.ws + ((size_t(tile) * e_ksplit + ks) * kTileM + r) * e_bn;
        for (int c = cq * 16; c < e_bn; c += 64) {
          uint32_t v[16];
          tmem_ld16(t_row + c, v);
          tmem_ld_wait(v);
          float4* wp = reinterpret_cast<float4*>(wsp + c);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            wp[q] = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
        if (g.sk_last) {
          __threadfence();
          asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
          volatile uint32_t* s_last = tmem_slot + 1;
          if (threadIdx.x == 64) {
            int* cnt = g.counters + 2 * tile;
            const bool last = (atomicAdd(cnt, 1) == e_ksplit - 1);
            if (last) *cnt = 0;   // every slice has arrived: the next user of this counter is a later launch / graph replay
            *s_last = last ? 1u : 0u;
          }
          asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
          if (*s_last) {
            __threadfence();
            const int chunks = e_bn >> 4;
            const float* base = g.ws + size_t(tile) * e_ksplit * kTileM * e_bn;
            int img0 = 0, rr = 0, tyi = 0;
            if (e_mode != 0) {
              img0 = e_dpi.div(mt);
              rr = mt - img0 * e_per_img;
              tyi = e_dtx.div(rr);
            }
            const int rows_img = g.tw * g.th, tw_ = g.tw;
            for (int w = (threadIdx.x - 64); w < kTileM * chunks; w += kEpiThreads) {
              const int rr_ = w / chunks, c = (w - rr_ * chunks) << 4;
              if (n0 + c >= g.N) continue;
              long long pix2;
              bool valid2;
              if (e_mode == 0) {
                pix2 = (long long)mt * kTileM + rr_;
                valid2 = pix2 < g.M;
              } else {
                const int sub = (e_nb > 1) ? rr_ / rows_img : 0;
                const int rloc = rr_ - sub * rows_img;
                const int img = img0 * e_nb + sub;
                const int ty = rloc / tw_, tx = rloc - ty * tw_;
                const int oy = tyi * e_th + ty;
                const int ox = (rr - tyi * e_tiles_x) * e_twv + tx;
                valid2 = (sub < e_nb) && (img < e_batch) && (ty < e_th) && (tx < e_twv) && (oy < e_Ho) && (ox < e_Wo);
                pix2 = ((long long)img * e_Ho + oy) * e_Wo + ox;
              }
              float x[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) x[j] = 0.f;
              for (int sidx = 0; sidx < e_ksplit; ++sidx) {
                const float4* pp = reinterpret_cast<const float4*>(base + (size_t(sidx) * kTileM + rr_) * e_bn + c);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const float4 t = __ldcg(pp + q);
                  x[4 * q] += t.x; x[4 * q + 1] += t.y; x[4 * q + 2] += t.z; x[4 * q + 3] += t.w;
                }
              }
              epi_store16(g, e, x, n0 + c, pix2, valid2);
            }
          }
        } else {
          // default: DISTRIBUTED reduction -- each of the ksplit CTAs of a tile waits for the tile's arrival counter and then
          // reduces its share of the 128 rows (slice order => deterministic sums).  Measured 10-45 % faster per split-K launch
          // than the wait-free variant above (one CTA re-reads all partials at the per-SM L2 rate), at the price of an
          // inter-CTA wait: safe because the grid is at most one wave and the hardware dispatches the CTAs of an earlier
          // launch before those of later ones (tools/coop_test, profiles/r2_notes.md 5); a wait longer than 2 s traps.
          __threadfence();
          asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
          int* cnt = g.counters + 2 * tile;
          if (threadIdx.x == 64) {
            atomicAdd(cnt, 1);
            long long t0 = clock64();
            while (*reinterpret_cast<volatile int*>(cnt) < g.ksplit) {
              if (clock64() - t0 > 4000000000LL) { printf("b2p: split-K arrival timeout (tile %d)\n", tile); __trap(); }
            }
          }
          asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
          __threadfence();
          const int rows_per = (kTileM + g.ksplit - 1) / g.ksplit;
          const int row0 = ks * rows_per, row1 = min(kTileM, row0 + rows_per);
          const int chunks = g.bn >> 4;
          const float* base = g.ws + size_t(tile) * g.ksplit * kTileM * g.bn;
          for (int w = (threadIdx.x - 64); w < (row1 - row0) * chunks; w += kEpiThreads) {
            const int rr_ = row0 + w / chunks, c = (w % chunks) << 4;
            if (n0 + c >= g.N) continue;
            long long pix2;
            bool valid2;
            if (g.mode == 0) {
              pix2 = (long long)mt * kTileM + rr_;
              valid2 = pix2 < g.M;
            } else {
              const int per_img = g.tiles_x * g.tiles_y;
              const int img0 = mt / per_img;
              const int rr = mt - img0 * per_img;
              const int rows_img = g.tw * g.th;
              const int sub = (g.nb > 1) ? rr_ / rows_img : 0;
              const int rloc = rr_ - sub * rows_img;
              const int img = img0 * g.nb + sub;
              const int ty = rloc / g.tw, tx = rloc - ty * g.tw;
              const int oy = (rr / g.tiles_x) * g.th + ty;
              const int ox = (rr % g.tiles_x) * g.tw_valid + tx;
              valid2 = (sub < g.nb) && (img < g.batch) && (ty < g.th) && (tx < g.tw_valid) && (oy < g.Ho) && (ox < g.Wo);
              pix2 = ((long long)img * g.Ho + oy) * g.Wo + ox;
            }
            float x[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = 0.f;
            // two slices per round trip: the loads of both are in flight before the first add (one slice at a time cost one L2
            // latency per slice: 4 us of the 8.8 us fc2 epilogue at split 6); the adds keep the slice order
            const size_t sl_stride = size_t(kTileM) * g.bn;
            const float* pbase = base + size_t(rr_) * g.bn + c;
            int sidx = 0;
            for (; sidx + 2 <= g.ksplit; sidx += 2) {
              const float4* p0 = reinterpret_cast<const float4*>(pbase + size_t(sidx) * sl_stride);
              const float4* p1 = reinterpret_cast<const float4*>(pbase + size_t(sidx + 1) * sl_stride);
              float4 t0[4], t1[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) { t0[q] = __ldcg(p0 + q); t1[q] = __ldcg(p1 + q); }
#pragma unroll
              for (int q = 0; q < 4; ++q) { x[4 * q] += t0[q].x; x[4 * q + 1] += t0[q].y; x[4 * q + 2] += t0[q].z; x[4 * q + 3] += t0[q].w; }
#pragma unroll
              for (int q = 0; q < 4; ++q) { x[4 * q] += t1[q].x; x[4 * q + 1] += t1[q].y; x[4 * q + 2] += t1[q].z; x[4 * q + 3] += t1[q].w; }
            }
            if (sidx < g.ksplit) {
              const float4* pp = reinterpret_cast<const float4*>(pbase + size_t(sidx) * sl_stride);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 t = __ldcg(pp + q);
                x[4 * q] += t.x; x[4 * q + 1] += t.y; x[4 * q + 2] += t.z; x[4 * q + 3] += t.w;
              }
            }
            epi_store16(g, e, x, n0 + c, pix2, valid2);
          }
          asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
          if (threadIdx.x == 64) {
            // the last CTA to finish its share resets both counters for the next launch / graph replay
            if (atomicAdd(cnt + 1, 1) == g.ksplit - 1) { cnt[1] = 0; cnt[0] = 0; __threadfence(); }
          }
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if constexpr (kTrace) { if (threadIdx.x == 64) trace_stamp<kTrace>(g, kTrLastEpiEnd); }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
  if (threadIdx.x == 0) trace_stamp<kTrace>(g, kTrExit);
}

__global__ void __launch_bounds__(kThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs g) {
  gemm_body<false>(tmA, tmB, g);
}

// Same kernel with globaltimer stamps at the phase boundaries (selected by B2P_TRACE=1; never used otherwise).
__global__ void __launch_bounds__(kThreads, 1)
gemm_tcgen05_kernel_trace(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmArgs g) {
  gemm_body<true>(tmA, tmB, g);
}

// ------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

static int encode(CUtensorMap* m, int bf16, int rank, const void* base, const cuuint64_t* dims,
                  const cuuint64_t* strides_bytes, const cuuint32_t* box, int bk) {
  EncodeTiledFn fn = get_encode();
  if (!fn) return set_error("cuTensorMapEncodeTiled entry point unavailable");
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank,
                  const_cast<void*>(base), dims, strides_bytes, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  bk == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[256];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed: CUresult %d (rank %d, dims %llu %llu, box %u %u)", int(r),
             rank, (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
    return set_error(buf);
  }
  return 0;
}

static int g_num_sms = 0;
// Split-K scratch is per stream (two streams may run split-K GEMMs concurrently): a few slots are allocated up
// front (never inside a graph capture) and handed to streams in order of first use.
static constexpr int kWsSlots = 24;
static float* g_ws[kWsSlots] = {};
static int* g_counters[kWsSlots] = {};
static cudaStream_t g_ws_owner[kWsSlots] = {};
static int g_ws_used = 0;
static std::mutex g_ws_mu;
static int ws_slot_for(cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_ws_mu);
  for (int i = 0; i < g_ws_used; ++i)
    if (g_ws_owner[i] == st) return i;
  if (g_ws_used < kWsSlots) { g_ws_owner[g_ws_used] = st; return g_ws_used++; }
  return -1;   // more concurrent streams than slots: the caller disables split-K for this launch
}
static constexpr size_t kWsBytes = size_t(64) << 20;     // split-K partial tiles (per slot)
static constexpr int kMaxCounterTiles = 1 << 12;   // split-K only ever covers < #SMs tiles

static int g_max_smem = 0;

// B2P_TRACE=1 (debugging aid, tools/trace_gemm.py): launches go through gemm_tcgen05_kernel_trace and leave per-CTA
// globaltimer stamps; b2p_trace_read() hands them out together with the launch shapes.
static constexpr int kTraceCap = 1024, kTraceCtas = 160, kTraceSlots = 16;
static unsigned long long* g_trace = nullptr;
static int g_trace_n = 0;
static int g_trace_meta[kTraceCap][8];
static std::mutex g_trace_mu;

static std::mutex g_setup_mu;
static int device_setup() {
  if (int e = bind_device()) return e;
  std::lock_guard<std::mutex> lk(g_setup_mu);
  if (g_num_sms) return 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return set_error("cudaGetDevice failed (no CUDA device?)");
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) return set_error("cudaGetDeviceProperties failed");
  if (p.major != 10) return set_error("libb200parse requires an sm_100 (Blackwell B200) device");
  g_num_sms = p.multiProcessorCount;
  g_max_smem = int(p.sharedMemPerBlockOptin);
  if (cudaFuncSetAttribute(gemm_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, g_max_smem) != cudaSuccess)
    return set_error("cudaFuncSetAttribute(max dynamic smem) failed");
  if (getenv("B2P_TRACE")) {
    if (cudaFuncSetAttribute(gemm_tcgen05_kernel_trace, cudaFuncAttributeMaxDynamicSharedMemorySize, g_max_smem) != cudaSuccess ||
        cudaMalloc(&g_trace, sizeof(unsigned long long) * kTraceCap * kTraceCtas * kTraceSlots) != cudaSuccess)
      return set_error("B2P_TRACE: setup of the traced kernel failed");
    cudaMemset(g_trace, 0, sizeof(unsigned long long) * kTraceCap * kTraceCtas * kTraceSlots);
  }
  for (int i = 0; i < kWsSlots; ++i) {
    if (cudaMalloc(&g_ws[i], kWsBytes) != cudaSuccess || cudaMalloc(&g_counters[i], 2 * kMaxCounterTiles * sizeof(int)) != cudaSuccess)
      return set_error("cudaMalloc for the split-K workspace failed");
    cudaMemset(g_counters[i], 0, 2 * kMaxCounterTiles * sizeof(int));
  }
  return 0;
}


// Choose the N tile and the split-K factor with a small time model (microseconds per CTA):
//   per k-block  max(MMA issue, smem fill): MMA = bn*bk/32 cycles at ~1.9 GHz; fill = (A + B bytes) / ~70 GB/s per SM
//   (measured: L2 -> SM delivery tops out near 12 TB/s chip-wide, profiles/r1_gemm_notes.md)
//   per item     ~2.5 us pipeline fill/drain + epilogue (~0.012 us per output column) + split-K partial store/reduce.
static void pick_tiling(int N, int m_tiles, int num_kb, int bk, uint32_t a_bytes, int bn_max, bool allow_split, bool x3,
                        int* bn_out, int* ksplit_out) {
  static const int cand[] = {256, 192, 128, 96, 64, 48, 32, 16};
  // single-wave launches: measured constants + a charge per occupied SM (B2P_DENSE_GRIDS=1 restores the round-1 model that
  // spreads every launch over as many SMs as it can; B2P_CTA_PENALTY = microseconds charged per CTA, default 0.02: with the
  // grouped caption schedule of the second half of round 2, 0.02 / 0.04 / 0.08 / dense grids measured 14.42 / 14.54 / 14.82 /
  // 14.63 ms per step and 4.47 / 4.73 / 4.90 / 4.43 ms per stand-alone detector forward)
  static const bool few_ctas = getenv("B2P_DENSE_GRIDS") == nullptr;
  static const double cta_penalty = getenv("B2P_CTA_PENALTY") ? atof(getenv("B2P_CTA_PENALTY")) : 0.02;
  const int n16 = (N + 15) / 16 * 16;
  double best_cost = -1;
  int best = 16, best_ks = 1;
  for (int c : cand) {
    if (c > bn_max) continue;
    if (c > n16 && c != 16) {
      bool smaller_covers = false;
      for (int d : cand) if (d < c && d >= n16) smaller_covers = true;
      if (smaller_covers) continue;
    }
    const long n_tiles = (N + c - 1) / c;
    const long tiles = n_tiles * m_tiles;
    // fp16x3 operands: three MMAs and two (hi, lo) tile pairs per logical k-block
    const double t_mma = (x3 ? 3.0 : 1.0) * double(c) * bk / 32.0 / 1900.0;
    const double t_fill = (x3 ? 2.0 : 1.0) * (double(a_bytes) + double(c) * bk * 2.0) / 70000.0;
    if (x3 && 2 * (2 * kASlot + 2 * ((c * bk * 2 + 1023) & ~1023)) + 2048 > g_max_smem) continue;   // needs >= 2 stages
    const double t_kb = t_mma > t_fill ? t_mma : t_fill;
    int max_ks = 1;
    if (allow_split && tiles * 2 <= g_num_sms && tiles * 2 <= kMaxCounterTiles) {
      max_ks = int(g_num_sms / tiles);          // one wave of (tile, slice) items (a performance choice: nothing spins)
      if (max_ks > num_kb / 2) max_ks = num_kb / 2;
      if (max_ks > 32) max_ks = 32;
      if (max_ks < 1) max_ks = 1;
    }
    for (int ks = 1; ks <= max_ks; ++ks) {
      const int kb_per = (num_kb + ks - 1) / ks;
      const int ks_eff = (num_kb + kb_per - 1) / kb_per;
      if (ks_eff != ks) continue;
      if (ks > 1 && size_t(tiles) * ks * 128 * c * 4 > kWsBytes) continue;
      const long items = tiles * ks;
      const long waves = (items + g_num_sms - 1) / g_num_sms;
      // split-K overhead: store one fp32 partial tile + read one tile's worth back (distributed reduce) at ~100 GB/s/SM
      double t_split = ks > 1 ? 2.0 + 2.0 * (128.0 * c * 4.0 / 100000.0) : 0.0;
      double t_kb_ = t_kb;
      double occupancy_penalty = 0.0;
      if (few_ctas && waves == 1) {
        // measured (profiles/r2_notes.md 2): a single-wave launch takes ~11 us whatever its tiling (split-K's store / arrive /
        // reduce costs ~6 us, a CTA of a sparse grid fills at ~100 GB/s), so equal-latency tilings are resolved by a charge per
        // occupied SM: the sparser grid leaves SMs to the other streams of the pipelined parser (bench: 19.2 -> 18.1 ms/step)
        if (ks > 1) t_split = 5.0 + double(ks) * (128.0 * c * 4.0 / 100000.0);
        if (items < 128) t_kb_ = t_mma > t_fill * 0.7 ? t_mma : t_fill * 0.7;
        occupancy_penalty = cta_penalty * double(items);
      }
      const double per_item = 2.5 + kb_per * t_kb_ + 0.012 * c + t_split;
      const double cost = waves * per_item + occupancy_penalty;
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = c; best_ks = ks; }
    }
  }
  *bn_out = best;
  *ksplit_out = best_ks;
}

int gemm_launch(const ConvGemm& d, cudaStream_t st) {
  if (int e = device_setup()) return e;
  GemmArgs g{};
  CUtensorMap tmA, tmB;
  const int Ktot = (d.mode == 0) ? d.K : 9 * d.Cin;
  const int kred = (d.mode == 0) ? d.K : d.Cin;
  const int bk = (kred % 64 == 0) ? 64 : 32;
  if (d.mode != 0 && kred % 32 != 0) return set_error("conv3x3: Cin must be a multiple of 32");
  if (d.mode == 0 && (d.K % 8 != 0 || d.lda % 8 != 0)) return set_error("gemm: K and lda must be multiples of 8");
  if ((reinterpret_cast<uintptr_t>(d.A) & 15) || (reinterpret_cast<uintptr_t>(d.B) & 15)) return set_error("gemm: operands must be 16-byte aligned");
  static const bool no_halo = getenv("B2P_NO_HALO") != nullptr;
  static const bool no_halo32 = getenv("B2P_NO_HALO32") != nullptr;
  const bool halo = (d.mode == 1) && !no_halo && (bk == 64 || !no_halo32) && !d.x3;
  if (d.x3 && (kred % bk != 0)) return set_error("gemm: fp16x3 operands need K (Cin) to be a multiple of 32");
  if (d.x3 && d.bf16) return set_error("gemm: fp16x3 operands are fp16");
  const int xk = d.x3 ? 2 : 1;   // operand rows carry [hi | lo]
  g.x3 = d.x3 ? 1 : 0;
  // lo-plane offset of A: [hi(K) | lo(K)] rows by default; a channel slice of a wider [hi(Ctot) | lo(Ctot)] pixel passes Ctot
  const long long lo_a = d.x3 ? (d.lo_a > 0 ? d.lo_a : (long long)kred) : 0;
  const long long a_span = d.x3 ? lo_a + kred : (long long)kred;   // columns of A the tensor map must cover
  if (d.x3 && (lo_a % 8 != 0 || lo_a < kred)) return set_error("gemm: fp16x3 lo-plane offset of A must be a multiple of 8 and >= K");
  g.lo_a = int(lo_a); g.lo_b = kred;
  g.b_tap = xk * d.Cin;
  g.mode = halo ? 3 : d.mode;
  g.N = d.N;
  g.bk = bk;
  g.cin = d.Cin;
  g.desc_hi = make_desc_hi(bk);
  g.out = d.out; g.ldc = d.ldc; g.out_f32 = d.out_f32; g.bias = d.bias; g.res = d.res; g.ldr = d.ldr; g.act = d.act;
  g.split = (d.split_out && !d.out_f32) ? int(d.lo_out > 0 ? d.lo_out : d.N) : 0;
  if (g.split && ((d.N % 8) || (g.split % 8))) return set_error("gemm: split (fp16x3) output needs N % 8 == 0 and an 8-aligned lo-plane offset");
  if (g.split && (g.split < d.N || d.ldc < (long long)g.split + d.N)) return set_error("gemm: split (fp16x3) output rows are [hi(N) .. | lo(N) ..]: ldc must be >= lo offset + N");
  g.res_lo = (d.res && !d.out_f32 && d.lo_res > 0) ? int(d.lo_res) : 0;
  if (g.res_lo % 8) return set_error("gemm: residual lo-plane offset must be a multiple of 8");

  if (d.mode == 0) {
    g.M = d.M;
    g.tw_valid = 0;
    g.num_kb = (d.K + bk - 1) / bk;
    g.m_tiles = (d.M + kTileM - 1) / kTileM;
    g.a_bytes = kTileM * bk * 2;
    cuuint64_t dims[2] = {cuuint64_t(a_span), cuuint64_t(d.M)};
    cuuint64_t str[1] = {cuuint64_t(d.lda) * 2};
    cuuint32_t box[2] = {cuuint32_t(bk), cuuint32_t(kTileM)};
    if (d.x3 && d.lda < a_span) return set_error("gemm: fp16x3 A rows are [hi(K) .. | lo(K) ..]: lda must be >= lo offset + K");
    if (int e = encode(&tmA, d.bf16, 2, d.A, dims, str, box, bk)) return e;
  } else {
    const int s = (d.mode == 2) ? 2 : 1;
    if (s == 2 && ((d.H & 1) || (d.W & 1))) return set_error("conv3x3 s2: H and W must be even");
    if (d.lda % 8 != 0) return set_error("conv3x3: input pixel stride must be a multiple of 8 channels");
    if (d.x3 && d.lda < a_span) return set_error("conv3x3: fp16x3 pixels are [hi(Cin) .. | lo(Cin) ..]: pixel stride must be >= lo offset + Cin");
    g.Ho = d.H / s; g.Wo = d.W / s; g.batch = d.batch;
    g.cin_blocks = d.Cin / bk;
    g.num_kb = 9 * g.cin_blocks;
    // spatial tile tw x th <= 128 output pixels: maximise useful rows per 128-row MMA tile
    int btw = 1, bth = 1; double bu = -1;
    for (int tw = 1; tw <= g.Wo && tw <= 128; ++tw) {
      int th = 128 / tw; if (th > g.Ho) th = g.Ho; if (th < 1) continue;
      const long tiles = long((g.Wo + tw - 1) / tw) * ((g.Ho + th - 1) / th);
      const double u = double(g.Ho) * g.Wo / (double(tiles) * 128.0);
      if (u > bu + 1e-9 || (u > bu - 1e-9 && tw > btw)) { bu = u; btw = tw; bth = th; }
    }
    if (halo) {
      // halo tile: (th+2) x (tw+2) input pixels loaded once per 64-channel block; the 128 MMA rows are 128 consecutive
      // positions of that tile (row pitch tw+2), so 2 of every tw+2 rows are halo columns and carry no output.
      btw = 1; bth = 1; bu = -1;
      for (int tw = 1; tw <= g.Wo && tw <= 126; ++tw) {
        int th = 128 / (tw + 2); if (th > g.Ho) th = g.Ho; if (th < 1) continue;
        const long tiles = long((g.Wo + tw - 1) / tw) * ((g.Ho + th - 1) / th);
        const double u = double(g.Ho) * g.Wo / (double(tiles) * 128.0);
        if (u > bu + 1e-9 || (u > bu - 1e-9 && tw > btw)) { bu = u; btw = tw; bth = th; }
      }
      g.tw = btw + 2; g.tw_valid = btw; g.th = bth;
      g.num_kb = g.cin_blocks;                                  // pipeline unit = one channel block (9 taps)
      g.a_bytes = uint32_t(bth + 2) * (btw + 2) * uint32_t(2 * bk);
      g.a_slot = (uint32_t(2 * (btw + 2) + 2 + 128) * uint32_t(2 * bk) + 1023) & ~1023u;
    } else {
      g.tw = btw; g.tw_valid = btw; g.th = bth;
      g.a_bytes = uint32_t(btw) * bth * bk * 2;
    }
    g.nb = 1;
    g.tiles_x = (g.Wo + btw - 1) / btw; g.tiles_y = (g.Ho + bth - 1) / bth;
    if (!halo && g.tiles_x == 1 && g.tiles_y == 1 && btw == g.Wo && bth == g.Ho && btw * bth * 2 <= 128 && d.batch > 1) {
      // tiny maps (DaViT stages at 64x64 crops: 8x8, 4x4, 2x2 outputs): one TMA box spans nb whole images so the 128
      // MMA rows are full instead of 64/16/4 valid ones
      int nb = 128 / (btw * bth);
      if (nb > d.batch) nb = d.batch;
      g.nb = nb;
      g.a_bytes *= uint32_t(nb);
    }
    g.m_tiles = (g.nb > 1) ? (d.batch + g.nb - 1) / g.nb : g.tiles_x * g.tiles_y * d.batch;
    const cuuint64_t ld = cuuint64_t(d.lda);
    if (halo) {
      cuuint64_t dims[4] = {cuuint64_t(d.Cin), cuuint64_t(d.W), cuuint64_t(d.H), cuuint64_t(d.batch)};
      cuuint64_t str[3] = {ld * 2, ld * 2 * d.W, ld * 2 * d.W * d.H};
      cuuint32_t box[4] = {cuuint32_t(bk), cuuint32_t(btw + 2), cuuint32_t(bth + 2), 1};
      if (int e = encode(&tmA, d.bf16, 4, d.A, dims, str, box, bk)) return e;
    } else if (d.mode == 1) {
      cuuint64_t dims[4] = {cuuint64_t(a_span), cuuint64_t(d.W), cuuint64_t(d.H), cuuint64_t(d.batch)};
      cuuint64_t str[3] = {ld * 2, ld * 2 * d.W, ld * 2 * d.W * d.H};
      cuuint32_t box[4] = {cuuint32_t(bk), cuuint32_t(btw), cuuint32_t(bth), cuuint32_t(g.nb)};
      if (int e = encode(&tmA, d.bf16, 4, d.A, dims, str, box, bk)) return e;
    } else {
      // (x parity, channel) merged in dim0: element (n, 2*yo+py, 2*xo+px, c) at c + px*ld  (+ xo*2ld + py*W*ld + yo*2W*ld)
      g.ldpar = int(d.lda);   // producer adds px * ldA to the channel coordinate
      cuuint64_t dims[5] = {ld + cuuint64_t(a_span), cuuint64_t(d.W / 2), 2, cuuint64_t(d.H / 2), cuuint64_t(d.batch)};
      cuuint64_t str[4] = {ld * 4, ld * 2 * d.W, ld * 4 * d.W, ld * 2 * d.W * d.H};
      cuuint32_t box[5] = {cuuint32_t(bk), cuuint32_t(btw), 1, cuuint32_t(bth), cuuint32_t(g.nb)};
      if (int e = encode(&tmA, d.bf16, 5, d.A, dims, str, box, bk)) return e;
    }
  }
  int bn = 16, ksplit = 1;
  static const bool no_split = getenv("B2P_NO_SPLITK") != nullptr;
  const int slot = (no_split || d.no_split) ? -1 : ws_slot_for(st);
  pick_tiling(d.N, g.m_tiles, g.num_kb, halo ? 9 * bk : bk, g.a_bytes, d.bn_max > 0 ? d.bn_max : 256, slot >= 0, d.x3 != 0, &bn, &ksplit);
  // Resident weights: one N tile, no split-K, at least one full wave of M tiles, and the whole weight matrix + a >= 2-deep
  // A ring must fit in shared memory (see GemmArgs::bres).
  static const bool no_res = getenv("B2P_NO_BRES") != nullptr;
  bool bres = false;
  int res_slots = 0, res_stagesA = 0;
  const uint32_t a_slot_sep = halo ? g.a_slot : uint32_t(kASlot);
  if (!no_res && !d.x3 && d.N <= 256 && g.m_tiles >= g_num_sms && (d.bn_max <= 0 || d.bn_max >= d.N)) {
    static const int cand[] = {16, 32, 48, 64, 96, 128, 192, 256};
    int bnr = 256;
    for (int c : cand) if (c >= d.N) { bnr = c; break; }
    const uint32_t bslot = (uint32_t(bnr) * bk * 2 + 1023) & ~1023u;
    res_slots = halo ? g.cin_blocks * 9 : g.num_kb;
    const long long bar_bytes = 8LL * (2 * res_slots + 4 + 2 * 8) + 64;
    const long long avail = (long long)g_max_smem - 1024 - ((bar_bytes + 1023) & ~1023LL) - (long long)res_slots * bslot;
    if (avail >= 2LL * a_slot_sep) {
      bres = true;
      bn = bnr;
      ksplit = 1;
      res_stagesA = int(avail / a_slot_sep);
      if (res_stagesA > 8) res_stagesA = 8;
    }
  }
  g.bres = bres ? 1 : 0;
  g.sep = (halo || bres) ? 1 : 0;
  g.taps = halo ? 9 : 1;
  g.bn = bn;
  static const bool sk_last = getenv("B2P_SPLITK_LAST") != nullptr;
  g.sk_last = sk_last ? 1 : 0;
  g.ksplit = ksplit;
  g.kb_per = (g.num_kb + ksplit - 1) / ksplit;
  g.ws = slot >= 0 ? g_ws[slot] : nullptr;
  g.counters = slot >= 0 ? g_counters[slot] : nullptr;
  g.n_tiles = (d.N + bn - 1) / bn;
  // co-scheduled CTAs should share the LARGER operand through L2: weights bigger than activations -> M tiles fastest
  g.mt_fast = (d.mode == 0 && g.m_tiles > 1 && (long long)d.N > (long long)d.M) ? 1 : 0;
  g.b_bytes = uint32_t(bn) * bk * 2;
  g.b_slot = (g.b_bytes + 1023) & ~1023u;
  g.idesc = make_idesc(bn, d.bf16);
  {
    cuuint64_t dims[2] = {cuuint64_t(xk) * cuuint64_t(Ktot), cuuint64_t(d.N)};
    cuuint64_t str[1] = {cuuint64_t(xk) * cuuint64_t(Ktot) * 2};
    cuuint32_t box[2] = {cuuint32_t(bk), cuuint32_t(bn)};
    if (int e = encode(&tmB, d.bf16, 2, d.B, dims, str, box, bk)) return e;
  }
  g.d_ksplit = FastDiv::make(g.ksplit); g.d_ntiles = FastDiv::make(g.n_tiles); g.d_mtiles = FastDiv::make(g.m_tiles);
  g.d_perimg = FastDiv::make(d.mode != 0 ? g.tiles_x * g.tiles_y : 1); g.d_tilesx = FastDiv::make(d.mode != 0 ? g.tiles_x : 1);
  g.d_cinb = FastDiv::make(d.mode != 0 ? g.cin_blocks : 1);
  const int stage_bytes = g.sep ? int(g.b_slot) : xk * (kASlot + int(g.b_slot));
  int stages, bar_space = 512;
  if (bres) {
    g.a_slot = a_slot_sep;
    g.stagesA = res_stagesA;
    stages = res_slots;                                   // every B k-block (x tap) owns a slot for the whole launch
    bar_space = int((8LL * (2 * stages + 4 + 2 * g.stagesA) + 64 + 1023) & ~1023LL);
  } else if (halo) {
    // B ring first (up to 8 taps in flight), then as deep an A ring as fits (2..4 halo tiles)
    stages = (g_max_smem - 1024 - 512 - 2 * int(g.a_slot)) / stage_bytes;
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages < 2) stages = 2;
    int sa = (g_max_smem - 1024 - 512 - stages * stage_bytes) / int(g.a_slot);
    g.stagesA = sa > 4 ? 4 : (sa < 2 ? 2 : sa);
  } else {
    g.stagesA = 0;
    stages = (g_max_smem - 1024 - 512) / stage_bytes;
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages > g.kb_per && g.kb_per >= 2 && g.ksplit == 1) stages = g.kb_per;
    if (stages < 2) stages = 2;
  }
  const int a_region = g.sep ? g.stagesA * int(g.a_slot) : 0;
  g.stages = stages;
  const size_t smem = size_t(a_region) + size_t(stages) * stage_bytes + 1024 + bar_space;
  if (smem > size_t(g_max_smem)) return set_error("gemm: internal error, shared-memory plan exceeds the device limit");
  // vector epilogue needs 16-byte aligned rows in out / residual and bias
  const int esz = d.out_f32 ? 4 : 2;
  g.vec_ok = ((reinterpret_cast<uintptr_t>(d.out) & 15) == 0) && ((d.ldc * esz) % 16 == 0) &&
             (!d.res || (((reinterpret_cast<uintptr_t>(d.res) & 15) == 0) && ((d.ldr * esz) % 16 == 0))) &&
             (!d.bias || ((reinterpret_cast<uintptr_t>(d.bias) & 15) == 0));
  {
    static const bool no_v256 = getenv("B2P_NO_V256") != nullptr;
    auto a32 = [](const void* p, long long ld, int es) { return (reinterpret_cast<uintptr_t>(p) & 31) == 0 && (ld * es) % 32 == 0; };
    g.vec32_ok = !no_v256 && g.vec_ok && a32(d.out, d.ldc, esz) && (!d.res || a32(d.res, d.ldr, esz)) &&
                 (g.split * esz) % 32 == 0 && (g.res_lo * esz) % 32 == 0;
  }
  static const bool dbg = getenv("B2P_DEBUG") != nullptr;
  static const bool no_pdl = getenv("B2P_NO_PDL") != nullptr;
  const int total = g.m_tiles * g.n_tiles * g.ksplit;
  static const int max_grid = getenv("B2P_MAX_GRID") ? atoi(getenv("B2P_MAX_GRID")) : 0;   // experiment: leave SMs to other streams
  int grid = total < g_num_sms ? total : g_num_sms;
  if (max_grid > 0 && grid > max_grid && ksplit == 1) grid = max_grid;
  if (grid <= 0) return 0;
  if (dbg)
    fprintf(stderr, "b2p_gemm mode=%d M=%d N=%d Ktot=%d bk=%d bn=%d tw=%d th=%d m_tiles=%d n_tiles=%d stages=%d grid=%d act=%d f32=%d res=%d ksplit=%d x3=%d bres=%d stagesA=%d\n",
            g.mode, d.mode == 0 ? d.M : g.m_tiles * 128, d.N, Ktot, bk, bn, g.tw, g.th, g.m_tiles, g.n_tiles, stages, grid,
            d.act, d.out_f32, d.res != nullptr, ksplit, g.x3, g.bres, g.stagesA);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = no_pdl ? 0 : 1;
  bool traced = false;
  if (g_trace && grid <= kTraceCtas) {
    std::lock_guard<std::mutex> lk(g_trace_mu);
    if (g_trace_n < kTraceCap) {
      const int m[8] = {g.mode, d.mode == 0 ? d.M : g.m_tiles * 128, d.N, Ktot, bn, ksplit, g.x3, grid};
      for (int i = 0; i < 8; ++i) g_trace_meta[g_trace_n][i] = m[i];
      g.trace = g_trace + size_t(g_trace_n) * kTraceCtas * kTraceSlots;
      ++g_trace_n;
      traced = true;
    }
  }
  cudaError_t ce = traced ? cudaLaunchKernelEx(&cfg, gemm_tcgen05_kernel_trace, tmA, tmB, g)
                          : cudaLaunchKernelEx(&cfg, gemm_tcgen05_kernel, tmA, tmB, g);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  if (ce != cudaSuccess) return set_error(cudaGetErrorString(ce));
  count_launch();
  return 0;
}

// -> number of traced launches since the last call; stamps [n][kTraceCtas = 160][16] (ns, 0 = not written), meta [n][8] =
// {mode, M, N, K, bn, ksplit, x3, grid}.  Synchronises the device.
int trace_read(unsigned long long* stamps, int* meta, int max_launches) {
  if (!g_trace) return set_error("tracing is off (set B2P_TRACE=1 before the first GEMM launch)");
  cudaDeviceSynchronize();
  std::lock_guard<std::mutex> lk(g_trace_mu);
  const int n = g_trace_n < max_launches ? g_trace_n : max_launches;
  const size_t per = size_t(kTraceCtas) * kTraceSlots;
  if (n > 0 && cudaMemcpy(stamps, g_trace, sizeof(unsigned long long) * per * n, cudaMemcpyDeviceToHost) != cudaSuccess)
    return set_error("trace_read: copy failed");
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < 8; ++j) meta[i * 8 + j] = g_trace_meta[i][j];
  cudaMemset(g_trace, 0, sizeof(unsigned long long) * per * kTraceCap);
  g_trace_n = 0;
  return n;
}

}  // namespace b2p
