// Internal declarations shared by the .cu translation units of libb200parse.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2p {

int set_error(const char* msg);   // records msg for b2p_last_error(); returns -1
// One process drives ONE GPU (include/b200parse.h): the first launch binds the library to the current device; a later
// call made with another device current fails loudly instead of reusing the first device's workspaces and attributes.
int bind_device();
void count_launch(int n = 1);     // bumps the kernel-launch counter read by b2p_launch_count()

#define B2P_CHECK_LAUNCH()                                          \
  do {                                                              \
    cudaError_t _e = cudaGetLastError();                            \
    if (_e != cudaSuccess) return b2p::set_error(cudaGetErrorString(_e)); \
    b2p::count_launch();                                            \
  } while (0)

// Descriptor of one dense contraction for gemm_launch().
struct ConvGemm {
  int mode;            // 0 = GEMM rows, 1 = conv3x3 s1 p1, 2 = conv3x3 s2 p1   (NHWC)
  int bf16;            // operand type: 0 = fp16, 1 = bf16
  const void* A;       // mode 0: [M][lda]; conv: NHWC input (channel slice allowed, lda = channels per pixel)
  long long lda;
  const void* B;       // weights [N][K] (conv: K = 9*Cin ordered (ky,kx,c))
  int M, N, K;         // mode 0 only: M rows, K reduction
  int batch, H, W, Cin;  // conv only: input geometry
  void* out;           // [pixels][ldc] fp16 or fp32
  long long ldc;
  int out_f32;
  const float* bias;   // [N] or null
  const void* res;     // residual, same dtype as out, or null
  long long ldr;
  int act;             // 0 none, 1 SiLU, 2 GELU(erf)
  int bn_max;          // 0 = auto
  int no_split;        // 1 = never split K for this launch (tuning knob, flags bit 4)
  int split_out;       // fp16 output written as [hi(N) | lo(N)] (row stride ldc >= 2N): operand of a fp16x3 GEMM
  int x3;              // fp16x3 operands: A rows [hi(K) | lo(K)] (conv: per pixel [hi(Cin) | lo(Cin)]), B rows likewise;
                       // K / Cin are the LOGICAL sizes.  out = A_hi*B_hi + A_hi*B_lo + A_lo*B_hi, fp32 accumulate
  // fp16x3 "lo planes" (elements; 0 = the packed default): a channel slice of a wider [hi(Ctot) | lo(Ctot)] pixel / row
  // has its lo half Ctot elements after its hi half, not K (or N) elements after it.
  long long lo_a;      // A: lo half at column lo_a + k            (default K / Cin)
  long long lo_out;    // split_out: lo half at column lo_out + n  (default N)
  long long lo_res;    // fp16 residual is a hi/lo pair, lo at column lo_res + n (default: residual has no lo half)
};

int gemm_launch(const ConvGemm& d, cudaStream_t st);
int trace_read(unsigned long long* stamps, int* meta, int max_launches);   // B2P_TRACE=1 debugging aid

// Round-2 SIMT kernels of the caption encoder (florence_simt.cu).  Return 0 = launched, 1 = shape not covered (the caller
// falls back to the first-version kernel), < 0 = error (message recorded).
int dwconv_ln_v3_launch(const float* x, int B, int H, int W, int C, const float* w9c, const float* bias, float* y,
                        const float* gamma, const float* beta, float eps, void* out16, int split, cudaStream_t st);
int window_attn_crop_launch(const float* qkv, const float* qkv_bias, int B, int H, int W, int C, int heads, int win, void* out,
                            int split, cudaStream_t st);
int channel_attn_v3_launch(const float* qkv, int B, int N, int C, int groups, void* out, int split, cudaStream_t st);
int mha_short_launch(const float* q, long long ldq, const float* k, const float* v, long long ldk, int B, int Lq, int Lk, int heads,
                     void* out, long long ldo, int split, cudaStream_t st);

// Programmatic dependent launch for the small SIMT kernels: launched with the stream-serialization attribute they may
// be scheduled while the preceding (persistent, early-triggering) GEMM drains; each such kernel calls pdl_wait() before
// touching global memory.  They never trigger their own dependents early (their grids are not guaranteed resident).
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#endif

}  // namespace b2p
