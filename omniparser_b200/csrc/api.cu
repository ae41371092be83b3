// C-ABI glue of libb200parse.so: error string, launch counter, and the dense-contraction entry points.
// Declarations + the reference call sites each entry point replaces: include/b200parse.h.
#include "b2p_internal.h"
#include <atomic>
#include <mutex>
#include <string>
#include <stdlib.h>
#include <stdio.h>

namespace b2p {
static std::mutex g_err_mu;
static std::string g_err;
static std::atomic<long long> g_launches{0};

int set_error(const char* msg) {
  std::lock_guard<std::mutex> lk(g_err_mu);
  g_err = msg ? msg : "unknown error";
  return -1;
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
static std::atomic<int> g_bound_dev{-1};
int bind_device() {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return set_error("cudaGetDevice failed (no CUDA device?)");
  int expect = -1;
  if (g_bound_dev.compare_exchange_strong(expect, dev) || expect == dev) return 0;
  char buf[160];
  snprintf(buf, sizeof buf, "libb200parse is bound to CUDA device %d (one process drives one GPU); called with device %d current", expect, dev);
  return set_error(buf);
}
bool pdl_enabled() {
  // PDL on the small SIMT kernels is OFF by default: measured on the 2-stream pipelined parse it costs 20 % (their
  // early-launched CTAs sit blocked in griddepcontrol.wait and take SM slots from the other stream); the persistent
  // GEMM kernel keeps its own PDL (B2P_NO_PDL disables that one).
  static const bool on = getenv("B2P_PDL_SIMT") != nullptr;
  return on;
}
}  // namespace b2p

using namespace b2p;

extern "C" {

const char* b2p_last_error(void) {
  static thread_local std::string copy;
  std::lock_guard<std::mutex> lk(g_err_mu);
  copy = g_err;
  return copy.c_str();
}

long long b2p_launch_count(void) { return g_launches.load(); }

int b2p_abi_version(void) { return 3; }

// Debugging aid (B2P_TRACE=1): per-CTA phase timestamps of the traced GEMM launches, see gemm_tcgen05.cu::trace_read.
int b2p_trace_read(unsigned long long* stamps, int* meta, int max_launches) { return trace_read(stamps, meta, max_launches); }

// C[M,N] = act(A[M,K] * B[N,K]^T + bias) (+ residual); A, B fp16 (bf16 if flags&1); out fp16 or fp32 (flags&2);
// flags&4: fp16 output in the fp16x3 operand layout [hi(N) | lo(N)] (ldc >= 2N).
// flags&8: fp16x3 operands: A rows [hi(K) | lo(K)] (lda >= 2K), B rows [hi(K) | lo(K)]; K is the logical reduction size.
// `_planes` form: explicit lo-plane offsets (elements) for fp16x3 operands that are channel slices of a wider
// [hi(Ctot) | lo(Ctot)] buffer: lo_a (A), lo_out (flags&4 output), lo_res (fp16 residual given as a hi/lo pair); 0 = default.
int b2p_gemm_planes(const void* A, long long lda, const void* B, int M, int N, int K, void* out, long long ldc,
                    const float* bias, const void* residual, long long ldr, int act, int flags, long long lo_a,
                    long long lo_out, long long lo_res, cudaStream_t st) {
  ConvGemm d{};
  d.mode = 0; d.bf16 = flags & 1; d.A = A; d.lda = lda; d.B = B; d.M = M; d.N = N; d.K = K;
  d.out = out; d.ldc = ldc; d.out_f32 = (flags >> 1) & 1; d.bias = bias; d.res = residual; d.ldr = ldr; d.act = act;
  d.bn_max = (flags >> 8) & 0x1ff; d.no_split = (flags >> 4) & 1; d.split_out = (flags >> 2) & 1; d.x3 = (flags >> 3) & 1;
  d.lo_a = lo_a; d.lo_out = lo_out; d.lo_res = lo_res;
  return gemm_launch(d, st);
}
int b2p_gemm(const void* A, long long lda, const void* B, int M, int N, int K, void* out, long long ldc,
             const float* bias, const void* residual, long long ldr, int act, int flags, cudaStream_t st) {
  return b2p_gemm_planes(A, lda, B, M, N, K, out, ldc, bias, residual, ldr, act, flags, 0, 0, 0, st);
}

// 3x3 pad-1 convolution (stride 1 or 2) on an NHWC fp16 channel slice; weights [Cout][9*Cin] ordered (ky,kx,c).
// flags&8 (fp16x3 operands): pixels are [hi(Cin) | lo(Cin)], weights [Cout][9][hi(Cin) | lo(Cin)]; Cin is the logical size.
int b2p_conv3x3_planes(const void* in, long long ld_in, int batch, int H, int W, int Cin, int stride, const void* weight,
                       int Cout, void* out, long long ldc, const float* bias, const void* residual, long long ldr, int act,
                       int flags, long long lo_a, long long lo_out, long long lo_res, cudaStream_t st) {
  if (stride != 1 && stride != 2) return set_error("conv3x3: stride must be 1 or 2");
  ConvGemm d{};
  d.mode = stride; d.bf16 = flags & 1; d.A = in; d.lda = ld_in; d.B = weight; d.N = Cout;
  d.batch = batch; d.H = H; d.W = W; d.Cin = Cin;
  d.out = out; d.ldc = ldc; d.out_f32 = (flags >> 1) & 1; d.bias = bias; d.res = residual; d.ldr = ldr; d.act = act;
  d.bn_max = (flags >> 8) & 0x1ff; d.no_split = (flags >> 4) & 1; d.split_out = (flags >> 2) & 1; d.x3 = (flags >> 3) & 1;
  d.lo_a = lo_a; d.lo_out = lo_out; d.lo_res = lo_res;
  return gemm_launch(d, st);
}
int b2p_conv3x3(const void* in, long long ld_in, int batch, int H, int W, int Cin, int stride, const void* weight,
                int Cout, void* out, long long ldc, const float* bias, const void* residual, long long ldr, int act,
                int flags, cudaStream_t st) {
  return b2p_conv3x3_planes(in, ld_in, batch, H, W, Cin, stride, weight, Cout, out, ldc, bias, residual, ldr, act, flags, 0, 0, 0, st);
}

}  // extern "C"
