/* libb200parse.so -- C ABI of the B200-native OmniParser parse hot path.
 *
 * The reference (microsoft/OmniParser) has no FFI layer: its hot path is three Python functions
 * (util/utils.py: get_yolo_model :72-85, get_caption_model_processor :48-69, get_som_labeled_img :417-496) whose
 * arithmetic lives in third-party wheels (TorchScript/cuDNN, torchvision::nms, cv2, PIL, HF transformers).
 * Each entry point below replaces one of those library call sites; the reference file:line it stands in for is
 * cited per function.  omniparser_b200/_lib.py is the ctypes binding a maintainer would add (INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only (no torch types); every pointer is DEVICE memory unless its name
 * ends in _host; all launches are asynchronous on `stream`; return 0 on success, -1 on error with the message in
 * b2p_last_error(); the caller owns every buffer; a process uses one GPU (cudaSetDevice before the first call).
 * Feature maps are NHWC fp16 "channel slices": base pointer already offset to the first channel, `ld` = channels
 * per pixel of the owning buffer, so concatenations are pointer arithmetic.
 */
#ifndef B200PARSE_H
#define B200PARSE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* b2p_stream_t; /* == cudaStream_t */

/* ---- library state ---- */
const char* b2p_last_error(void);
long long b2p_launch_count(void); /* kernels launched by this library since load (bench.py gpu_launches) */
int b2p_abi_version(void);
/* Debugging aid, not on the hot path: with B2P_TRACE=1 in the environment every GEMM/conv launch runs an instrumented
 * instantiation of the kernel that leaves globaltimer stamps per CTA; this returns the launches recorded since the
 * last call: stamps [n][160][16] (ns; slots: entry, prologue, dependency wait, first TMA, first full stage, first
 * accumulator issued, first epilogue start, last epilogue end, exit), meta [n][8] = {mode, M, N, K, bn, ksplit, x3, grid}. */
int b2p_trace_read(unsigned long long* stamps, int* meta, int max_launches);

/* ---- dense contractions (tcgen05 + TMA + TMEM), ref:util/yolov9.py:120-121 and ref:util/utils.py:125 ----
 * flags: bit0 operands bf16 (else fp16) | bit1 output fp32 (else fp16) | bit2 fp16 output in the "fp16x3" operand
 * layout [hi(N) | lo(N)] (ldc >= 2N) | bit3 fp16x3 OPERANDS: A rows [hi(K) | lo(K)] (lda >= 2K; conv: pixels
 * [hi(Cin) | lo(Cin)]), weight rows [hi | lo] likewise (conv: per tap), K / Cin the logical sizes; the kernel loads each
 * half once per k-block and accumulates hi*hi + hi*lo + lo*hi in fp32 | bit4 never split K (tuning) | bits 8.. maximum N tile (0 = auto).
 * act: 0 none, 1 SiLU, 2 exact GELU.
 * out = act(A[M,K] * B[N,K]^T + bias[N]) + residual (residual has the dtype of out). */
int b2p_gemm(const void* A, long long lda, const void* B, int M, int N, int K, void* out, long long ldc,
             const float* bias, const void* residual, long long ldr, int act, int flags, b2p_stream_t stream);
/* 3x3, pad 1, stride 1|2 convolution as implicit GEMM; weight [Cout][9*Cin] ordered (ky, kx, c). */
int b2p_conv3x3(const void* in, long long ld_in, int batch, int H, int W, int Cin, int stride, const void* weight,
                int Cout, void* out, long long ldc, const float* bias, const void* residual, long long ldr, int act,
                int flags, b2p_stream_t stream);

/* `_planes` forms (fp16x3 operands that are channel slices of a wider [hi(Ctot) | lo(Ctot)] pixel / row): explicit
 * lo-plane offsets in elements -- lo_a: A's lo half at column lo_a + k (default K / Cin); lo_out: with flags bit2 the
 * output's lo half at column lo_out + n (default N); lo_res: the fp16 residual is a hi/lo pair whose lo half sits at
 * column lo_res + n (default 0: the residual has no lo half).  This is what the parity-grade (fp16x3) detector mode uses:
 * every YOLOv9-E feature map stays a hi/lo pair inside its concat buffer (ref:util/yolov9.py:120-121 in fp32). */
int b2p_gemm_planes(const void* A, long long lda, const void* B, int M, int N, int K, void* out, long long ldc,
                    const float* bias, const void* residual, long long ldr, int act, int flags, long long lo_a,
                    long long lo_out, long long lo_res, b2p_stream_t stream);
int b2p_conv3x3_planes(const void* in, long long ld_in, int batch, int H, int W, int Cin, int stride, const void* weight,
                       int Cout, void* out, long long ldc, const float* bias, const void* residual, long long ldr, int act,
                       int flags, long long lo_a, long long lo_out, long long lo_res, b2p_stream_t stream);

/* ---- YOLOv9-E graph helpers (inside the TorchScript archive, ref:util/yolov9.py:120-121) ----
 * `_x3` forms: every map is an fp16 hi/lo pair (lo plane `lo*` elements after the hi plane, 0 = plain fp16); the
 * arithmetic runs on the exact fp32 sums hi + lo and the result is re-split. */
int b2p_adown_pool(const void* x, long long ldx, int B, int H, int W, int C, void* x1, long long ld1, void* x2,
                   long long ld2, b2p_stream_t stream);
int b2p_adown_pool_x3(const void* x, long long ldx, int B, int H, int W, int C, void* x1, long long ld1, void* x2,
                      long long ld2, long long lox, long long lo1, long long lo2, b2p_stream_t stream);
int b2p_maxpool_s1(const void* x, long long ldx, int B, int H, int W, int C, int k, void* y, long long ldy,
                   b2p_stream_t stream);
int b2p_maxpool_s1_x3(const void* x, long long ldx, int B, int H, int W, int C, int k, void* y, long long ldy,
                      long long lox, long long loy, b2p_stream_t stream);
int b2p_upsample2x(const void* x, long long ldx, int B, int H, int W, int C, void* y, long long ldy,
                   b2p_stream_t stream);
int b2p_upsample2x_x3(const void* x, long long ldx, int B, int H, int W, int C, void* y, long long ldy, long long lox,
                      long long loy, b2p_stream_t stream);
/* explicit 3x3 / pad-1 im2col of an NHWC f16 map -> [B*Ho*Wo][9*C] (tap-major), for convs whose output map is far
 * smaller than one 128-pixel implicit-GEMM tile (DaViT patch-embed convs of the 64x64-crop mode, hf:modeling_florence2.py
 * ConvEmbed, reached from ref:util/utils.py:125 generate) */
int b2p_im2col3x3(const void* x, long long ldx, int B, int H, int W, int C, int stride, int halves, void* out,
                  b2p_stream_t stream);   /* halves = 2: fp16x3 pixels [hi(C) | lo(C)] -> rows [hi: 9C | lo: 9C] */
int b2p_cbfuse(int nsrc, const void* const* srcs_host, const long long* lds_host, const int* shifts_host,
               const void* last, long long ldl, int B, int H, int W, int C, void* y, long long ldy,
               b2p_stream_t stream);
int b2p_cbfuse_x3(int nsrc, const void* const* srcs_host, const long long* lds_host, const int* shifts_host,
                  const long long* los_host, const void* last, long long ldl, int B, int H, int W, int C, void* y,
                  long long ldy, long long lol, long long loy, b2p_stream_t stream);

/* ---- detector pre/post-processing ----
 * b2p_letterbox: PIL Image.resize(LANCZOS) + paste on a 114 canvas, ref:util/yolov9.py:73-84 (bit-exact).
 * b2p_im2col_u8: /255 (ref:util/yolov9.py:85) or CLIP rescale+normalise (ref:util/utils.py:121) via `lut` [3][256]
 *                + im2col of the 3-channel stem conv; split != 0 writes the fp16x3 layout.
 * b2p_yolo_decode: ref:util/yolov9.py:89-108 (_decode) and :123-129 (class max, strict conf filter, un-letterbox).
 * b2p_batched_nms: torchvision.ops.batched_nms + [:max_det] + clamp, ref:util/yolov9.py:131-135 (bit-exact).
 * b2p_lanczos_coeffs_host: Pillow's coefficient table on the host (unit-testable without a GPU). */
int b2p_lanczos_coeffs_host(int in_size, int out_size, int* ksize_host, int* bounds_host, int* kk_host, int kk_capacity);
int b2p_letterbox(const unsigned char* src, int B, int H, int W, int Wr, int Hr, int Tw, int Th, int pad_l, int pad_t,
                  unsigned char* tmp, unsigned char* canvas, b2p_stream_t stream);
/* Pillow-exact u8 resize, filter 0 LANCZOS / 1 BICUBIC (CLIP processor resample=3, ref:util/utils.py:123 CPU branch) */
int b2p_resize_u8(const unsigned char* src, int B, int H, int W, int Wr, int Hr, int filter, unsigned char* tmp,
                  unsigned char* out, b2p_stream_t stream);
int b2p_im2col_u8(const unsigned char* img, int B, int H, int W, int k, int s, int p, int Kpad, const float* lut,
                  void* out, int split, b2p_stream_t stream);
int b2p_yolo_decode(const float* const* cls_host, const float* const* box_host, const int* Hs_host, const int* Ws_host,
                    int nc, int B, float conf, const float* pad_l, const float* pad_t, const float* scale, int cap,
                    float* cand_box, float* cand_score, int* cand_cls, int* cand_count, float* dense_ltrb,
                    float* dense_score, b2p_stream_t stream);
int b2p_batched_nms(const float* box, const float* score, const int* cls, const int* count, int B, int cap,
                    double iou_thr, int max_det, const float* img_w, const float* img_h, int* keep_idx, float* out_box,
                    float* out_score, int* out_count, b2p_stream_t stream);

/* ---- overlap filter on the device, ref:util/utils.py:241-319 (remove_overlap_new), :411-415 (int_box_area), :432, :444-451 ----
 * Per screenshot b: the detector's kept boxes box_px[b][0..count[b]) (pixels, fp32, b2p_batched_nms output) and ocr_count[b]
 * OCR boxes as fp32 RATIO boxes (int_box_area-filtered on the host, where their strings stay).  Same float64 arithmetic,
 * comparisons and list order as the reference.  Outputs: icon_state[b][i] = 0 dropped | 1 kept, needs a caption | 2 kept,
 * labelled by OCR text; label_mask[b][i][max_ocr/32] bit k = OCR box k labels icon i; ocr_removed[b][k]; icon_ratio = the
 * fp32 ratio boxes (:432); crop_box / crop_img = the state-1 boxes of the whole batch in order (the crop list of
 * b2p_crop_resize); crop_counts[0..B) per screenshot, crop_counts[B] the total.  `arrive` is a zeroed int the kernel resets. */
int b2p_overlap_filter(const float* box_px, const int* count, int B, int max_det, const float* img_w, const float* img_h,
                       const float* ocr_ratio, const int* ocr_count, int max_ocr, double iou_thr, int* icon_state,
                       unsigned* label_mask, int* ocr_removed, float* icon_ratio, float* crop_box, int* crop_img,
                       int* crop_counts, int* arrive, b2p_stream_t stream);

/* ---- crop + resize, ref:util/utils.py:97-103 (numpy slice + cv2.resize(.., (64,64)), bit-exact) ---- */
int b2p_crop_resize(const unsigned char* imgs, const int* img_hw, const long long* img_off, const float* boxes_ratio,
                    const int* box_img, int n_box, int out_hw, unsigned char* out, int* status, b2p_stream_t stream);

/* ---- Florence-2 (HF generate, ref:util/utils.py:125): non-GEMM kernels; `split` selects the fp16x3 layout ---- */
int b2p_layernorm(const float* x, long long ldx, const float* gamma, const float* beta, float eps, int T, int C,
                  void* out16, long long ld16, float* out32, long long ld32, int split, b2p_stream_t stream);
int b2p_dwconv_ln(const float* x, int B, int H, int W, int C, const float* w9c, const float* bias, float* y,
                  const float* gamma, const float* beta, float eps, void* out16, int split, b2p_stream_t stream);
int b2p_window_attn(const float* qkv, const float* qkv_bias, int B, int H, int W, int C, int heads, int win, void* out,
                    int split, b2p_stream_t stream);
int b2p_channel_attn(const float* qkv, int B, int N, int C, int groups, void* out, int split, b2p_stream_t stream);
int b2p_mha(const float* q, long long ldq, const float* k, const float* v, long long ldk, int B, int Lq, int Lk,
            int heads, void* out, long long ldo, int split, b2p_stream_t stream);
int b2p_mha_cached(const float* q, long long ldq, const float* knew, const float* vnew, long long ldnew, float* kcache,
                   float* vcache, int tmax, const int* step, int B, int heads, void* out, long long ldo, int split,
                   b2p_stream_t stream);
int b2p_encoder_embed(const float* img, int n_img, const float* E, const int* prompt, int n_prompt, const float* P,
                      int B, int C, float* out, b2p_stream_t stream);
int b2p_decoder_embed(const float* E, const int* seq, int seq_ld, const int* step, const float* P, int B, int C,
                      float* out, b2p_stream_t stream);
int b2p_projector_prep(const float* x, const float* pos, int B, int HW, int C, void* out, int split,
                       b2p_stream_t stream);
/* HF greedy step with no_repeat_ngram / forced BOS / forced EOS processors, hf:generation/utils.py:2727-2805 */
int b2p_greedy_pick(const float* logits, long long ld, int V, int B, int* seq, int seq_ld, int* finished,
                    const int* step, int ngram, int forced_bos, int forced_eos, int eos, int pad, int max_len,
                    float* dump, int* n_unfinished, b2p_stream_t stream);
int b2p_step_advance(int* step, b2p_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200PARSE_H */
