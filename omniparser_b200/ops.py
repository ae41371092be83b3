"""Torch-tensor front ends of the C-ABI ops (device memory and streams come from PyTorch; the math does not).

A feature map is a :class:`Map`: an NHWC fp16 channel slice ``(ptr, B, H, W, C, ld)`` inside a larger buffer,
so concatenations (``torch.cat`` in the reference graph) are never materialised.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass

import torch

from . import _lib

ACT_NONE, ACT_SILU, ACT_GELU = 0, 1, 2
_CAPTURE_STREAMS = {}
CAPTURE_LOCK = threading.RLock()   # one CUDA-graph capture at a time across the pipeline's threads


def capture_stream(tag, device):
    """One capture stream per engine: split-K scratch is keyed by stream, and graphs of different engines may replay
    concurrently on different streams."""
    key = (tag, str(device))
    if key not in _CAPTURE_STREAMS:
        _CAPTURE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _CAPTURE_STREAMS[key]


GRAPH_LAUNCHES = [0]   # kernels replayed through CUDA graphs (the C-side counter only sees direct launches)
_GRAPH_LAUNCHES_LOCK = threading.Lock()


def count_graph_launches(n: int):
    """the detect and caption threads of the pipelined parser replay graphs concurrently"""
    with _GRAPH_LAUNCHES_LOCK:
        GRAPH_LAUNCHES[0] += n
FLAG_BF16, FLAG_OUT_F32, FLAG_SPLIT, FLAG_X3, FLAG_NO_SPLITK = 1, 2, 4, 8, 16


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    if t is None:
        return C.c_void_p(0)
    if isinstance(t, int):
        return C.c_void_p(t)
    return C.c_void_p(t.data_ptr())


@dataclass
class Map:
    """NHWC channel slice: element (b, y, x, c) lives at ptr + 2*(((b*H + y)*W + x)*ld + c) bytes (fp16).
    ``lo`` > 0 (parity-grade fp16x3 maps): every value is an fp16 hi/lo pair, the lo half ``lo`` elements after the hi
    half (pixel layout [hi(Ctot) | lo(Ctot)], so a channel slice keeps the same ``lo`` = Ctot)."""

    buf: torch.Tensor   # owning buffer [B, H, W, ld]
    c0: int
    C: int
    lo: int = 0

    @property
    def B(self): return self.buf.shape[0]
    @property
    def H(self): return self.buf.shape[1]
    @property
    def W(self): return self.buf.shape[2]
    @property
    def ld(self): return self.buf.shape[3]
    @property
    def ptr(self): return self.buf.data_ptr() + self.c0 * self.buf.element_size()

    def slice(self, c0, C_):
        assert 0 <= c0 and c0 + C_ <= self.C
        return Map(self.buf, self.c0 + c0, C_, self.lo)

    def torch(self):
        """NCHW float32 copy (tests / debugging only)."""
        t = self.buf[..., self.c0:self.c0 + self.C].permute(0, 3, 1, 2).float()
        if self.lo:
            t = t + self.buf[..., self.lo + self.c0:self.lo + self.c0 + self.C].permute(0, 3, 1, 2).float()
        return t


def new_map(B, H, W, Ctot, device, dtype=torch.float16, x3=False):
    """x3: hi/lo-pair map, pixel layout [hi(Ctot) | lo(Ctot)]."""
    if x3:
        assert dtype == torch.float16 and Ctot % 8 == 0
        return Map(torch.empty((B, H, W, 2 * Ctot), device=device, dtype=dtype), 0, Ctot, Ctot)
    return Map(torch.empty((B, H, W, Ctot), device=device, dtype=dtype), 0, Ctot)


def gemm(a_ptr, lda, w, M, N, K, out_ptr, ldc, bias=None, res_ptr=None, ldr=0, act=ACT_NONE, out_f32=False,
         bf16=False, bn_max=0, split=False, x3=False, no_splitk=False):
    """x3: fp16x3 operands -- A rows [hi(K) | lo(K)], w rows [hi(K) | lo(K)], K logical; split: fp16 output as [hi | lo]."""
    flags = ((FLAG_BF16 if bf16 else 0) | (FLAG_OUT_F32 if out_f32 else 0) | (FLAG_SPLIT if split else 0) |
             (FLAG_X3 if x3 else 0) | (FLAG_NO_SPLITK if no_splitk else 0) | (bn_max << 8))
    _lib.check(_lib.lib().b2p_gemm(_p(a_ptr), lda, _p(w), M, N, K, _p(out_ptr), ldc, _p(bias), _p(res_ptr), ldr, act,
                                   flags, _stream()))


def linear(x: torch.Tensor, w: torch.Tensor, bias=None, res=None, act=ACT_NONE, out_dtype=torch.float16, out=None,
           bn_max=0):
    """out[M,N] = act(x[M,K] @ w[N,K]^T + bias) + res ; x, w fp16 row-major (x may be a strided row view)."""
    assert x.dim() == 2 and w.dim() == 2 and x.shape[1] == w.shape[1] and x.stride(1) == 1 and w.is_contiguous()
    M, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), device=x.device, dtype=out_dtype)
    assert out.stride(1) == 1
    if res is not None:
        assert res.dtype == out.dtype and res.stride(1) == 1
    gemm(x, x.stride(0), w, M, N, K, out, out.stride(0), bias, res, res.stride(0) if res is not None else 0, act,
         out_f32=(out.dtype == torch.float32), bf16=(x.dtype == torch.bfloat16), bn_max=bn_max)
    return out


def conv1x1(x: Map, w, out: Map, bias=None, res: Map | None = None, act=ACT_SILU, out_f32=False):
    M = x.B * x.H * x.W
    if x.lo:   # parity-grade hi/lo maps: fp16x3 operands, hi/lo output unless it is fp32
        flags = FLAG_X3 | (FLAG_OUT_F32 if out_f32 else FLAG_SPLIT)
        _lib.check(_lib.lib().b2p_gemm_planes(_p(x.ptr), x.ld, _p(w), M, out.C, x.C, _p(out.ptr), out.ld, _p(bias),
                                              _p(res.ptr if res else None), res.ld if res else 0, act, flags, x.lo,
                                              0 if out_f32 else out.lo, res.lo if res else 0, _stream()))
        return
    gemm(x.ptr, x.ld, w, M, out.C, x.C, out.ptr, out.ld, bias, res.ptr if res else None, res.ld if res else 0, act,
         out_f32=out_f32)


def conv3x3(x: Map, w, out: Map, stride=1, bias=None, res: Map | None = None, act=ACT_SILU, out_f32=False, bn_max=0,
            split=False, x3=False):
    """x3: fp16x3 operands -- pixels [hi(Cin) | lo(Cin)] (x.C = 2*Cin), w [Cout][9][hi(Cin) | lo(Cin)].
    Hi/lo-pair maps (``x.lo``): the same operand mode with explicit lo planes (x.C stays the logical Cin)."""
    if x.lo:
        flags = FLAG_X3 | (FLAG_OUT_F32 if out_f32 else FLAG_SPLIT) | (bn_max << 8)
        _lib.check(_lib.lib().b2p_conv3x3_planes(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C, stride, _p(w), out.C, _p(out.ptr), out.ld,
                                                 _p(bias), _p(res.ptr if res else None), res.ld if res else 0, act, flags,
                                                 x.lo, 0 if out_f32 else out.lo, res.lo if res else 0, _stream()))
        return
    flags = (FLAG_OUT_F32 if out_f32 else 0) | (FLAG_SPLIT if split else 0) | (FLAG_X3 if x3 else 0) | (bn_max << 8)
    _lib.check(_lib.lib().b2p_conv3x3(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C // 2 if x3 else x.C, stride, _p(w), out.C, _p(out.ptr), out.ld,
                                      _p(bias), _p(res.ptr if res else None), res.ld if res else 0, act, flags,
                                      _stream()))


def adown_pool(x: Map, x1: Map, x2: Map):
    if x.lo:
        _lib.check(_lib.lib().b2p_adown_pool_x3(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C, _p(x1.ptr), x1.ld, _p(x2.ptr), x2.ld,
                                                x.lo, x1.lo, x2.lo, _stream()))
        return
    _lib.check(_lib.lib().b2p_adown_pool(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C, _p(x1.ptr), x1.ld, _p(x2.ptr), x2.ld,
                                         _stream()))


def maxpool_s1(x: Map, y: Map, k=5):
    if x.lo:
        _lib.check(_lib.lib().b2p_maxpool_s1_x3(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C, k, _p(y.ptr), y.ld, x.lo, y.lo, _stream()))
        return
    _lib.check(_lib.lib().b2p_maxpool_s1(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C, k, _p(y.ptr), y.ld, _stream()))


def upsample2x(x: Map, y: Map):
    if x.lo:
        _lib.check(_lib.lib().b2p_upsample2x_x3(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C, _p(y.ptr), y.ld, x.lo, y.lo, _stream()))
        return
    _lib.check(_lib.lib().b2p_upsample2x(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C, _p(y.ptr), y.ld, _stream()))


def im2col3x3(x: Map, stride, out, halves=1):
    """out [B*Ho*Wo, 9*x.C] f16 (tap-major) for a 3x3 / pad 1 conv over the NHWC map ``x``; halves=2: fp16x3 pixels
    [hi(C) | lo(C)] (x.C = 2C) -> rows [hi: 9C | lo: 9C]."""
    _lib.check(_lib.lib().b2p_im2col3x3(_p(x.ptr), x.ld, x.B, x.H, x.W, x.C // halves, stride, halves, _p(out), _stream()))


def cbfuse(srcs: list[Map], last: Map, out: Map):
    n = len(srcs)
    ptrs = (C.c_void_p * max(n, 1))(*[s.ptr for s in srcs])
    lds = (C.c_longlong * max(n, 1))(*[s.ld for s in srcs])
    shifts = (C.c_int * max(n, 1))(*[(last.H // s.H).bit_length() - 1 for s in srcs])
    if last.lo:
        los = (C.c_longlong * max(n, 1))(*[s.lo for s in srcs])
        _lib.check(_lib.lib().b2p_cbfuse_x3(n, ptrs, lds, shifts, los, _p(last.ptr), last.ld, last.B, last.H, last.W, last.C,
                                            _p(out.ptr), out.ld, last.lo, out.lo, _stream()))
        return
    _lib.check(_lib.lib().b2p_cbfuse(n, ptrs, lds, shifts, _p(last.ptr), last.ld, last.B, last.H, last.W, last.C,
                                     _p(out.ptr), out.ld, _stream()))


def yolo_decode(cls, box, hw, nc, B, conf, pad_l, pad_t, scale, cap, cand_box, cand_score, cand_cls, cand_count,
                dense_ltrb=None, dense_score=None):
    cp = (C.c_void_p * 3)(*[t.data_ptr() for t in cls])
    bp = (C.c_void_p * 3)(*[t.data_ptr() for t in box])
    Hs = (C.c_int * 3)(*[h for h, _ in hw])
    Ws = (C.c_int * 3)(*[w for _, w in hw])
    _lib.check(_lib.lib().b2p_yolo_decode(cp, bp, Hs, Ws, nc, B, conf, _p(pad_l), _p(pad_t), _p(scale), cap,
                                          _p(cand_box), _p(cand_score), _p(cand_cls), _p(cand_count),
                                          _p(dense_ltrb), _p(dense_score), _stream()))


def batched_nms(box, score, cls, count, B, cap, iou, max_det, img_w, img_h, keep_idx, out_box, out_score, out_count):
    _lib.check(_lib.lib().b2p_batched_nms(_p(box), _p(score), _p(cls), _p(count), B, cap, float(iou), max_det,
                                          _p(img_w), _p(img_h), _p(keep_idx), _p(out_box), _p(out_score),
                                          _p(out_count), _stream()))


def letterbox(src_u8, B, H, W, Wr, Hr, Tw, Th, pad_l, pad_t, tmp, canvas):
    _lib.check(_lib.lib().b2p_letterbox(_p(src_u8), B, H, W, Wr, Hr, Tw, Th, pad_l, pad_t, _p(tmp), _p(canvas),
                                        _stream()))


def resize_u8(src_u8, B, H, W, Wr, Hr, filt, tmp, out):
    """Pillow-exact resize; filt 0 = LANCZOS, 1 = BICUBIC."""
    _lib.check(_lib.lib().b2p_resize_u8(_p(src_u8), B, H, W, Wr, Hr, filt, _p(tmp), _p(out), _stream()))


def im2col_u8(img, B, H, W, k, s, p, Kpad, lut, out, split=False):
    _lib.check(_lib.lib().b2p_im2col_u8(_p(img), B, H, W, k, s, p, Kpad, _p(lut), _p(out), int(split), _stream()))


def overlap_filter(box_px, count, B, max_det, img_w, img_h, ocr_ratio, ocr_count, max_ocr, iou_thr, icon_state, label_mask,
                   ocr_removed, icon_ratio, crop_box, crop_img, crop_counts, arrive):
    _lib.check(_lib.lib().b2p_overlap_filter(_p(box_px), _p(count), B, max_det, _p(img_w), _p(img_h), _p(ocr_ratio), _p(ocr_count),
                                             max_ocr, float(iou_thr), _p(icon_state), _p(label_mask), _p(ocr_removed),
                                             _p(icon_ratio), _p(crop_box), _p(crop_img), _p(crop_counts), _p(arrive), _stream()))


def crop_resize(imgs, img_hw, img_off, boxes, box_img, n_box, out_hw, out, status):
    _lib.check(_lib.lib().b2p_crop_resize(_p(imgs), _p(img_hw), _p(img_off), _p(boxes), _p(box_img), n_box, out_hw,
                                          _p(out), _p(status), _stream()))


# ------------------------------------------------------------------------------------------ Florence-2 ops
# `split=True` writes fp16 activations in the fp16x3 operand layout [hi(C) | lo(C)] (row stride 2*C).
def layernorm(x, gamma, beta, T, C, out16=None, out32=None, eps=1e-5, split=False):
    _lib.check(_lib.lib().b2p_layernorm(_p(x), C, _p(gamma), _p(beta), eps, T, C, _p(out16), 2 * C if split else C,
                                        _p(out32), C, int(split), _stream()))


def dwconv_ln(x, B, H, W, C, w9c, bias, y, gamma, beta, out16, eps=1e-5, split=False, v3=False):
    """y = dwconv3x3(x) + bias + x (fp32) and out16 = LayerNorm(y) as the next GEMM operand, one kernel.  v3: strip kernel
    with register-resident weights (csrc/florence_simt.cu; shapes it does not cover fall back to the per-token kernel)."""
    _lib.check(_lib.lib().b2p_dwconv_ln(_p(x), B, H, W, C, _p(w9c), _p(bias), _p(y), _p(gamma), _p(beta), eps, _p(out16),
                                        int(bool(split)) | (4 if v3 else 0), _stream()))


def window_attn(qkv32, qkv_bias, B, H, W, C, heads, out, win=12, split=False, v3=False):
    """v3: maps no larger than one window run one CTA per (image, head group) (csrc/florence_simt.cu)."""
    _lib.check(_lib.lib().b2p_window_attn(_p(qkv32), _p(qkv_bias), B, H, W, C, heads, win, _p(out),
                                          int(bool(split)) | (4 if v3 else 0), _stream()))


def channel_attn(qkv32, B, N, C, groups, out, split=False, v3=False):
    """v3: register-tiled kernel (csrc/florence_simt.cu)."""
    _lib.check(_lib.lib().b2p_channel_attn(_p(qkv32), B, N, C, groups, _p(out), int(bool(split)) | (4 if v3 else 0), _stream()))


def mha(q, ldq, k, v, ldk, B, Lq, Lk, heads, out, ldo, split=False, v3=False):
    """v3: sequences of <= 16 keys run one warp per (batch, head) with K / V in registers (csrc/florence_simt.cu)."""
    _lib.check(_lib.lib().b2p_mha(_p(q), ldq, _p(k), _p(v), ldk, B, Lq, Lk, heads, _p(out), ldo,
                                  int(bool(split)) | (4 if v3 else 0), _stream()))


def mha_cached(q, ldq, knew, vnew, ldnew, kcache, vcache, tmax, step, B, heads, out, ldo, split=False):
    _lib.check(_lib.lib().b2p_mha_cached(_p(q), ldq, _p(knew), _p(vnew), ldnew, _p(kcache), _p(vcache), tmax, _p(step),
                                         B, heads, _p(out), ldo, int(split), _stream()))


def encoder_embed(img, n_img, E32, prompt, n_prompt, P, B, C, out):
    _lib.check(_lib.lib().b2p_encoder_embed(_p(img), n_img, _p(E32), _p(prompt), n_prompt, _p(P), B, C, _p(out), _stream()))


def decoder_embed(E32, seq, seq_ld, step, P, B, C, out):
    _lib.check(_lib.lib().b2p_decoder_embed(_p(E32), _p(seq), seq_ld, _p(step), _p(P), B, C, _p(out), _stream()))


def projector_prep(x, pos, B, HW, C, out, split=False):
    _lib.check(_lib.lib().b2p_projector_prep(_p(x), _p(pos), B, HW, C, _p(out), int(split), _stream()))


def greedy_pick(logits, ld, V, B, seq, seq_ld, finished, step, ngram, forced_bos, forced_eos, eos, pad, max_len,
                dump=None, n_unfinished=None):
    _lib.check(_lib.lib().b2p_greedy_pick(_p(logits), ld, V, B, _p(seq), seq_ld, _p(finished), _p(step), ngram,
                                          forced_bos, forced_eos, eos, pad, max_len, _p(dump), _p(n_unfinished),
                                          _stream()))


def step_advance(step):
    _lib.check(_lib.lib().b2p_step_advance(_p(step), _stream()))
