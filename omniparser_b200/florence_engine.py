"""Florence-2 icon captioner on the B200 kernels (replaces ``model.generate`` at ref:util/utils.py:125).

DaViT tower -> projector -> BART encoder run once per batch of crops; the greedy decoder runs one fused step per
token (KV cache, cross-attention over precomputed K/V, tied LM head, HF logits processors and argmax on device)
replayed as a CUDA graph whose kernels read the step index from device memory.  GEMM operands are fp16, every
residual stream / LayerNorm / softmax is fp32.  Weight names follow ``transformers`` 5.5 ``models/florence2``.

Only the reference's CUDA-branch input mode is planned here: 64x64 crops, ``do_resize=False`` -> 2x2 final map ->
5 image tokens (ref:util/utils.py:120-121; SURVEY.md finding 3).
"""
from __future__ import annotations

import os
from typing import Dict, List

import numpy as np
import torch

from . import ops
from .ops import ACT_GELU, ACT_NONE

IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)


def _h(t, dev):
    return t.detach().to(device=dev, dtype=torch.float16).contiguous()


def _wpack(w2d, dev, x3):
    """[N, K] fp32 -> fp16 GEMM operand.  x3: [W_hi(K) | W_lo(K)] (pairs with activations [A_hi(K) | A_lo(K)])."""
    w2d = w2d.detach().float()
    hi = w2d.half()
    if not x3:
        return hi.contiguous().to(dev)
    lo = (w2d - hi.float()).half()
    return torch.cat([hi, lo], 1).contiguous().to(dev)


def _f(t, dev):
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


class _Lin:
    def __init__(self, sd, name, dev, cat: List[str] | None = None, x3=False):
        if cat:
            w = torch.cat([sd[f"{name}.{c}.weight"] for c in cat], 0)
            b = torch.cat([sd[f"{name}.{c}.bias"] for c in cat], 0)
        else:
            w = sd[name + ".weight"]
            b = sd.get(name + ".bias")
        self.w = _wpack(w, dev, x3)
        self.b = _f(b, dev) if b is not None else None
        self.N = self.w.shape[0]
        self.K = self.Klog = w.shape[1]          # logical reduction size (the packed row is 2K wide in fp16x3 mode)


class _LN:
    def __init__(self, sd, name, dev):
        self.g, self.b = _f(sd[name + ".weight"], dev), _f(sd[name + ".bias"], dev)


class FlorenceWeights:
    def __init__(self, sd: Dict[str, torch.Tensor], device, gen_cfg: dict, precision: str = "fp16x3"):
        """precision: "fp16x3" (parity grade: fp16 hi/lo operand split, three tensor-core products per term,
        fp32 accumulate -> near-fp32 GEMMs) or "fp16" (single fp16 product; ~5e-3 logit drift)."""
        assert precision in ("fp16", "fp16x3")
        from .yolo_engine import _TrackedState
        sd = _TrackedState(sd)
        dev = device
        self.device = dev
        self.x3 = x3 = precision == "fp16x3"
        self.precision = precision
        self.gen = dict(gen_cfg)
        V = "model.vision_tower."
        self.dims = (128, 256, 512, 1024)
        self.heads = (4, 8, 16, 32)
        self.groups = (4, 8, 16, 32)
        self.depths = tuple(sum(1 for k in sd if k.startswith(f"{V}blocks.{s}.") and k.endswith("spatial_block.norm1.weight")) for s in range(4))
        self.conv_embed, self.conv_norm, self.blocks = [], [], []
        for s in range(4):
            w = sd[f"{V}convs.{s}.conv.weight"].float()
            co = w.shape[0]
            m = w.permute(0, 2, 3, 1).reshape(co, -1)   # (ky,kx,c)
            lin = type("W", (), {})()
            if s == 0:
                m = torch.cat([m, torch.zeros(co, 160 - m.shape[1])], 1)
                wp = _wpack(m, dev, x3)
                lin.w_col = wp
            else:
                t = w.permute(0, 2, 3, 1)                      # [co, 3, 3, ci]
                hi = t.half()
                lo = (t - hi.float()).half()
                # implicit-GEMM conv: per tap [hi(ci) | lo(ci)]; im2col + GEMM route: [hi: 9*ci | lo: 9*ci]
                wp = (torch.cat([hi, lo], 3) if x3 else hi).reshape(co, -1).contiguous().to(dev)
                lin.w_col = _wpack(m, dev, x3)
            lin.w, lin.b, lin.N, lin.K, lin.Klog = wp, _f(sd[f"{V}convs.{s}.conv.bias"], dev), co, m.shape[1], m.shape[1]
            self.conv_embed.append(lin)
            self.conv_norm.append(_LN(sd, f"{V}convs.{s}.norm", dev))
            stage = []
            for d in range(self.depths[s]):
                blk = {}
                for kind, attn in (("spatial_block", "window_attn"), ("channel_block", "channel_attn")):
                    p = f"{V}blocks.{s}.{d}.{kind}."
                    e = dict(
                        dw1_w=_f(sd[p + "conv1.weight"].reshape(-1, 9).t(), dev), dw1_b=_f(sd[p + "conv1.bias"], dev),
                        dw2_w=_f(sd[p + "conv2.weight"].reshape(-1, 9).t(), dev), dw2_b=_f(sd[p + "conv2.bias"], dev),
                        n1=_LN(sd, p + "norm1", dev), n2=_LN(sd, p + "norm2", dev),
                        qkv=_Lin(sd, p + attn + ".qkv", dev, x3=x3), proj=_Lin(sd, p + attn + ".proj", dev, x3=x3),
                        fc1=_Lin(sd, p + "ffn.fc1", dev, x3=x3), fc2=_Lin(sd, p + "ffn.fc2", dev, x3=x3))
                    blk[kind] = e
                stage.append(blk)
            self.blocks.append(stage)
        P = "model.multi_modal_projector."
        self.img_proj = _Lin(sd, P + "image_projection", dev, x3=x3)
        self.img_norm = _LN(sd, P + "image_proj_norm", dev)
        col, row = sd[P + "image_position_embed.column_embeddings.weight"].float(), sd[P + "image_position_embed.row_embeddings.weight"].float()
        temporal = sd[P + "visual_temporal_embed.pos_idx_to_embed"].float()[0]
        self._pos_tables = (col, row, temporal)
        L = "model.language_model."
        self.E32 = _f(sd[L + "shared.weight"], dev)
        self.E16 = _wpack(sd[L + "shared.weight"], dev, x3)
        self.vocab = self.E16.shape[0]
        self.enc_pos = _f(sd[L + "encoder.embed_positions.weight"], dev)
        self.dec_pos = _f(sd[L + "decoder.embed_positions.weight"], dev)
        self.enc_ln_emb = _LN(sd, L + "encoder.layernorm_embedding", dev)
        self.dec_ln_emb = _LN(sd, L + "decoder.layernorm_embedding", dev)
        self.enc_layers, self.dec_layers = [], []
        n_enc = 1 + max(int(k.split(".")[4]) for k in sd if k.startswith(L + "encoder.layers."))
        n_dec = 1 + max(int(k.split(".")[4]) for k in sd if k.startswith(L + "decoder.layers."))
        for i in range(n_enc):
            p = f"{L}encoder.layers.{i}."
            self.enc_layers.append(dict(qkv=_Lin(sd, p + "self_attn", dev, ["q_proj", "k_proj", "v_proj"], x3=x3),
                                        o=_Lin(sd, p + "self_attn.out_proj", dev, x3=x3), ln1=_LN(sd, p + "self_attn_layer_norm", dev),
                                        fc1=_Lin(sd, p + "fc1", dev, x3=x3), fc2=_Lin(sd, p + "fc2", dev, x3=x3), ln2=_LN(sd, p + "final_layer_norm", dev)))
        for i in range(n_dec):
            p = f"{L}decoder.layers.{i}."
            self.dec_layers.append(dict(qkv=_Lin(sd, p + "self_attn", dev, ["q_proj", "k_proj", "v_proj"], x3=x3),
                                        o=_Lin(sd, p + "self_attn.out_proj", dev, x3=x3), ln1=_LN(sd, p + "self_attn_layer_norm", dev),
                                        cq=_Lin(sd, p + "encoder_attn.q_proj", dev, x3=x3), ckv=_Lin(sd, p + "encoder_attn", dev, ["k_proj", "v_proj"], x3=x3),
                                        co=_Lin(sd, p + "encoder_attn.out_proj", dev, x3=x3), ln2=_LN(sd, p + "encoder_attn_layer_norm", dev),
                                        fc1=_Lin(sd, p + "fc1", dev, x3=x3), fc2=_Lin(sd, p + "fc2", dev, x3=x3), ln3=_LN(sd, p + "final_layer_norm", dev)))
        # u8 -> normalised pixel table: rescale 1/255 then (x - mean) / std in fp32 (CLIP image processor order)
        lut = np.empty((3, 256), np.float32)
        for c in range(3):
            lut[c] = (np.arange(256, dtype=np.float32) * np.float32(1.0 / 255.0) - np.float32(IMAGENET_MEAN[c])) / np.float32(IMAGENET_STD[c])
        self.lut = torch.from_numpy(lut).to(dev)
        # the whole checkpoint must have been consumed; tied copies of the embedding are checked, not silently dropped
        shared = sd[L + "shared.weight"]
        for tied in (L + "encoder.embed_tokens.weight", L + "decoder.embed_tokens.weight", "lm_head.weight"):
            if tied in sd and not (sd[tied].shape == shared.shape and torch.equal(sd[tied], shared)):
                raise ValueError(f"{tied} is not tied to the shared embedding: untied heads are not on this path")
        if "final_logits_bias" in sd and bool((sd["final_logits_bias"] != 0).any()):
            raise ValueError("non-zero final_logits_bias is not supported (Florence-2 checkpoints carry zeros)")
        left = sorted(k for k in sd if k not in sd.used)
        if left:
            raise KeyError(f"Florence-2 checkpoint has {len(left)} parameters this loader does not know: {left[:8]} ...")

    def pos_table(self, h, w):
        col, row, temporal = self._pos_tables
        pos = torch.cat([col[:w].unsqueeze(0).repeat(h, 1, 1), row[:h].unsqueeze(1).repeat(1, w, 1)], -1)
        return _f(pos.reshape(h * w, -1) + temporal[None], self.device)


POOL_DEFAULT = "1"     # pooled layout: validated against the GPU parity tests (round 2); B2P_BUFFER_POOL=0 restores one buffer per intermediate


class FlorencePlan:
    """Buffers + launch sequences for a fixed number of crop rows K (64x64 crops)."""

    D = 768
    HEADS = 12

    def __init__(self, w: FlorenceWeights, K: int, max_new_tokens: int, prompt_ids: List[int], use_graph=True, size: int = 64, instance: int = 0):
        """instance: plans of different instances own disjoint buffers and capture streams (split-K scratch is keyed by
        stream), so they may run concurrently on different streams.  size = 64: the reference's CUDA branch (crops fed un-resized, 5 image tokens, ref:util/utils.py:121);
        size = 768: its CPU branch (CLIP processor bicubic resize of every crop to 768x768, 577 image tokens, :123)."""
        assert size in (64, 768)
        self.S = size
        self.tag = f"florence{instance}"
        self.warmed = False
        import threading
        self.lock = threading.Lock()
        self.w, self.K, self.dev = w, K, w.device
        self.x3 = w.x3
        self.KX = 2 if w.x3 else 1
        self.T = max_new_tokens
        self.max_len = max_new_tokens + 1
        dev = self.dev
        self.use_graph = use_graph and os.environ.get("B2P_NO_GRAPH") is None   # eager launches for profiling
        self.crops = torch.zeros((K, 64, 64, 3), dtype=torch.uint8, device=dev)
        self.prompt = torch.tensor(prompt_ids, dtype=torch.int32, device=dev)
        self.n_prompt = len(prompt_ids)
        self.n_img = (size // 32) ** 2 + 1
        self.L = self.n_img + self.n_prompt
        self.seq = torch.zeros((K, self.max_len + 1), dtype=torch.int32, device=dev)
        self.finished = torch.zeros((K,), dtype=torch.int32, device=dev)
        # row pitch padded to 8 floats so the LM-head epilogue takes the 16-byte vector store path (51290 is not)
        self._logits_buf = torch.zeros((K, (w.vocab + 7) // 8 * 8), dtype=torch.float32, device=dev)
        self.logits = self._logits_buf[:, :w.vocab]
        self.enc_ops, self.dec_ops = [], []
        self._pools = {}
        # B2P_BUFFER_POOL=1: re-use intermediates across blocks / layers (see _pool); 0 = one buffer per intermediate
        self.pool = os.environ.get("B2P_BUFFER_POOL", POOL_DEFAULT) != "0"
        self.flops_enc = 0   # logical (useful) FLOPs; the fp16x3 mode executes 3x this on the tensor cores
        self.flops_dec = 0
        self._build_vision_encoder()
        self._build_decoder()
        self.g_enc = None
        self.g_enc_nr = None

    # ------------------------------------------------------------------ helpers
    def _e(self, *shape, dt=torch.float32):
        return torch.zeros(shape, dtype=dt, device=self.dev)   # zeros: recycled allocator blocks may hold NaN patterns

    def _act(self, T, C):
        """fp16 GEMM-operand buffer for T rows of logical width C ([hi(C) | lo(C)] in fp16x3 mode)."""
        return torch.zeros((T, self.KX * C), dtype=torch.float16, device=self.dev)

    def _pool(self, role, T, C, act=False):
        """One buffer per (role, shape) for the whole plan: the blocks of a DaViT stage / the BART encoder layers run one after
        the other, so block i+1 re-uses the intermediates of block i (a plan at 416 crops drops from ~7.5 GB to ~1.5 GB, and
        caption grouping / a third lane / many crop-count buckets stop exhausting HBM).  Roles are chosen so that no kernel
        reads a buffer it writes: see the liveness notes at the call sites."""
        if not self.pool:
            return self._act(T, C) if act else self._e(T, C)
        key = (role, T, C, act)
        if key not in self._pools:
            self._pools[key] = self._act(T, C) if act else self._e(T, C)
        return self._pools[key]

    def _gemm(self, lst, a, lin, out, act=ACT_NONE, res=None, enc=True, split=False):
        M = a.shape[0]
        assert a.shape[1] == self.KX * lin.K, (a.shape, lin.K)
        f = 2 * M * lin.N * lin.Klog
        if enc:
            self.flops_enc += f
        else:
            self.flops_dec += f
        lst.append(lambda: ops.gemm(a, a.stride(0), lin.w, M, lin.N, lin.K, out, out.stride(0), lin.b, res,
                                    res.stride(0) if res is not None else 0, act, out_f32=(out.dtype == torch.float32),
                                    split=split, x3=self.x3))

    def _ln(self, lst, x, ln, T, C, o16=None, o32=None):
        lst.append(lambda: ops.layernorm(x, ln.g, ln.b, T, C, o16, o32, split=self.x3))

    # ------------------------------------------------------------------ DaViT + projector + BART encoder
    def _build_vision_encoder(self):
        w, K, ops_, x3, S = self.w, self.K, self.enc_ops, self.x3, self.S
        if S == 64:
            src = self.crops
        else:   # Pillow-exact bicubic 64x64 -> SxS on the u8 crops (what the HF CLIP image processor does on the host)
            self.crops_in = torch.zeros((K, S, S, 3), dtype=torch.uint8, device=self.dev)
            tmp = torch.empty((K, 64, S, 3), dtype=torch.uint8, device=self.dev)
            ops_.append(lambda: ops.resize_u8(self.crops, K, 64, 64, S, S, 1, tmp, self.crops_in))
            src = self.crops_in
        H = S // 4
        T = K * H * H
        A0 = self._act(T, 160)
        ops_.append(lambda: ops.im2col_u8(src, K, S, S, 7, 4, 3, 160, w.lut, A0, split=x3))
        y = self._e(T, 128)
        self._gemm(ops_, A0, w.conv_embed[0], y)
        x = self._e(T, 128)
        self._ln(ops_, y, w.conv_norm[0], T, 128, None, x)
        for s in range(4):
            C = w.dims[s]
            if s > 0:
                Cp = w.dims[s - 1]
                hmap = ops.new_map(K, H, H, self.KX * Cp, self.dev)
                self._ln(ops_, x, w.conv_norm[s], T, Cp, hmap.buf, None)
                H //= 2
                T = K * H * H
                xo = ops.new_map(K, H, H, C, self.dev, torch.float32)
                ce = w.conv_embed[s]
                if H * H <= 32:
                    # 4x4 / 2x2 output maps (64x64-crop mode): a 128-pixel implicit-GEMM tile would be 8x / 32x padding, so
                    # gather the taps explicitly (row copies) and run the dense GEMM on [T, 9*Cs]
                    col = torch.empty((T, 9 * hmap.C), dtype=torch.float16, device=self.dev)
                    ops_.append(lambda hmap=hmap, col=col: ops.im2col3x3(hmap, 2, col, halves=self.KX))
                    xv = xo.buf.view(T, C)
                    lin = type("W", (), {})()
                    lin.w, lin.b, lin.N, lin.K, lin.Klog = ce.w_col, ce.b, C, 9 * Cp, 9 * Cp
                    self._gemm(ops_, col, lin, xv)
                else:
                    self.flops_enc += 2 * T * C * 9 * Cp
                    ops_.append(lambda hmap=hmap, xo=xo, ce=ce: ops.conv3x3(hmap, ce.w, xo, 2, ce.b, None, ACT_NONE, out_f32=True, x3=x3))
                x = xo.buf.view(T, C)
            # Buffer roles of a stage (fp32 [T, C] unless noted); every block re-uses them:
            #   xA: x1 = x + dw1(x), x3 = x2 + dw2(x2)      xB: x2 = proj(a) + x1, x4 = fc2(f) + x3 (the block output)
            #   act (fp16 operand): h = LN(x1) -> a = attention(qkv) -> h2 = LN(x3)      qkv [T, 3C]      f (fp16 operand, 4C)
            # Liveness: dw1 reads the block input (xB or the stage's fresh patch-embed output) and writes xA; the proj GEMM reads
            # a + residual xA and writes xB; dw2 reads xB, writes xA (x1 is dead: proj consumed it) and act (a is dead); fc2
            # reads f + residual xA and writes xB (x2 is dead: dw2 consumed it).  h dies at the qkv GEMM, before attention writes a.
            for blk in w.blocks[s]:
                for kind in ("spatial_block", "channel_block"):
                    e = blk[kind]
                    xA, xB = self._pool("xA", T, C), self._pool("xB", T, C)      # without pooling: fresh buffers per block
                    act_, qkv, f = self._pool("act", T, C, act=True), self._pool("qkv", T, 3 * C), self._pool("f", T, 4 * C, act=True)
                    x1, h = xA, act_
                    ops_.append(lambda x=x, x1=x1, h=h, e=e, H=H, C=C: ops.dwconv_ln(x, K, H, H, C, e["dw1_w"], e["dw1_b"], x1,
                                                                                 e["n1"].g, e["n1"].b, h, split=x3, v3=True))
                    self._gemm(ops_, h, e["qkv"], qkv)
                    a = act_
                    if kind == "spatial_block":
                        hd = w.heads[s]
                        ops_.append(lambda qkv=qkv, a=a, e=e, H=H, C=C, hd=hd: ops.window_attn(qkv, e["qkv"].b, K, H, H, C, hd, a, split=x3, v3=True))
                    else:
                        gr = w.groups[s]
                        ops_.append(lambda qkv=qkv, a=a, H=H, C=C, gr=gr: ops.channel_attn(qkv, K, H * H, C, gr, a, split=x3, v3=True))
                    x2 = xB
                    self._gemm(ops_, a, e["proj"], x2, res=x1)
                    x3_, h2 = xA, act_
                    ops_.append(lambda x2=x2, x3_=x3_, h2=h2, e=e, H=H, C=C: ops.dwconv_ln(x2, K, H, H, C, e["dw2_w"], e["dw2_b"], x3_,
                                                                                      e["n2"].g, e["n2"].b, h2, split=x3, v3=True))
                    self._gemm(ops_, h2, e["fc1"], f, act=ACT_GELU, split=x3)
                    x4 = xB
                    self._gemm(ops_, f, e["fc2"], x4, res=x3_)
                    x = x4
        self.vision_out = x                     # [K*HW, 1024] fp32, H = 2
        HW = H * H
        pos = w.pos_table(H, H)
        pp = self._act(K * (HW + 1), 1024)
        ops_.append(lambda x=x: ops.projector_prep(x, pos, K, HW, 1024, pp, split=x3))
        pf = self._e(K * (HW + 1), self.D)
        self._gemm(ops_, pp, w.img_proj, pf)
        self.img_feat = self._e(K * (HW + 1), self.D)
        self._ln(ops_, pf, w.img_norm, K * (HW + 1), self.D, None, self.img_feat)
        assert HW + 1 == self.n_img
        # BART encoder
        L, D = self.L, self.D
        TE = K * L
        e0 = self._e(TE, D)
        ops_.append(lambda: ops.encoder_embed(self.img_feat, self.n_img, w.E32, self.prompt, self.n_prompt, w.enc_pos, K, D, e0))
        x = self._e(TE, D)
        h = self._act(TE, D)
        self._ln(ops_, e0, w.enc_ln_emb, TE, D, h, x)
        # encoder layers re-use five buffers: qkv; a (the fp16 operand buffer h: h dies at the qkv GEMM, before attention writes
        # a, and a dies at the out-proj GEMM, before LayerNorm writes the next h); y (GEMM + residual output, consumed by the
        # LayerNorm that follows); x (the LayerNorm output overwrites the residual the GEMM has already consumed); f
        for lay in w.enc_layers:
            qkv, f = self._pool("eqkv", TE, 3 * D), self._pool("ef", TE, 4 * D, act=True)
            self._gemm(ops_, h, lay["qkv"], qkv)
            a = h if self.pool else self._act(TE, D)
            ops_.append(lambda qkv=qkv, a=a: ops.mha(qkv, 3 * D, qkv[:, D:], qkv[:, 2 * D:], 3 * D, K, L, L, self.HEADS, a, a.stride(0), split=x3, v3=True))
            y = self._pool("ey", TE, D)
            self._gemm(ops_, a, lay["o"], y, res=x)
            if not self.pool:
                x, h = self._e(TE, D), self._act(TE, D)
            self._ln(ops_, y, lay["ln1"], TE, D, h, x)
            self._gemm(ops_, h, lay["fc1"], f, act=ACT_GELU, split=x3)
            y = self._pool("ey", TE, D)
            self._gemm(ops_, f, lay["fc2"], y, res=x)
            if not self.pool:
                x, h = self._e(TE, D), self._act(TE, D)
            self._ln(ops_, y, lay["ln2"], TE, D, h, x)
        self.enc_out32, self.enc_out16 = x, h
        # cross-attention K/V of every decoder layer, once per batch (fp32: read by the attention kernel)
        self.cross_kv = []
        for lay in w.dec_layers:
            kv = self._e(TE, 2 * D)
            self._gemm(ops_, h, lay["ckv"], kv)
            self.cross_kv.append(kv)

    # ------------------------------------------------------------------ one greedy decode step
    def _build_decoder(self):
        """The decode step: ~70 small, latency-bound launches over all K crop rows.  (Splitting the rows into concurrent
        chains measured slower on B200, -8 % with 2 chains: every chain re-streams the 0.5 GB of decoder weights.)"""
        w, D, x3, R = self.w, self.D, self.x3, self.K
        g = w.gen
        tmax = self.max_len
        ops_ = self.dec_ops
        seq, finished, logits = self.seq, self.finished, self.logits
        self.step = step = torch.zeros((1,), dtype=torch.int32, device=self.dev)
        self.n_unf = n_unf = torch.zeros((1,), dtype=torch.int32, device=self.dev)
        e0 = self._e(R, D)
        ops_.append(lambda: ops.decoder_embed(w.E32, seq, seq.stride(0), step, w.dec_pos, R, D, e0))
        x = self._e(R, D); h = self._act(R, D)
        self._ln(ops_, e0, w.dec_ln_emb, R, D, h, x)
        for li, lay in enumerate(w.dec_layers):
            qkv = self._e(R, 3 * D)
            self._gemm(ops_, h, lay["qkv"], qkv, enc=False)
            kc = torch.zeros((R, tmax, D), dtype=torch.float32, device=self.dev)
            vc = torch.zeros((R, tmax, D), dtype=torch.float32, device=self.dev)
            a = self._act(R, D)
            ops_.append(lambda qkv=qkv, kc=kc, vc=vc, a=a: ops.mha_cached(qkv, 3 * D, qkv[:, D:], qkv[:, 2 * D:], 3 * D, kc, vc, tmax,
                                                                       step, R, self.HEADS, a, a.stride(0), split=x3))
            y = self._e(R, D)
            self._gemm(ops_, a, lay["o"], y, res=x, enc=False)
            x = self._e(R, D); h = self._act(R, D)
            self._ln(ops_, y, lay["ln1"], R, D, h, x)
            q = self._e(R, D)
            self._gemm(ops_, h, lay["cq"], q, enc=False)
            kv = self.cross_kv[li]
            a2 = self._act(R, D)
            ops_.append(lambda q=q, kv=kv, a2=a2: ops.mha(q, D, kv, kv[:, D:], 2 * D, R, 1, self.L, self.HEADS, a2, a2.stride(0), split=x3))
            y = self._e(R, D)
            self._gemm(ops_, a2, lay["co"], y, res=x, enc=False)
            x = self._e(R, D); h = self._act(R, D)
            self._ln(ops_, y, lay["ln2"], R, D, h, x)
            f = self._act(R, 4 * D)
            self._gemm(ops_, h, lay["fc1"], f, act=ACT_GELU, enc=False, split=x3)
            y = self._e(R, D)
            self._gemm(ops_, f, lay["fc2"], y, res=x, enc=False)
            x = self._e(R, D); h = self._act(R, D)
            self._ln(ops_, y, lay["ln3"], R, D, h, x)
        lm = type("W", (), {})()
        lm.w, lm.b, lm.N, lm.K, lm.Klog = w.E16, None, w.vocab, D, D
        self._gemm(ops_, h, lm, logits, enc=False)
        fb = g.get("forced_bos_token_id")
        fe = g.get("forced_eos_token_id")
        self.pick = lambda dump=None: ops.greedy_pick(logits, logits.stride(0), w.vocab, R, seq, seq.stride(0), finished, step,
                                                      g.get("no_repeat_ngram_size", 0) or 0, -1 if fb is None else fb,
                                                      -1 if fe is None else fe, g["eos_token_id"], g["pad_token_id"], self.max_len,
                                                      dump, n_unf)
        tail = [lambda: self.pick(None), lambda: ops.step_advance(step)]
        self.dec_full = ops_ + tail
        # Steps whose token is forced by the generation config (forced BOS at length 1, forced EOS at the last length:
        # hf:generation/logits_process.py:1552,1597) never look at the logits: the pick kernel writes the forced id without
        # reading them, so those steps replay a graph WITHOUT the LM head (51290 x 768, the largest GEMM of the step).  The
        # decoder layers still run: the KV cache of the step is needed by the following steps.
        self.dec_full_forced = ops_[:-1] + tail
        self.g_dec = None
        self.g_dec_forced = None

    # ------------------------------------------------------------------ running
    def _run(self, lst, key, tag, replay_after_capture=True):
        if not self.use_graph:
            for f in lst:
                f()
            return
        g = getattr(self, key)
        if g is None:
            # first use: one eager pass (lazy one-time setup must not happen inside a capture), capture, and -- unless the
            # caller keeps the eager results (B2P_EAGER_FIRST, debugging) -- the results come from replaying the graph, so
            # every real result of the graph path is produced by the same launch mechanism
            for f in lst:
                f()
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            with ops.CAPTURE_LOCK:   # one capture at a time across the pipeline's threads
                with torch.cuda.graph(g, stream=ops.capture_stream(tag, self.dev), capture_error_mode="thread_local"):
                    for f in lst:
                        f()
            setattr(self, key, g)
            if not replay_after_capture or os.environ.get("B2P_EAGER_FIRST"):
                return
        g.replay()
        ops.count_graph_launches(len(lst))

    def warm(self):
        """Build every CUDA graph of this plan on scratch inputs (call with the GPU otherwise idle: see
        ``PipelinedParser``); real results then only ever come from graph replays."""
        if not self.use_graph:
            return
        self.crops.zero_()
        self.encode()
        self.reset_decode(self.K)
        self.decode_step()
        torch.cuda.current_stream().synchronize()
        self.warmed = True

    def _warm_decode(self):
        """Capture the two decode-step graphs on scratch state (one eager step + capture each), before any real decoding."""
        if not self.use_graph or os.environ.get("B2P_EAGER_FIRST") or (self.g_dec is not None and self.g_dec_forced is not None):
            return
        self._reset_state(self.K)
        self.decode_step()
        self.decode_step(forced=True)     # the LM-head-free graph of the forced steps
        torch.cuda.current_stream().synchronize()

    def encode(self, from_resized: bool = False):
        """from_resized: the SxS crops are already in ``crops_in`` (host-side processor did the bicubic resize)."""
        if from_resized and self.S != 64:
            self._run(self.enc_ops[1:], "g_enc_nr", self.tag)
        else:
            self._run(self.enc_ops, "g_enc", self.tag)

    def reset_decode(self, n_active: int):
        self._warm_decode()
        self._reset_state(n_active)

    def _reset_state(self, n_active: int):
        self.seq.zero_()
        self.seq[:, 0] = self.w.gen["decoder_start_token_id"]
        self.finished.zero_()
        if n_active < self.K:
            self.finished[n_active:] = 1     # padding rows never gate the stop test
        self.step.zero_()
        self.n_unf.fill_(max(0, min(n_active, self.K)))

    def unfinished(self) -> int:
        return int(self.n_unf.item())

    def step_is_forced(self, t: int) -> bool:
        """True if the token of decode step t (0-based) is fixed by the generation config whatever the logits are."""
        g = self.w.gen
        return (t == 0 and g.get("forced_bos_token_id") is not None) or (t == self.T - 1 and g.get("forced_eos_token_id") is not None)

    def decode_step(self, dump=None, force_tokens=None, forced=False):
        """one token for every row; ``force_tokens`` [K] (teacher forcing) overwrites the picked ids.  forced: this step's
        token is forced by the generation config (``step_is_forced``): run the step without the LM head."""
        if dump is None and force_tokens is None:
            lst, key = (self.dec_full_forced, "g_dec_forced") if forced else (self.dec_full, "g_dec")
            self._run(lst, key, self.tag + "_dec0", replay_after_capture=False)
            return
        for f in self.dec_ops:   # eager path used by the parity tests
            f()
        self.pick(dump)
        if force_tokens is not None:
            t = int(self.step.item())
            self.seq[:, t + 1] = force_tokens
        ops.step_advance(self.step)

    def join(self):
        """No-op, kept for callers that synchronise with the decoder before reading ``seq``: the decode step runs on the
        caller's stream, so stream order already covers it."""
