"""GPU parity tests of the individual kernels, called through the C-ABI (ctypes) on cuda:0.

Dense contractions are compared with a plain PyTorch fp32 reference on the same fp16-rounded operands
(tolerance: fp32 accumulation order only); byte/index kernels are compared bit-exactly with the oracle
(Pillow / OpenCV / torchvision / oracle.ref_restate)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from omniparser_b200 import ops  # noqa: E402
from oracle import ref_restate as R  # noqa: E402

DEV = "cuda:0"


def _act(x, act):
    if act == ops.ACT_SILU:
        return F.silu(x)
    if act == ops.ACT_GELU:
        return F.gelu(x)
    return x


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (128, 64, 128), (256, 256, 256), (300, 200, 192), (37, 24, 32),
                                   (1000, 320, 160), (129, 1, 256), (4096, 768, 768), (60, 3072, 768),
                                   (480, 1000, 3072), (25600, 128, 32), (13, 51289, 768),
                                   (416, 768, 9216), (416, 2304, 2304), (100, 64, 4608),
                                   # >= one wave of M tiles with N <= 256: the weight-resident path (GemmArgs::bres)
                                   (30000, 64, 64), (40000, 256, 256), (20001, 192, 256), (19000, 16, 32), (25600, 128, 128)])
@pytest.mark.parametrize("cfg", [dict(), dict(bias=True, act=ops.ACT_SILU), dict(bias=True, act=ops.ACT_GELU, res=True),
                                 dict(bias=True, res=True, out_f32=True)])
def test_gemm(M, N, K, cfg):
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N * 3 + K)
    a = (torch.randn(M, K, generator=g) * 0.5).half().to(DEV)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).half().to(DEV)
    bias = torch.randn(N, generator=g).to(DEV) if cfg.get("bias") else None
    odt = torch.float32 if cfg.get("out_f32") else torch.float16
    res = torch.randn(M, N, generator=g).to(DEV).to(odt) if cfg.get("res") else None
    out = ops.linear(a, w, bias, res, cfg.get("act", 0), odt)
    torch.cuda.synchronize()
    ref = a.float() @ w.float().t()
    if bias is not None:
        ref = ref + bias
    ref = _act(ref, cfg.get("act", 0))
    if res is not None:
        ref = ref + res.float()
    tol = 2e-3 if odt == torch.float32 else 1e-2
    err = (out.float() - ref).abs().max().item()
    assert err < tol * max(1.0, ref.abs().max().item()), f"max abs err {err}"


def test_gemm_strided_views():
    """A is a column slice of a wider buffer, out/res are channel slices (concat elimination)."""
    g = torch.Generator(device="cpu").manual_seed(5)
    big = (torch.randn(500, 384, generator=g) * 0.5).half().to(DEV)
    a = big[:, 128:256]
    w = (torch.randn(96, 128, generator=g) / 11).half().to(DEV)
    outbuf = torch.zeros(500, 256, device=DEV, dtype=torch.float16)
    resbuf = torch.randn(500, 160, generator=g).half().to(DEV)
    ops.linear(a, w, None, resbuf[:, 32:128], ops.ACT_SILU, out=outbuf[:, 64:160])
    torch.cuda.synchronize()
    ref = F.silu(a.float() @ w.float().t()) + resbuf[:, 32:128].float()
    assert (outbuf[:, 64:160].float() - ref).abs().max().item() < 1e-2
    assert outbuf[:, :64].abs().max().item() == 0 and outbuf[:, 160:].abs().max().item() == 0


@pytest.mark.parametrize("B,H,W,Cin,Cout,stride", [(1, 20, 20, 64, 128, 1), (2, 20, 20, 512, 256, 1),
                                                    (1, 80, 80, 32, 32, 1), (1, 40, 40, 128, 64, 1),
                                                    (3, 34, 60, 64, 64, 1), (1, 160, 160, 64, 64, 1),
                                                    (1, 40, 40, 256, 64, 2), (2, 80, 80, 128, 128, 2),
                                                    (1, 320, 320, 64, 128, 2), (1, 22, 38, 32, 48, 2),
                                                    (37, 16, 16, 128, 64, 2), (10, 8, 8, 256, 96, 2), (5, 4, 4, 64, 48, 2),
                                                    # weight-resident path: halo (s1) and parity-view (s2) convs with >= 148 tiles
                                                    (4, 160, 160, 32, 32, 1), (2, 160, 160, 64, 64, 1), (8, 80, 80, 64, 64, 1),
                                                    (2, 320, 320, 64, 128, 2), (3, 160, 160, 32, 64, 2), (2, 161, 159, 32, 48, 1)])
def test_conv3x3(B, H, W, Cin, Cout, stride):
    g = torch.Generator(device="cpu").manual_seed(B + H + Cin + Cout + stride)
    ld = Cin + 64
    buf = (torch.randn(B, H, W, ld, generator=g) * 0.5).half().to(DEV)
    x = ops.Map(buf, 32, Cin)
    wt = (torch.randn(Cout, Cin, 3, 3, generator=g) / (3 * Cin ** 0.5)).half()
    wpk = wt.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous().to(DEV)
    bias = torch.randn(Cout, generator=g).to(DEV)
    Ho, Wo = H // stride, W // stride
    out = ops.new_map(B, Ho, Wo, Cout + 32, DEV)
    out.buf.zero_()
    o = out.slice(16, Cout)
    res = None
    if stride == 1 and Cin == Cout:
        res = x
    ops.conv3x3(x, wpk, o, stride=stride, bias=bias, res=res, act=ops.ACT_SILU)
    torch.cuda.synchronize()
    xin = buf[..., 32:32 + Cin].permute(0, 3, 1, 2).float()
    ref = F.silu(F.conv2d(xin, wt.float().to(DEV), bias, stride=stride, padding=1))
    if res is not None:
        ref = ref + xin
    err = (o.torch() - ref).abs().max().item()
    assert err < 1e-2 * max(1.0, ref.abs().max().item()), f"max abs err {err}"
    assert out.buf[..., :16].abs().max().item() == 0 and out.buf[..., 16 + Cout:].abs().max().item() == 0


def test_detect_elementwise_ops():
    g = torch.Generator(device="cpu").manual_seed(11)
    B, H, W, C = 2, 40, 40, 256
    x = ops.Map(torch.randn(B, H, W, C + 32, generator=g).half().to(DEV), 16, C)
    xin = x.torch()
    # ADown pooling
    x1 = ops.new_map(B, H, W, C // 2, DEV)
    x2 = ops.new_map(B, H // 2, W // 2, C // 2, DEV)
    ops.adown_pool(x, x1, x2)
    a = F.avg_pool2d(xin, 2, 1, 0, False, True)
    r1 = F.pad(a[:, :C // 2], (0, 1, 0, 1))
    r2 = F.max_pool2d(a[:, C // 2:], 3, 2, 1)
    assert (x1.torch() - r1).abs().max().item() < 2e-3
    assert (x2.torch() - r2).abs().max().item() < 2e-3
    # maxpool 5
    y = ops.new_map(B, H, W, C, DEV)
    ops.maxpool_s1(x, y, 5)
    assert torch.equal(y.torch(), F.max_pool2d(xin, 5, 1, 2))
    # upsample
    u = ops.new_map(B, 2 * H, 2 * W, C + 8, DEV)
    ops.upsample2x(x, u.slice(8, C))
    assert torch.equal(u.slice(8, C).torch(), F.interpolate(xin, scale_factor=2.0, mode="nearest"))
    # cbfuse: two coarser sources + last
    s1 = ops.Map(torch.randn(B, H // 2, W // 2, 3 * C, generator=g).half().to(DEV), C, C)
    s2 = ops.Map(torch.randn(B, H // 4, W // 4, 2 * C, generator=g).half().to(DEV), 0, C)
    out = ops.new_map(B, H, W, C, DEV)
    ops.cbfuse([s1, s2], x, out)
    ref = F.interpolate(s1.torch(), size=(H, W), mode="nearest") + F.interpolate(s2.torch(), size=(H, W), mode="nearest") + xin
    assert (out.torch() - ref).abs().max().item() < 4e-3
    torch.cuda.synchronize()


def _nms_gpu(boxes, scores, cls, iou, max_det=300, W=1920.0, H=1080.0):
    n = len(boxes)
    cap = max(n, 1)
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(DEV)
    b, s, c = d(boxes.reshape(-1, 4), torch.float32), d(scores, torch.float32), d(cls, torch.int32)
    cnt = torch.tensor([n], dtype=torch.int32, device=DEV)
    keep = torch.full((max_det,), -1, dtype=torch.int32, device=DEV)
    ob = torch.zeros(max_det, 4, device=DEV)
    os_ = torch.zeros(max_det, device=DEV)
    oc = torch.zeros(1, dtype=torch.int32, device=DEV)
    iw, ih = torch.tensor([W], device=DEV), torch.tensor([H], device=DEV)
    ops.batched_nms(b, s, c, cnt, 1, cap, iou, max_det, iw, ih, keep, ob, os_, oc)
    torch.cuda.synchronize()
    k = int(oc.item())
    return keep[:k].cpu().numpy().astype(np.int64), ob[:k].cpu(), os_[:k].cpu()


@pytest.mark.parametrize("n,nc", [(0, 1), (1, 1), (7, 1), (300, 1), (513, 1), (999, 3), (1000, 3), (1001, 3), (2500, 1), (8400, 1)])
def test_nms_bit_exact(n, nc):
    from torchvision.ops import batched_nms
    rng = np.random.default_rng(n + nc)
    xy = rng.uniform(0, 1800, size=(n, 2)).astype(np.float32)
    wh = rng.uniform(0, 200, size=(n, 2)).astype(np.float32)
    boxes = np.concatenate([xy, xy + wh], 1)
    scores = rng.uniform(0.05, 1, size=n).astype(np.float32)
    if 4 < n <= 1000:
        scores[rng.integers(0, n, size=n // 3)] = np.float32(0.5)
        boxes[1] = boxes[0]
        boxes[3, 2:] = boxes[3, :2]
    cls = rng.integers(0, nc, size=n).astype(np.int64)
    for iou in (0.1, 0.7):
        tb, ts, tc = torch.from_numpy(boxes), torch.from_numpy(scores), torch.from_numpy(cls)
        ref = batched_nms(tb, ts, tc, iou)[:300]
        got, ob, os_ = _nms_gpu(boxes, scores, cls, iou)
        assert np.array_equal(ref.numpy(), got), (n, nc, iou)
        rb = tb[ref].clone()
        rb[:, [0, 2]] = rb[:, [0, 2]].clamp(0, 1920)
        rb[:, [1, 3]] = rb[:, [1, 3]].clamp(0, 1080)
        assert torch.equal(rb, ob) and torch.equal(ts[ref], os_)


@pytest.mark.parametrize("size,imgsz", [((1920, 1080), 640), ((1919, 1079), 640), ((3240, 2160), 640),
                                        ((300, 200), 640), ((1920, 1080), (1080, 1920))])
def test_letterbox_bit_exact(size, imgsz):
    rng = np.random.default_rng(3)
    B = 2
    imgs = rng.integers(0, 256, size=(B, size[1], size[0], 3), dtype=np.uint8)
    tw, th, scale, rw, rh, pl, pt = R.letterbox_geometry(size[0], size[1], imgsz)
    src = torch.from_numpy(imgs).to(DEV)
    tmp = torch.empty(B, size[1], rw, 3, dtype=torch.uint8, device=DEV)
    canvas = torch.empty(B, th, tw, 3, dtype=torch.uint8, device=DEV)
    ops.letterbox(src, B, size[1], size[0], rw, rh, tw, th, pl, pt, tmp, canvas)
    torch.cuda.synchronize()
    for b in range(B):
        ref, *_ = R.letterbox_pil(imgs[b], imgsz)
        assert np.array_equal(ref, canvas[b].cpu().numpy())


@pytest.mark.parametrize("B,H,W,C,stride", [(3, 8, 8, 48, 2), (2, 4, 4, 768, 2), (2, 5, 7, 16, 1), (1, 9, 6, 24, 2)])
def test_im2col3x3_exact(B, H, W, C, stride):
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, H, W, C, generator=g).half().to(DEV)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    out = torch.empty(B * Ho * Wo, 9 * C, dtype=torch.float16, device=DEV)
    ops.im2col3x3(ops.Map(x, 0, C), stride, out)
    torch.cuda.synchronize()
    xp = torch.nn.functional.pad(x.cpu().float(), (0, 0, 1, 1, 1, 1))
    ref = torch.stack([xp[:, ky:ky + (Ho - 1) * stride + 1:stride, kx:kx + (Wo - 1) * stride + 1:stride] for ky in range(3) for kx in range(3)], 3)
    assert torch.equal(out.cpu().float(), ref.reshape(B * Ho * Wo, 9 * C))
    if C % 16 == 0:   # fp16x3 pixels [hi(C/2) | lo(C/2)] -> rows [hi: 9*C/2 | lo: 9*C/2]
        ops.im2col3x3(ops.Map(x, 0, C), stride, out, halves=2)
        torch.cuda.synchronize()
        h = C // 2
        ref2 = torch.cat([ref[..., :h].reshape(B * Ho * Wo, 9 * h), ref[..., h:].reshape(B * Ho * Wo, 9 * h)], 1)
        assert torch.equal(out.cpu().float(), ref2)


@pytest.mark.parametrize("filt", [0, 1])
@pytest.mark.parametrize("src_hw,dst_wh", [((64, 64), (768, 768)), ((37, 53), (100, 80)), ((300, 200), (64, 48))])
def test_resize_u8_bit_exact_vs_pillow(filt, src_hw, dst_wh):
    """b2p_resize_u8 == PIL Image.resize (LANCZOS / BICUBIC): the CLIP image processor's resize in the 768 caption mode."""
    from PIL import Image
    rng = np.random.default_rng(11)
    B = 2
    H, W = src_hw
    Wr, Hr = dst_wh
    imgs = rng.integers(0, 256, size=(B, H, W, 3), dtype=np.uint8)
    src = torch.from_numpy(imgs).to(DEV)
    tmp = torch.empty(B, H, Wr, 3, dtype=torch.uint8, device=DEV)
    out = torch.empty(B, Hr, Wr, 3, dtype=torch.uint8, device=DEV)
    ops.resize_u8(src, B, H, W, Wr, Hr, filt, tmp, out)
    torch.cuda.synchronize()
    res = Image.Resampling.BICUBIC if filt else Image.Resampling.LANCZOS
    for b in range(B):
        ref = np.asarray(Image.fromarray(imgs[b]).resize((Wr, Hr), res))
        assert np.array_equal(ref, out[b].cpu().numpy())


def test_crop_resize_bit_exact():
    import cv2
    rng = np.random.default_rng(4)
    H, W = 1080, 1920
    imgs = rng.integers(0, 256, size=(2, H, W, 3), dtype=np.uint8)
    n = 200
    x0 = rng.uniform(0, 0.9, size=n); y0 = rng.uniform(0, 0.9, size=n)
    bw = rng.uniform(0.001, 0.1, size=n); bh = rng.uniform(0.002, 0.15, size=n)
    boxes = np.stack([x0, y0, np.minimum(x0 + bw, 1.0), np.minimum(y0 + bh, 1.0)], 1).astype(np.float32)
    boxes[0] = (np.float32(100 / W), np.float32(100 / H), np.float32(228.5 / W), np.float32(228.5 / H))   # 128x128 -> area path
    boxes[1] = (np.float32(10 / W), np.float32(10 / H), np.float32(74.5 / W), np.float32(74.5 / H))      # 64x64 identity
    boxes[2] = (0.5, 0.5, 0.5, 0.6)   # empty crop
    bimg = rng.integers(0, 2, size=n).astype(np.int32)
    d_img = torch.from_numpy(imgs).to(DEV)
    hw = torch.tensor([[H, W], [H, W]], dtype=torch.int32, device=DEV)
    off = torch.tensor([0, H * W * 3], dtype=torch.int64, device=DEV)
    out = torch.empty(n, 64, 64, 3, dtype=torch.uint8, device=DEV)
    status = torch.empty(n, dtype=torch.int32, device=DEV)
    ops.crop_resize(d_img, hw, off, torch.from_numpy(boxes).to(DEV), torch.from_numpy(bimg).to(DEV), n, 64, out, status)
    torch.cuda.synchronize()
    tb = torch.from_numpy(boxes)
    ints = R.crop_boxes_int(tb, W, H)
    st = status.cpu().numpy()
    for i, (xa, ya, xb, yb) in enumerate(ints):
        crop = imgs[bimg[i]][ya:yb, xa:xb, :]
        if crop.shape[0] == 0 or crop.shape[1] == 0:
            assert st[i] == 1
            continue
        assert st[i] == 0
        assert np.array_equal(cv2.resize(crop, (64, 64)), out[i].cpu().numpy()), (i, crop.shape)


def test_im2col_stem():
    rng = np.random.default_rng(6)
    B, H, W = 2, 64, 96
    img = rng.integers(0, 256, size=(B, H, W, 3), dtype=np.uint8)
    lut = (np.arange(256, dtype=np.float32) / np.float32(255.0))[None].repeat(3, 0).copy()
    for (k, s, p, Kpad) in [(3, 2, 1, 32), (7, 4, 3, 160)]:
        Ho, Wo = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
        out = torch.empty(B * Ho * Wo, Kpad, dtype=torch.float16, device=DEV)
        ops.im2col_u8(torch.from_numpy(img).to(DEV), B, H, W, k, s, p, Kpad, torch.from_numpy(lut).to(DEV), out)
        torch.cuda.synchronize()
        x = torch.from_numpy(img.astype(np.float32) / np.float32(255.0)).permute(0, 3, 1, 2)
        cols = F.unfold(x, k, padding=p, stride=s)   # [B, 3*k*k, L] ordered (c, ky, kx)
        cols = cols.view(B, 3, k * k, Ho * Wo).permute(0, 3, 2, 1).reshape(B * Ho * Wo, k * k * 3)
        got = out.cpu().float()
        assert torch.equal(got[:, :k * k * 3], cols.half().float())
        assert got[:, k * k * 3:].abs().max().item() == 0


def _hilo(t):
    hi = t.half()
    return hi, (t - hi.float()).half()


@pytest.mark.parametrize("M,N,K", [(416, 3072, 768), (300, 256, 2048), (1000, 128, 64), (416, 768, 3072), (6656, 512, 160), (128, 51290, 768)])
def test_gemm_fp16x3_operands(M, N, K):
    """fp16x3 precision mode: A = [hi(K) | lo(K)], W = [hi(K) | lo(K)]; the kernel loads every half once per k-block and
    issues hi*hi + hi*lo + lo*hi -> near-fp32 products; the split epilogue writes the next operand in the same layout
    (small-M cases run the split-K path)."""
    g = torch.Generator(device="cpu").manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    a2 = torch.cat(_hilo(a), 1).to(DEV)
    w2 = torch.cat(_hilo(w), 1).contiguous().to(DEV)
    bias = torch.randn(N, generator=g).to(DEV)
    ref = F.gelu(a.double() @ w.double().t() + bias.cpu().double())
    tol = 2e-5 * max(1.0, ref.abs().max().item())
    if N % 8 == 0:
        out = torch.empty(M, 2 * N, dtype=torch.float16, device=DEV)
        ops.gemm(a2, 2 * K, w2, M, N, K, out, 2 * N, bias, None, 0, ops.ACT_GELU, split=True, x3=True)
        torch.cuda.synchronize()
        got = (out[:, :N].float() + out[:, N:].float()).cpu().double()
        assert (got - ref).abs().max().item() < tol
    res = torch.randn(M, N, generator=g).to(DEV)
    o32 = torch.empty(M, N, dtype=torch.float32, device=DEV)
    ops.gemm(a2, 2 * K, w2, M, N, K, o32, N, bias, res, N, ops.ACT_GELU, out_f32=True, x3=True)
    torch.cuda.synchronize()
    assert (o32.cpu().double() - (ref + res.cpu().double())).abs().max().item() < tol


@pytest.mark.parametrize("B,H,W,Ci,Co", [(3, 16, 16, 128, 256), (2, 24, 24, 64, 96), (5, 8, 8, 256, 512)])
def test_conv3x3_s2_fp16x3_operands(B, H, W, Ci, Co):
    """stride-2 implicit-GEMM conv with [hi(Ci) | lo(Ci)] pixels and [Co][9][hi | lo] weights vs fp64 conv2d."""
    g = torch.Generator(device="cpu").manual_seed(B * H + Ci + Co)
    x = torch.randn(B, H, W, Ci, generator=g)
    w = torch.randn(Co, Ci, 3, 3, generator=g) / (9 * Ci) ** 0.5
    bias = torch.randn(Co, generator=g)
    xm = ops.Map(torch.cat(_hilo(x), 3).contiguous().to(DEV), 0, 2 * Ci)
    wt = w.permute(0, 2, 3, 1)
    wp = torch.cat(_hilo(wt), 3).reshape(Co, -1).contiguous().to(DEV)
    out = ops.new_map(B, H // 2, W // 2, Co, DEV, torch.float32)
    ops.conv3x3(xm, wp, out, 2, bias.to(DEV), None, ops.ACT_NONE, out_f32=True, x3=True)
    torch.cuda.synchronize()
    ref = F.conv2d(x.permute(0, 3, 1, 2).double(), w.double(), bias.double(), stride=2, padding=1).permute(0, 2, 3, 1)
    assert (out.buf.cpu().double() - ref).abs().max().item() < 2e-5 * max(1.0, ref.abs().max().item())


# ---------------------------------------------------------------------------------------------- round-2 SIMT kernels (csrc/florence_simt.cu)
def _pair_val(o, C, split):
    """fp16 activation buffer -> float64 values ([hi | lo] pairs summed)."""
    o = o.double()
    return o[:, :C] + o[:, C:2 * C] if split else o


def _act_close(a, b, C, split):
    va, vb = _pair_val(a.cpu(), C, split), _pair_val(b.cpu(), C, split)
    tol = (4e-6 if split else 1.5e-3) * max(1.0, vb.abs().max().item())     # pairs carry ~22 bits, plain fp16 11
    err = (va - vb).abs().max().item()
    assert err <= tol, (err, tol)


@pytest.mark.parametrize("B,H,C", [(5, 4, 512), (3, 2, 1024), (4, 8, 256), (3, 16, 128), (2, 5, 256), (2, 3, 128)])
@pytest.mark.parametrize("split", [False, True])
def test_dwconv_ln_v3_equals_first_version(B, H, C, split):
    """strip kernel with register-resident weights: y bit-identical (same tap order), LayerNorm output within rounding."""
    g = torch.Generator().manual_seed(B * H + C + 1)
    x = torch.randn(B, H, H, C, generator=g).to(DEV)
    w9c = (torch.randn(9, C, generator=g) * 0.2).to(DEV)
    bias = torch.randn(C, generator=g).to(DEV)
    gam = torch.randn(C, generator=g).to(DEV)
    bet = torch.randn(C, generator=g).to(DEV)
    outs = []
    for v3 in (False, True):
        y = torch.zeros(B * H * H, C, device=DEV)
        o16 = torch.zeros(B * H * H, (2 if split else 1) * C, dtype=torch.float16, device=DEV)
        ops.dwconv_ln(x, B, H, H, C, w9c, bias, y, gam, bet, o16, split=split, v3=v3)
        torch.cuda.synchronize()
        outs.append((y.cpu(), o16))
    assert torch.equal(outs[0][0], outs[1][0])
    _act_close(outs[1][1], outs[0][1], C, split)
    # and against torch (fp64) directly
    xr = x.cpu().double().permute(0, 3, 1, 2)
    yr = F.conv2d(xr, w9c.cpu().double().t().reshape(C, 1, 3, 3), bias.cpu().double(), padding=1, groups=C) + xr
    yr = yr.permute(0, 2, 3, 1).reshape(-1, C)
    assert (outs[1][0].double() - yr).abs().max().item() < 1e-5 * max(1.0, yr.abs().max().item())
    hr = F.layer_norm(yr, (C,), gam.cpu().double(), bet.cpu().double(), 1e-5)
    tol = (2e-5 if split else 1.5e-3) * max(1.0, hr.abs().max().item())
    assert (_pair_val(outs[1][1].cpu(), C, split) - hr).abs().max().item() < tol


def _window_attn_ref(qkv, bias, B, H, W, C, heads, win=12):
    """torch fp64 restatement of hf:models/florence2/modeling_florence2.py:346-383 for a map inside ONE window: the map is
    zero-padded to win x win AFTER the qkv projection's input norm, so padded tokens have qkv = bias."""
    qkv = qkv.double().reshape(B, H, W, 3 * C)
    full = bias.double().reshape(1, 1, 1, 3 * C).repeat(B, win, win, 1).clone()
    full[:, :H, :W] = qkv
    full = full.reshape(B, win * win, 3, heads, C // heads).permute(2, 0, 3, 1, 4)
    q, k, v = full[0] * (C // heads) ** -0.5, full[1], full[2]
    a = torch.softmax(q @ k.transpose(-2, -1), -1) @ v                       # [B, heads, win*win, d]
    a = a.transpose(1, 2).reshape(B, win, win, C)[:, :H, :W]
    return a.reshape(B * H * W, C)


@pytest.mark.parametrize("B,H,C,heads", [(7, 4, 512, 16), (5, 2, 1024, 32), (3, 8, 256, 8), (2, 3, 128, 4), (2, 12, 128, 4)])
@pytest.mark.parametrize("split", [False, True])
def test_window_attn_v3_equals_first_version_and_torch(B, H, C, heads, split):
    g = torch.Generator().manual_seed(B * H + C + 2)
    qkv = torch.randn(B * H * H, 3 * C, generator=g).to(DEV)
    bias = torch.randn(3 * C, generator=g).to(DEV)
    outs = []
    for v3 in (False, True):
        o = torch.zeros(B * H * H, (2 if split else 1) * C, dtype=torch.float16, device=DEV)
        ops.window_attn(qkv, bias, B, H, H, C, heads, o, split=split, v3=v3)
        torch.cuda.synchronize()
        outs.append(o)
    _act_close(outs[1], outs[0], C, split)
    ref = _window_attn_ref(qkv.cpu(), bias.cpu(), B, H, H, C, heads)
    tol = (2e-5 if split else 1.5e-3) * max(1.0, ref.abs().max().item())
    assert (_pair_val(outs[1].cpu(), C, split) - ref).abs().max().item() < tol


@pytest.mark.parametrize("B,H,C,heads", [(3, 16, 128, 4), (2, 20, 128, 4), (2, 13, 256, 8)])
@pytest.mark.parametrize("split", [False, True])
def test_window_attn_multi_window_maps_v3_flag(B, H, C, heads, split):
    """maps larger than one 12x12 window (16x16 in the 64x64-crop mode: windows of 144 / 48 / 48 / 16 real tokens) are not
    covered by the one-window kernel: with the v3 flag the call must fall through to the per-window kernel, same results."""
    g = torch.Generator().manual_seed(B * H + C + 5)
    qkv = torch.randn(B * H * H, 3 * C, generator=g).to(DEV)
    bias = torch.randn(3 * C, generator=g).to(DEV)
    outs = []
    for v3 in (False, True):
        o = torch.zeros(B * H * H, (2 if split else 1) * C, dtype=torch.float16, device=DEV)
        ops.window_attn(qkv, bias, B, H, H, C, heads, o, split=split, v3=v3)
        torch.cuda.synchronize()
        outs.append(o)
    _act_close(outs[1], outs[0], C, split)


@pytest.mark.parametrize("B,N,C", [(7, 16, 512), (5, 4, 1024), (3, 9, 256), (3, 64, 256), (2, 256, 128), (2, 100, 128)])
@pytest.mark.parametrize("split", [False, True])
def test_channel_attn_v3_equals_first_version_and_torch(B, N, C, split):
    g = torch.Generator().manual_seed(B * N + C + 3)
    qkv = torch.randn(B * N, 3 * C, generator=g).to(DEV)
    outs = []
    for v3 in (False, True):
        o = torch.zeros(B * N, (2 if split else 1) * C, dtype=torch.float16, device=DEV)
        ops.channel_attn(qkv, B, N, C, C // 32, o, split=split, v3=v3)
        torch.cuda.synchronize()
        outs.append(o)
    _act_close(outs[1], outs[0], C, split)
    # hf:models/florence2/modeling_florence2.py:228-264
    t = qkv.cpu().double().reshape(B, N, 3, C // 32, 32).permute(2, 0, 3, 1, 4)
    q, k, v = t[0] * N ** -0.5, t[1], t[2]
    a = torch.softmax(q.transpose(-1, -2) @ k, -1)
    ref = (a @ v.transpose(-1, -2)).transpose(-1, -2).transpose(1, 2).reshape(B * N, C)
    tol = (2e-5 if split else 1.5e-3) * max(1.0, ref.abs().max().item())
    assert (_pair_val(outs[1].cpu(), C, split) - ref).abs().max().item() < tol


@pytest.mark.parametrize("B,L", [(9, 13), (3, 16), (4, 5), (2, 3)])
@pytest.mark.parametrize("split", [False, True])
def test_mha_short_equals_first_version(B, L, split):
    """warp-per-(batch, head) attention with K / V in registers == the warp-per-query kernel."""
    D, heads = 768, 12
    g = torch.Generator().manual_seed(B * L + 4)
    qkv = torch.randn(B * L, 3 * D, generator=g).to(DEV)
    outs = []
    for v3 in (False, True):
        o = torch.zeros(B * L, (2 if split else 1) * D, dtype=torch.float16, device=DEV)
        ops.mha(qkv, 3 * D, qkv[:, D:], qkv[:, 2 * D:], 3 * D, B, L, L, heads, o, o.stride(0), split=split, v3=v3)
        torch.cuda.synchronize()
        outs.append(o)
    _act_close(outs[1], outs[0], D, split)
    t = qkv.cpu().double().reshape(B, L, 3, heads, 64).permute(2, 0, 3, 1, 4)
    ref = (torch.softmax(t[0] * 0.125 @ t[1].transpose(-1, -2), -1) @ t[2]).transpose(1, 2).reshape(B * L, D)
    tol = (2e-5 if split else 1.5e-3) * max(1.0, ref.abs().max().item())
    assert (_pair_val(outs[1].cpu(), D, split) - ref).abs().max().item() < tol


# ---------------------------------------------------------------------------------------------- overlap filter (8f-2)
def _overlap_device(px_list, ocr_px_list, W, H, thr, max_det=300, max_ocr=256):
    """b2p_overlap_filter on a batch: px_list[b] fp32 [n_b,4] pixel boxes (NMS output format), ocr_px_list[b] (texts, int boxes)
    -> per screenshot (elements via host_glue.elements_from_flags, crop boxes, crop image ids)."""
    from omniparser_b200 import host_glue
    B = len(px_list)
    f32, i32 = dict(dtype=torch.float32, device=DEV), dict(dtype=torch.int32, device=DEV)
    box = torch.zeros((B, max_det, 4), **f32)
    cnt = torch.zeros((B,), **i32)
    whwh = torch.Tensor([W, H, W, H])
    ocr_elems = []
    oc = torch.zeros((B, max_ocr, 4), **f32)
    ocnt = torch.zeros((B,), **i32)
    for b, (px, (texts, ob)) in enumerate(zip(px_list, ocr_px_list)):
        box[b, :len(px)] = px.to(DEV)
        cnt[b] = len(px)
        el = host_glue.ocr_elements((torch.tensor(ob) / whwh).tolist() if ob else None, texts, W, H)
        ocr_elems.append(el)
        if el:
            oc[b, :len(el)] = torch.tensor([e["bbox"] for e in el], dtype=torch.float32).to(DEV)
        ocnt[b] = len(el)
    state = torch.full((B, max_det), -7, **i32); mask = torch.full((B, max_det, max_ocr // 32), -1, **i32)
    removed = torch.full((B, max_ocr), -7, **i32); ratio = torch.zeros((B, max_det, 4), **f32)
    cbox = torch.zeros((B * max_det, 4), **f32); cimg = torch.zeros((B * max_det,), **i32)
    ccnt = torch.zeros((B + 1,), **i32); arrive = torch.zeros((1,), **i32)
    iw = torch.full((B,), float(W), **f32); ih = torch.full((B,), float(H), **f32)
    for _ in range(2):   # twice: the arrival counter must reset itself
        ops.overlap_filter(box, cnt, B, max_det, iw, ih, oc, ocnt, max_ocr, thr, state, mask, removed, ratio, cbox, cimg, ccnt, arrive)
    torch.cuda.synchronize()
    assert int(arrive.item()) == 0
    out = []
    ccnt = ccnt.cpu().tolist()
    for b in range(B):
        n = len(px_list[b])
        el = host_glue.elements_from_flags(ratio[b, :n].cpu().tolist(), state[b, :n].cpu().tolist(),
                                           mask[b, :n].cpu().numpy().view("uint32"), ocr_elems[b], removed[b, :len(ocr_elems[b])].cpu().tolist())
        out.append(el)
    tot = ccnt[B]
    assert tot == sum(ccnt[:B])
    return out, cbox[:tot].cpu().tolist(), cimg[:tot].cpu().tolist(), ccnt


@pytest.mark.parametrize("thr", [0.7, 0.9, 0.1])
def test_overlap_filter_equals_reference_list_logic(thr):
    """Device overlap filter == the reference-pinned host list logic (host_glue.build_elements, itself equal to the unmodified
    ref:util/utils.py remove_overlap_new in tests/test_host_glue_cpu.py): identical element lists (order, sources, float box
    values, OCR label strings) and identical crop lists, on the adversarial cases of the CPU tests + empty / no-OCR screenshots."""
    from omniparser_b200 import host_glue
    from test_host_glue_cpu import _case, _dense_case, W, H
    whwh = torch.Tensor([W, H, W, H])
    px_list, ocr_list = [], []
    for seed in range(10):
        icons, ob, texts = _dense_case(seed) if seed % 2 else _case(seed)
        px_list.append((icons * whwh).to(torch.float32))
        ocr_list.append((texts, ob))
    px_list.append(torch.zeros((0, 4)));            ocr_list.append((["a"], [[10, 10, 60, 30]]))     # no detections
    px_list.append(px_list[0].clone());             ocr_list.append(([], []))                          # no OCR
    px_list.append(px_list[1][:1].clone());         ocr_list.append(ocr_list[1])
    dup_t, dup_b = ocr_list[3]
    px_list.append(px_list[3].clone());             ocr_list.append((dup_t + [dup_t[0]] * 2, dup_b + [dup_b[0]] * 2))   # equal OCR dicts
    got, cbox, cimg, ccnt = _overlap_device(px_list, ocr_list, W, H, thr)
    exp_box, exp_img = [], []
    labelled = 0
    for b, (px, (texts, ob)) in enumerate(zip(px_list, ocr_list)):
        xyxy = (px / whwh).tolist()
        oratio = (torch.tensor(ob) / whwh).tolist() if ob else None
        ref, _ = host_glue.build_elements(xyxy, oratio, texts, W, H, thr)
        assert got[b] == ref, f"screenshot {b}: element lists differ"
        labelled += sum(e["source"] == "box_yolo_content_ocr" for e in ref)
        for e in ref:
            if e["content"] is None:
                exp_box.append([float(np.float32(v)) for v in e["bbox"]]); exp_img.append(b)
    assert labelled > 0
    assert cbox == exp_box and cimg == exp_img
