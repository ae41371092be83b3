"""One launch of each SIMT kernel of interest at the bench shapes (416 crops / batch 8), for `ncu --set full`:
  ncu --set full --clock-control none --import-source on -k regex:'dwconv|window_attn|channel_attn|mha|adown|cbfuse|layernorm' \
      -o gpurun_out/simt python tools/prof_simt.py
Prints the label of every launch in order (labels file for tools/ncu_extract.py)."""
import sys
sys.path.insert(0, ".")
import torch
from omniparser_b200 import ops
DEV = "cuda:0"
g = torch.Generator().manual_seed(0)
K = 416
labels = []


def rnd(*shape, dt=torch.float32):
    return torch.randn(*shape, generator=g).to(DEV).to(dt)


def dw(H, C, **kw):
    x = rnd(K, H, H, C); w = rnd(9, C) * 0.2; b = rnd(C); ga = rnd(C); be = rnd(C)
    y = torch.zeros(K * H * H, C, device=DEV); o = torch.zeros(K * H * H, 2 * C, dtype=torch.float16, device=DEV)
    ops.dwconv_ln(x, K, H, H, C, w, b, y, ga, be, o, split=True, **kw)
    labels.append(f"dwconv_ln {H}x{H}x{C} {kw}")


def wa(H, C, heads, v3):
    qkv = rnd(K * H * H, 3 * C); bias = rnd(3 * C); o = torch.zeros(K * H * H, 2 * C, dtype=torch.float16, device=DEV)
    ops.window_attn(qkv, bias, K, H, H, C, heads, o, split=True, v3=v3)
    labels.append(f"window_attn {H}x{H}x{C} v3={v3}")


def ca(N, C, **kw):
    qkv = rnd(K * N, 3 * C); o = torch.zeros(K * N, 2 * C, dtype=torch.float16, device=DEV)
    ops.channel_attn(qkv, K, N, C, C // 32, o, split=True, **kw)
    labels.append(f"channel_attn N={N} C={C} {kw}")


def mh(v3):
    D, L = 768, 13
    qkv = rnd(K * L, 3 * D); o = torch.zeros(K * L, 2 * D, dtype=torch.float16, device=DEV)
    ops.mha(qkv, 3 * D, qkv[:, D:], qkv[:, 2 * D:], 3 * D, K, L, L, 12, o, o.stride(0), split=True, v3=v3)
    labels.append(f"mha L=13 v3={v3}")


dw(4, 512, v3=True); dw(16, 128, v3=True); dw(16, 128)
wa(4, 512, 16, True); wa(4, 512, 16, False); wa(8, 256, 8, True)
ca(16, 512, v3=True); ca(256, 128, v3=True); ca(256, 128)
mh(True); mh(False)
x = ops.new_map(8, 160, 160, 256, DEV); x.buf.normal_()
x1 = ops.new_map(8, 160, 160, 128, DEV); x2 = ops.new_map(8, 80, 80, 128, DEV)
ops.adown_pool(x, x1, x2); labels.append("adown_pool 8x160x160x256")
last = ops.new_map(8, 320, 320, 64, DEV); last.buf.normal_()
out = ops.new_map(8, 320, 320, 64, DEV)
srcs = []
for s in range(5):
    m = ops.new_map(8, 320 >> s, 320 >> s, 64, DEV); m.buf.normal_(); srcs.append(m)
ops.cbfuse(srcs, last, out); labels.append("cbfuse 8x320x320x64 5 srcs")
xl = rnd(106496, 128); ga = rnd(128); be = rnd(128); o32 = torch.zeros(106496, 128, device=DEV)
ops.layernorm(xl, ga, be, 106496, 128, None, o32, split=True); labels.append("layernorm 106496x128 -> fp32")
torch.cuda.synchronize()
print("\n".join(labels))
