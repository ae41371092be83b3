"""Live (no profiler) per-op cost of the caption plan and the detector plan: every recorded launch is captured alone in a
CUDA graph of REPS back-to-back copies and timed with CUDA events (L2-warm, launch overhead amortised by the graph).
  python tools/time_ops.py [florence|yolo|all] [K=416] > gpurun_out/ops.txt
Output: one line per op (index, C-ABI entry point, key arguments, us per launch) and per-entry-point totals per stage."""
import collections, sys
sys.path.insert(0, ".")
import torch
from omniparser_b200 import ops

REPS = 20
what = sys.argv[1] if len(sys.argv) > 1 else "all"
K = int(sys.argv[2]) if len(sys.argv) > 2 else 416
dev = torch.device("cuda", 0)

_last = [None]


def _wrap(name):
    fn = getattr(ops, name)

    def w(*a, **k):
        desc = []
        for x in a:
            if isinstance(x, (int, float)):
                desc.append(str(x))
            elif isinstance(x, ops.Map):
                desc.append(f"map{x.B}x{x.H}x{x.W}x{x.C}")
        _last[0] = (name, " ".join(desc[:8]))
        return fn(*a, **k)
    return w


for n in ("gemm", "conv1x1", "conv3x3", "adown_pool", "maxpool_s1", "upsample2x", "im2col3x3", "cbfuse", "im2col_u8", "layernorm",
          "dwconv_ln", "window_attn", "channel_attn", "mha", "mha_cached", "encoder_embed", "decoder_embed", "projector_prep",
          "greedy_pick", "step_advance", "resize_u8"):
    setattr(ops, n, _wrap(n))


def time_ops(lst, stage):
    st = torch.cuda.Stream(device=dev)
    tot = collections.defaultdict(lambda: [0, 0.0])
    total = 0.0
    with torch.cuda.stream(st):
        for i, f in enumerate(lst):
            f(); f()
            st.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                for _ in range(REPS):
                    f()
            g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            g.replay()
            e1.record(st)
            st.synchronize()
            us = 1e3 * e0.elapsed_time(e1) / REPS
            name, desc = _last[0]
            print(f"{stage} {i:4d} {name:16s} {us:8.2f} us  {desc}")
            tot[name][0] += 1; tot[name][1] += us
            total += us
            del g
    print(f"== {stage}: {len(lst)} ops, sum {total:.1f} us (back-to-back, per-op)")
    for n, (c, u) in sorted(tot.items(), key=lambda kv: -kv[1][1]):
        print(f"== {stage} {n:16s} n={c:4d} {u:9.1f} us  avg {u / c:7.2f}")
    sys.stdout.flush()


if what in ("florence", "all"):
    from omniparser_b200.florence_engine import FlorencePlan, FlorenceWeights
    from standin import florence as FS
    fl = FS.florence_standin(0)
    w = FlorenceWeights(fl.state_dict(), dev, FS.GEN, "fp16x3")
    del fl
    plan = FlorencePlan(w, K, 8, FS.PROMPT_IDS, use_graph=False)
    plan.crops.random_(0, 255)
    plan.encode()
    plan.reset_decode(K)
    plan.decode_step()
    torch.cuda.synchronize()
    time_ops(plan.enc_ops, "enc")
    time_ops(plan.dec_ops + [lambda: plan.pick(None)], "dec")

if what in ("yolo", "all"):
    from omniparser_b200.yolo_engine import YoloPlan, YoloWeights
    from standin.yolo_weights import yolo_standin
    yw = YoloWeights(yolo_standin(0).state_dict(), dev)
    yp = YoloPlan(yw, 8, 640, 640, use_graph=False)
    yp.canvas.random_(0, 255)
    yp.run()
    torch.cuda.synchronize()
    time_ops(yp.ops, "yolo")
