"""CPU dry run of the launch plans: the C library is replaced by a recorder that type-checks every call against the ctypes
prototypes (``_lib.PROTOTYPES`` = include/b200parse.h) and re-states the argument checks of the C side (row pitches vs
logical sizes, fp16x3 flags), so a slip in the host-side plumbing (argument order, a stride that still assumes another
operand layout, a flag that is not forwarded) fails here and not only on the GPU box.  No arithmetic runs."""
import contextlib
import ctypes as C

import pytest
import torch

from omniparser_b200 import _lib, ops
from standin import florence as FS


class _Stream:
    cuda_stream = 0

    def __init__(self, *a, **k):
        pass

    def synchronize(self):
        pass

    def wait_stream(self, other):
        pass


class _Recorder:
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        res, argtypes = _lib.PROTOTYPES[name]

        def f(*args):
            assert len(args) == len(argtypes), f"{name}: {len(args)} arguments, prototype has {len(argtypes)}"
            vals = []
            for t, a in zip(argtypes, args):
                t.from_param(a)                      # raises if the Python value cannot become this C type
                vals.append(a.value if hasattr(a, "value") else a)
            self.calls.append((name, vals))
            _check(name, vals)
            return 0
        return f


def _check(name, a):
    """the argument checks gemm_launch / the SIMT launchers make on the device side, restated"""
    if name == "b2p_gemm":
        _A, lda, _B, M, N, K, _out, ldc, _bias, _res, ldr, act, flags, _st = a
        x3, split, f32 = bool(flags & 8), bool(flags & 4), bool(flags & 2)
        assert M > 0 and N > 0 and K % 8 == 0
        assert lda >= (2 if x3 else 1) * K, ("A row pitch", lda, K, x3)
        assert ldc >= (2 * N if split else N), ("out row pitch", ldc, N, split)
        assert not (split and f32)
        if x3:
            assert K % 32 == 0
        assert act in (0, 1, 2)
    elif name == "b2p_conv3x3":
        _in, ld_in, batch, H, W, Cin, stride, _w, Cout, _out, ldc, _bias, _res, ldr, act, flags, _st = a
        x3 = bool(flags & 8)
        assert stride in (1, 2) and Cin % 32 == 0 and ld_in >= (2 if x3 else 1) * Cin and ldc >= Cout
        if stride == 2:
            assert H % 2 == 0 and W % 2 == 0
    elif name == "b2p_gemm_planes":
        _A, lda, _B, M, N, K, _out, ldc, _bias, _res, ldr, act, flags, lo_a, lo_out, lo_res, _st = a
        x3, split, f32 = bool(flags & 8), bool(flags & 4), bool(flags & 2)
        assert x3 and M > 0 and N > 0 and K % 32 == 0 and (split != f32)
        assert lo_a % 8 == 0 and lo_a >= K and lda >= lo_a + K, ("A planes", lda, lo_a, K)
        if split:
            assert N % 8 == 0 and lo_out % 8 == 0 and lo_out >= N and ldc >= lo_out + N, ("out planes", ldc, lo_out, N)
        assert lo_res % 8 == 0 and (lo_res == 0 or _res)
    elif name == "b2p_conv3x3_planes":
        _in, ld_in, batch, H, W, Cin, stride, _w, Cout, _out, ldc, _bias, _res, ldr, act, flags, lo_a, lo_out, lo_res, _st = a
        x3, split, f32 = bool(flags & 8), bool(flags & 4), bool(flags & 2)
        assert x3 and stride in (1, 2) and Cin % 32 == 0 and (split != f32)
        assert lo_a % 8 == 0 and lo_a >= Cin and ld_in >= lo_a + Cin
        if split:
            assert Cout % 8 == 0 and lo_out >= Cout and ldc >= lo_out + Cout
        if _res:
            assert lo_res > 0 and ldr >= lo_res + Cout
        if stride == 2:
            assert H % 2 == 0 and W % 2 == 0
    elif name in ("b2p_adown_pool_x3", "b2p_maxpool_s1_x3", "b2p_upsample2x_x3"):
        n_lo = 3 if name == "b2p_adown_pool_x3" else 2
        assert all(v > 0 and v % 8 == 0 for v in a[-1 - n_lo:-1]), (name, a[-1 - n_lo:-1])
    elif name == "b2p_cbfuse_x3":
        assert a[-3] > 0 and a[-2] > 0
    elif name == "b2p_layernorm":
        _x, ldx, _g, _b, eps, T, Cc, o16, ld16, o32, ld32, split, _st = a
        assert ldx >= Cc and (o16 is None or ld16 >= (2 if split else 1) * Cc) and (o32 is None or ld32 >= Cc)
    elif name in ("b2p_dwconv_ln", "b2p_channel_attn", "b2p_window_attn", "b2p_mha", "b2p_mha_cached", "b2p_projector_prep"):
        split = a[-2]
        if name in ("b2p_dwconv_ln", "b2p_channel_attn", "b2p_window_attn", "b2p_mha"):
            assert split in (0, 1, 4, 5)  # bit 0: [hi | lo] output, bit 2: florence_simt.cu kernels
        else:
            assert split in (0, 1)


@pytest.fixture()
def rec(monkeypatch):
    r = _Recorder()
    monkeypatch.setattr(_lib, "_lib", r)
    monkeypatch.setattr(ops, "_stream", lambda: C.c_void_p(0))
    monkeypatch.setattr(torch.cuda, "device", lambda *a, **k: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "Stream", _Stream)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: _Stream())
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    return r


@pytest.fixture(scope="module")
def florence():
    return FS.florence_standin(0)


@pytest.mark.parametrize("prec", ["fp16x3", "fp16"])
def test_florence_plan_64(rec, florence, prec):
    from omniparser_b200.florence_engine import FlorencePlan, FlorenceWeights
    w = FlorenceWeights(florence.state_dict(), torch.device("cpu"), FS.GEN, prec)
    p = FlorencePlan(w, 2, 4, FS.PROMPT_IDS, use_graph=False, size=64)
    p.encode()
    n_enc = len(rec.calls)
    p.reset_decode(2)
    p.decode_step()
    n_dec = len(rec.calls) - n_enc
    names = [c[0] for c in rec.calls]
    assert n_enc == 232 and n_dec == 71                                   # launch counts quoted in DESIGN.md / profiles
    assert names.count("b2p_im2col3x3") == 2 and names.count("b2p_conv3x3") == 1   # 4x4 / 2x2 patch-embeds via im2col + GEMM
    x3_flags = {bool(c[1][12] & 8) for c in rec.calls if c[0] == "b2p_gemm"}
    assert x3_flags == {prec == "fp16x3"}
    # every decode step ends with the LM head into the padded logits pitch, the pick and the step counter
    assert names[-3:] == ["b2p_gemm", "b2p_greedy_pick", "b2p_step_advance"]
    lm = rec.calls[-3][1]
    assert lm[4] == 51290 and lm[7] % 8 == 0 and lm[7] >= 51290
    # steps whose token the generation config forces (BOS at length 1, EOS at the last length) run without the LM head
    assert p.step_is_forced(0) and p.step_is_forced(p.T - 1) and not any(p.step_is_forced(t) for t in range(1, p.T - 1))
    n0 = len(rec.calls)
    p.decode_step(forced=True)
    forced = [c[0] for c in rec.calls[n0:]]
    assert len(forced) == n_dec - 1 and forced[-3:] == ["b2p_layernorm", "b2p_greedy_pick", "b2p_step_advance"]


def test_florence_plan_768(rec, florence):
    from omniparser_b200.florence_engine import FlorencePlan, FlorenceWeights
    w = FlorenceWeights(florence.state_dict(), torch.device("cpu"), FS.GEN, "fp16x3")
    p = FlorencePlan(w, 1, 2, FS.PROMPT_IDS, use_graph=False, size=768)
    assert p.n_img == 577 and p.L == 585
    p.encode()
    names = [c[0] for c in rec.calls]
    assert names[0] == "b2p_resize_u8" and names.count("b2p_conv3x3") == 3 and "b2p_im2col3x3" not in names
    n_all = len(names)
    rec.calls.clear()
    p.encode(from_resized=True)          # processor already resized on the host: same plan minus the device resize
    assert len(rec.calls) == n_all - 1 and rec.calls[0][0] == "b2p_im2col_u8"


def test_simt_flags_fixed_and_retired_switches_ignored(rec, florence, monkeypatch):
    """every SIMT entry point of the encode asks for the florence_simt.cu kernel (bit 2) and, in fp16x3 mode, for the
    [hi | lo] output (bit 0); the environment switches of the retired kernel variants no longer change anything"""
    from omniparser_b200.florence_engine import FlorencePlan, FlorenceWeights
    retired = ("B2P_NO_SIMT_V3", "B2P_NO_DWCONV_TILE", "B2P_NO_CHATTN_SMALL", "B2P_GEMM_LN", "B2P_NO_FORCED_SKIP", "B2P_DECODE_PARTS")
    for prec, want in (("fp16x3", 5), ("fp16", 4)):
        w = FlorenceWeights(florence.state_dict(), torch.device("cpu"), FS.GEN, prec)
        for env in ("", "2"):
            for k in retired:
                if env:
                    monkeypatch.setenv(k, env)
                else:
                    monkeypatch.delenv(k, raising=False)
            rec.calls.clear()
            p = FlorencePlan(w, 2, 2, FS.PROMPT_IDS, use_graph=False, size=64)
            p.encode()
            for name in ("b2p_dwconv_ln", "b2p_window_attn", "b2p_channel_attn", "b2p_mha"):
                assert {c[1][-2] for c in rec.calls if c[0] == name} == {want}, (name, prec, env)
            n_enc = len(rec.calls)
            p.reset_decode(2)
            p.decode_step()
            names = [c[0] for c in rec.calls[n_enc:]]
            assert len(names) == 71 and names.count("b2p_layernorm") == 1 + 3 * 6 and p.step_is_forced(0), (prec, env)


# ---- data flow of the pooled caption-encoder plan -------------------------------------------------------------------
_ROLES = {   # op -> (indices of tensor inputs, indices of tensor outputs) in the positional arguments of ops.<op>
    "im2col_u8": ((0,), (9,)), "gemm": ((0, 9), (6,)), "layernorm": ((0,), (5, 6)), "dwconv_ln": ((0,), (7, 10)),
    "window_attn": ((0,), (7,)), "channel_attn": ((0,), (5,)), "mha": ((0, 2, 3), (9,)), "conv3x3": ((0, 5), (2,)),
    "im2col3x3": ((0,), (2,)), "projector_prep": ((0,), (5,)), "encoder_embed": ((0,), (8,)), "resize_u8": ((0,), (7, 8)),
}


def _storage(t):
    if t is None:
        return None
    if isinstance(t, ops.Map):
        t = t.buf
    return t.untyped_storage().data_ptr() if isinstance(t, torch.Tensor) else None


def _trace_ops(monkeypatch):
    """wrap the ops.* front ends of the encode launches: (name, storages read, storages written) per call"""
    trace = []

    def wrap(name, fn):
        ins, outs = _ROLES[name]

        def w(*a, **k):
            full = list(a) + [None] * 12
            if name == "gemm" and "res" in k:
                full[9] = k["res"]
            if name == "conv3x3" and "res" in k:
                full[5] = k["res"]
            if name == "layernorm":
                full[5], full[6] = k.get("out16", full[5]), k.get("out32", full[6])
            trace.append((name, [_storage(full[i]) for i in ins], [_storage(full[i]) for i in outs]))
            return fn(*a, **k)
        return w
    for name in _ROLES:
        monkeypatch.setattr(ops, name, wrap(name, getattr(ops, name)))
    return trace


def _dataflow(trace, monkeypatch, florence, pool):
    """[(op, producers of its inputs)]: for every input tensor of every encode launch, the index of the launch that last wrote
    the buffer it lives in (-1 = never written by the plan: crops, weights)."""
    from omniparser_b200.florence_engine import FlorencePlan, FlorenceWeights
    monkeypatch.setenv("B2P_BUFFER_POOL", "1" if pool else "0")
    del trace[:]
    w = FlorenceWeights(florence.state_dict(), torch.device("cpu"), FS.GEN, "fp16x3")
    p = FlorencePlan(w, 2, 2, FS.PROMPT_IDS, use_graph=False, size=64)
    p.encode()
    last_writer, flow = {}, []
    for i, (name, ins, outs) in enumerate(trace):
        flow.append((name, [last_writer.get(s, -1) if s is not None else None for s in ins]))
        assert not (set(s for s in ins if s is not None) & set(s for s in outs if s is not None)), (i, name, "reads a buffer it writes")
        for s in outs:
            if s is not None:
                last_writer[s] = i
    return flow, len(last_writer), p     # the plan is returned so that its buffers stay alive (storage pointers stay unique)


def test_buffer_pool_preserves_dataflow(rec, florence, monkeypatch):
    """The pooled caption-encoder plan (five buffers per DaViT stage / BART encoder instead of one per intermediate) must have
    the SAME data flow as the one-buffer-per-intermediate plan: every input of every launch is produced by the same launch."""
    trace = _trace_ops(monkeypatch)
    flow_pool, n_pool, keep1 = _dataflow(trace, monkeypatch, florence, True)
    flow_flat, n_flat, keep2 = _dataflow(trace, monkeypatch, florence, False)
    assert len(flow_pool) == len(flow_flat) == 232
    for i, (a, b) in enumerate(zip(flow_pool, flow_flat)):
        assert a == b, (i, a, b)
    assert n_pool < n_flat / 4, (n_pool, n_flat)        # and it really is pooled


def test_yolo_plan(rec):
    from omniparser_b200.yolo_engine import YoloPlan, YoloWeights
    from standin.yolo_weights import yolo_standin
    w = YoloWeights(yolo_standin(0).state_dict(), torch.device("cpu"))
    plan = YoloPlan(w, 2, 384, 640, use_graph=False)
    plan.run()
    names = [c[0] for c in rec.calls]
    assert len(names) == 252 and plan.n_launches == 260                  # 8 b2p_adown_pool calls launch an average and a max kernel each
    assert names.count("b2p_gemm") + names.count("b2p_conv3x3") == 233   # the figure quoted in bench.py / DESIGN.md
    assert all(not (c[1][12] & 8) for c in rec.calls if c[0] == "b2p_gemm")      # detector: plain fp16 operands


def test_yolo_plan_parity_mode(rec):
    """precision="fp16x3": same launch sequence, every conv through the `_planes` entry points with hi/lo maps"""
    from omniparser_b200.yolo_engine import YoloPlan, YoloWeights
    from standin.yolo_weights import yolo_standin
    w = YoloWeights(yolo_standin(0).state_dict(), torch.device("cpu"), precision="fp16x3")
    plan = YoloPlan(w, 1, 384, 640, use_graph=False)
    plan.run()
    names = [c[0] for c in rec.calls]
    assert len(names) == plan.n_launches == 252
    assert names.count("b2p_gemm_planes") + names.count("b2p_conv3x3_planes") == 233
    assert "b2p_gemm" not in names and "b2p_conv3x3" not in names
    assert names.count("b2p_adown_pool_x3") == 8 and names.count("b2p_cbfuse_x3") == 5 and names.count("b2p_maxpool_s1_x3") == 3
    assert rec.calls[0][0] == "b2p_im2col_u8" and rec.calls[0][1][-2] == 1     # stem im2col writes [hi | lo]


class _Graph:
    replays = 0

    def replay(self):
        _Graph.replays += 1


def test_graph_paths_single_decode_chain(rec, florence, monkeypatch):
    """first-use capture, warm(), replay bookkeeping (CUDA graphs replaced by a stub that counts replays)"""
    from omniparser_b200.florence_engine import FlorencePlan, FlorenceWeights
    from omniparser_b200.yolo_engine import YoloPlan, YoloWeights
    from standin.yolo_weights import yolo_standin
    monkeypatch.setattr(torch.cuda, "CUDAGraph", _Graph)
    monkeypatch.setattr(torch.cuda, "graph", lambda *a, **k: contextlib.nullcontext())
    monkeypatch.delenv("B2P_NO_GRAPH", raising=False)
    _Graph.replays = 0
    g0 = ops.GRAPH_LAUNCHES[0]
    w = FlorenceWeights(florence.state_dict(), torch.device("cpu"), FS.GEN, "fp16x3")
    p = FlorencePlan(w, 2, 3, FS.PROMPT_IDS, use_graph=True, size=64)
    assert p.use_graph and not p.warmed
    p.warm()                                            # encode: eager + capture + replay; decode: eager + capture, then one replay
    assert p.warmed and p.g_enc is not None and p.g_dec is not None and p.g_dec_forced is not None
    n_eager = len(rec.calls)
    assert n_eager == 2 * (232 + 71 + 70)               # every op ran once eagerly and once inside the (stubbed) capture; the
                                                        # decode step exists with and without the LM head (forced tokens)
    p.encode(); p.reset_decode(2); p.decode_step(); p.decode_step()
    assert _Graph.replays == 2 + 3 and ops.GRAPH_LAUNCHES[0] - g0 == 2 * 232 + 3 * 71      # kernels, not calls
    assert sum(1 for c in rec.calls[n_eager:] if c[0].startswith("b2p_")) == 0     # steady state: graph replays only
    yw = YoloWeights(yolo_standin(0).state_dict(), torch.device("cpu"))
    yp = YoloPlan(yw, 1, 384, 640, use_graph=True)
    g1 = ops.GRAPH_LAUNCHES[0]
    yp.run(); yp.run()
    assert ops.GRAPH_LAUNCHES[0] - g1 == 2 * 260
