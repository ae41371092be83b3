#!/usr/bin/env python
"""Benchmark of the parse hot path (BASELINE.json metric: screenshots/sec on 1920x1080 synthetic screenshots with
~60 boxes; workload = configs[2]: detect + NMS + crop + Florence-2 caption, batch of 8 screenshots per GPU).

  python bench.py --gpus N --steps K --warmup W            # this repo (one process per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores (oracle port)

A "step" = one pass of the hot path over one batch of B synthetic screenshots per GPU: LANCZOS letterbox ->
YOLOv9-E -> decode/NMS -> overlap filter (device) -> crop+resize -> Florence-2 greedy caption, results gathered to
rank 0 with one NCCL gather.  `value` times it with the u8 screenshots already resident in HBM, `e2e` through the
public API with host buffers (H2D of the screenshots and D2H of boxes/ids inside the timed region).
Prints ONE JSON line on rank 0.

  python bench.py ... --dump-outputs DIR    # also write what the last timed step returned as DIR/*.npy (see dump_outputs)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

W, H = 1920, 1080
N_SETS = 4            # distinct input batches rotated between steps (4 x 8 x 6.2 MB = 199 MB > 126 MB L2)


_T0 = time.perf_counter()


def log(msg):
    if os.environ.get("B2P_BENCH_VERBOSE", "1") != "0":
        print(f"[bench {time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def host_threads() -> int:
    """Usable host cores: torch's default, capped by the affinity mask and the cgroup CPU quota (oversubscribing
    OpenMP threads on a quota-limited container stalls for minutes)."""
    # NOT torch.get_num_threads(): torchrun exports OMP_NUM_THREADS=1, which would make a multi-rank launch report a
    # one-thread reference (round-1 finding); the machine's cores, the affinity mask and the cgroup quota are what count
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, n)


def _dist():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons WHILE the timed region runs (B200_PROFILING.md recipe): NVML in-process every 20 ms
    (same counters nvidia-smi prints), falling back to the nvidia-smi command line if NVML cannot be loaded."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()   # samples: (sm_mhz, max_mhz, reason names)
        self.source, self.h, self.nv = "nvidia-smi", None, None
        try:
            import pynvml as nv
            nv.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.nv, self.source = nv, "nvml"
            self.sample()
            self.samples.clear()
        except Exception:
            self.nv = self.h = None
            self.source = "nvidia-smi"

    def sample(self):
        if self.nv is not None:
            nv = self.nv
            sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            try:
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.samples.append((int(sm), int(mx), [n for n, b in self.BITS if mask & b]))
            return
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        if out:
            f = [x.strip() for x in out.splitlines()[0].split(",")]
            names = [n for n, _ in self.BITS]
            self.samples.append((int(f[0]), int(f[1]), [names[i] for i in range(4) if f[2 + i].lower().startswith("active")]))

    def run(self):
        while not self.stop_flag.is_set():
            try:
                self.sample()
            except Exception:
                pass
            self.stop_flag.wait(0.02 if self.nv is not None else 0.2)

    def finish(self):
        self.stop_flag.set()
        self.join(timeout=15)
        return self.summary()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0, "source": self.source}
        sm = sorted(s[0] for s in self.samples)
        reasons = sorted({r for s in self.samples for r in s[2]})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0][1], "reasons": reasons, "samples": len(self.samples),
                "source": self.source}


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.is_file():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained") or d.get("bf16_tflops"), d.get("hbm_gbs"), "measured"
    return 1400.0, 6650.0, "fallback"   # B200_PROFILING.md fallback (sustained 1.4 PFLOP/s, 6.65 TB/s)


def _inputs(rank: int, B: int):
    from omniparser_b200 import synth
    sets = []
    for s in range(N_SETS):
        seeds = [rank * 1000 + s * B + i for i in range(B)]
        sets.append(([synth.screenshot(sd) for sd in seeds], [synth.ocr_boxes(sd) for sd in seeds]))
    return sets


# ------------------------------------------------------------------------------------------------ reference arm
REF_SAMPLE = 4        # screenshots of the step's batch the reference arm parses per step (bounded sample)


def run_reference(args):
    """The reference algorithm (oracle port, see oracle/pipeline_cpu.py) on ALL the host cores; rank 0 only.  Same
    workload, config, seeds and thresholds as the B200 arm: step j parses the first REF_SAMPLE screenshots of the batch
    rank 0 of the B200 arm parses at step j (a bounded sample of the step: the whole --steps/--warmup run must end within
    minutes at ~1 s per screenshot)."""
    rank, world, _ = _dist()
    if rank != 0:
        return
    from omniparser_b200 import synth
    from oracle.pipeline_cpu import OraclePipeline
    torch.set_num_threads(host_threads())
    pipe = OraclePipeline()
    B = args.batch
    k = min(REF_SAMPLE, B)
    times, nb, nbox = [], [], []
    for j in range(args.warmup + args.steps):
        seeds = [(j % N_SETS) * B + i for i in range(k)]      # = _inputs(rank 0)[j % N_SETS][:k]
        data = [(synth.screenshot(sd), synth.ocr_boxes(sd)) for sd in seeds]
        t0 = time.perf_counter()
        for img, (texts, boxes) in data:
            tm = {}
            pipe.parse(img, texts, boxes, BOX_TRESHOLD=args.box_threshold, iou_threshold=0.7, max_new_tokens=args.max_new_tokens,
                       caption_768=args.caption_768, timings=tm)
            if j >= args.warmup:
                nb.append(tm["n_crops"])
        dt = time.perf_counter() - t0
        if j >= args.warmup:
            times.append(dt)
    total = sum(times)
    val = k * len(times) / total
    sample = (f"{k} of the {B * args.gpus} screenshots of each step (same seeds as the B200 arm's rank 0), {len(times)} steps, "
              f"{np.mean(nb):.1f} crops per screenshot, caption mode "
              f"{'768 (reference CPU branch)' if args.caption_768 else '64 (mode-matched with the GPU path)'}, fp32, {torch.get_num_threads()} threads")
    line = {"impl": "reference", "metric": "screenshots/sec", "value": val, "unit": "screenshots/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config(args, B),
            "cpu_baseline": {"value": val, "unit": "screenshots/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "screenshots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "crops_per_screenshot": float(np.mean(nb))}
    print(json.dumps(line), flush=True)


def _config(args, per_gpu_batch):
    return {"workload": "configs[2]: detect+NMS+crop+Florence-2 caption, synthetic 1920x1080 screenshots, ~60 boxes each",
            "screenshots_per_gpu_per_step": per_gpu_batch, "global_batch": per_gpu_batch * args.gpus,
            "detector_input": "letterbox 640x640 (API default, ref:util/utils.py:417 scale_img=False)",
            "caption_mode": "64x64 crops, 5 image tokens (reference CUDA branch, ref:util/utils.py:121)",
            "decode_tokens": args.max_new_tokens, "box_threshold": args.box_threshold, "weights": "seeded stand-ins (no checkpoints offline)",
            "caption_precision": args.precision, "detector_precision": "fp16 operands, fp32 accumulate",
            "l2": f"inputs rotate over {N_SETS} distinct batches ({N_SETS * per_gpu_batch * W * H * 3 / 1e6:.0f} MB/GPU) > 126 MB L2",
            "parallelism": f"dp{args.gpus} (screenshots sharded, one NCCL gather of results per step, issued off the parse loop)",
            "schedule": "one batch at a time" if getattr(args, "no_pipeline", False) else
                        f"pipeline across steps: detect(i+1) on stream A | host list logic(i) | {args.caption_lanes} caption lanes (batches i-1.. on own streams/plans), caption group {args.caption_group}; fill and drain are inside the timed region"}


# ------------------------------------------------------------------------------------------------ this repo
SOURCES = ("box_ocr_content_ocr", "box_yolo_content_ocr", "box_yolo_content_yolo")


def output_arrays(out):
    """One step's results, ``[(elements, caption_ids)]`` per screenshot, as float64 arrays:
    ``elements`` [N, 8] = screenshot, x0, y0, x1, y1 (ratios), interactivity, source (index into SOURCES), row of its
    caption in ``caption_ids`` (-1: no caption); ``caption_ids`` [M, T] = greedy token ids, short rows padded with -1."""
    elems, caps = [], []
    for i, (el, ids) in enumerate(out):
        first = len(caps)
        caps.extend(ids.tolist())
        row = first
        for e in el:
            src = SOURCES.index(e["source"])
            elems.append([i, *e["bbox"], float(e["interactivity"]), src, row if src == 2 else -1])
            row += src == 2
        assert row == len(caps), "captioned elements and caption rows disagree"
    width = max((len(r) for r in caps), default=0)
    ids = np.full((len(caps), width), -1, np.float64)
    for r, c in enumerate(caps):
        ids[r, :len(c)] = c
    return {"elements": np.asarray(elems, np.float64).reshape(-1, 8), "caption_ids": ids}


def dump_outputs(arrays, out_dir):
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a)
    log(f"outputs of the last timed step written to {d}: " + ", ".join(f"{k} {tuple(a.shape)}" for k, a in arrays.items()))


def run_b200(args):
    rank, world, local = _dist()
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as ge
    from omniparser_b200 import _lib, ops, shard
    from omniparser_b200.utils import ParseTimings, parse_screenshots
    _lib.lib()   # raises if the CUDA extension is missing: no fallback
    torch.set_num_threads(max(1, host_threads() // max(1, world)))   # CPU-side model generation: stay inside the core quota
    log("building stand-in models")
    model, cmp_ = ge.standin_models(dev, args.precision)
    log("models ready; generating inputs")
    B = args.batch
    sets = _inputs(rank, B)
    pipe = shard.GatherPipe(rank, world, dev, B, args.max_new_tokens, keep=False)   # one NCCL gather per step, on its own thread + stream
    stats = {"boxes": 0, "crops": 0, "n": 0}
    last = [None]   # the results of the most recent step (--dump-outputs)

    def step(i, resident):
        imgs, ocr = sets[i % N_SETS]
        tm = ParseTimings()
        if resident:
            io_ = model._get_io(B, H, W, 640, 300)
            io_["src"].copy_(dsets[i % N_SETS], non_blocking=True)      # device-to-device: input already in HBM
        out = parse_screenshots(imgs, model, cmp_, ocr, BOX_TRESHOLD=args.box_threshold, iou_threshold=0.7,
                                max_new_tokens=args.max_new_tokens, timings=tm, _skip_h2d=resident)
        last[0] = out
        stats["boxes"] += tm["n_boxes"]; stats["crops"] += tm["n_crops"]; stats["n"] += B
        pipe.submit(out)   # one gather of fixed-size padded records per step (SURVEY.md §8e); no-op at world 1
        return tm

    dsets = [torch.from_numpy(np.stack(s[0])).to(dev) for s in sets]
    hsets = [torch.from_numpy(np.stack(s[0])).pin_memory() for s in sets]   # the e2e leg's host-side inputs (pinned)
    log("inputs ready; warm-up")
    for i in range(args.warmup):
        step(i, True)
        step(i, False)
        log(f"warm-up step {i} done")
    torch.cuda.synchronize()

    from omniparser_b200.utils import PipelinedParser
    pp = PipelinedParser(model, cmp_, BOX_TRESHOLD=args.box_threshold, iou_threshold=0.7, max_new_tokens=args.max_new_tokens,
                         caption_lanes=args.caption_lanes, caption_group=args.caption_group)

    def run_steps(n_steps, resident):
        if args.no_pipeline:
            return [step(i, resident) for i in range(n_steps)]
        # e2e leg: each step's screenshots start in page-locked host memory and are DMA'd to the GPU inside the timed region
        batches = ((hsets[i % N_SETS] if not resident else sets[i % N_SETS][0], sets[i % N_SETS][1]) for i in range(n_steps))
        res = (dsets[i % N_SETS] for i in range(n_steps)) if resident else None
        tm0 = dict(pp.timings)
        for out in pp.run(batches, res):
            last[0] = out
            stats["n"] += B
            pipe.submit(out)
        stats["boxes"] += pp.timings["n_boxes"] - tm0["n_boxes"]
        stats["crops"] += pp.timings["n_crops"] - tm0["n_crops"]
        d = {k: (pp.timings[k] - tm0[k]) / max(n_steps, 1) for k in ("detect_wait_s", "glue_s", "caption_s")}
        return [dict(detect_s=d["detect_wait_s"], glue_s=d["glue_s"], caption_s=d["caption_s"])]

    def run_steps_pageable(n_steps):
        """the path an unprepared caller hits: plain (pageable) numpy screenshots; the pipeline stages them through its
        own page-locked slot buffer"""
        for out in pp.run(((sets[i % N_SETS][0], sets[i % N_SETS][1]) for i in range(n_steps)), None):
            stats["n"] += B
            pipe.submit(out)
        return []

    def timed(mode):
        resident = mode == "resident"
        sampler = ClockSampler(local)
        pipe.drain()     # gathers of the warm-up steps are done before the barrier (collectives stay in one order on every rank)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0, g0 = _lib.launch_count(), ops.GRAPH_LAUNCHES[0]
        stats.update(boxes=0, crops=0, n=0)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        tms = run_steps(args.steps, resident) if mode != "pageable" else run_steps_pageable(args.steps)
        pipe.drain()            # every step's gather has completed (inside the timed region)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        wall = time.perf_counter() - t0
        clk = sampler.finish()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        launches = (_lib.launch_count() - l0) + (ops.GRAPH_LAUNCHES[0] - g0)
        return float(t.item()), wall, launches, clk, tms, dict(stats)

    if not args.no_pipeline:
        # every (crop-count bucket, lane) plan is built before anything is timed, whatever --steps / --warmup are
        counts = []
        for i in range(N_SETS):
            counts.append(step(i, True)["n_crops"])
        G = max(1, args.caption_group)   # grouped captioning: every run of up to G consecutive batches can form a group
        pp.prewarm(sorted({sum(counts[(s0 + j) % N_SETS] for j in range(r)) for s0 in range(N_SETS) for r in range(1, G + 1)}))
        run_steps(max(args.warmup, N_SETS, args.caption_lanes + 4, args.caption_lanes * G + G + 2), True)   # warm the pipelined path (every io slot, stream-local scratch)
        run_steps(2, False)
        torch.cuda.synchronize()
        log("pipelined warm-up done")
    ms_res, _, launches, clocks, tms, st = timed("resident")
    log(f"resident leg: {ms_res / args.steps:.1f} ms/step")
    outputs = output_arrays(last[0]) if args.dump_outputs else None   # the headline leg's last step, before later legs run
    ms_e2e, _, _, _, tms2, _ = timed("pinned")
    log(f"e2e leg: {ms_e2e / args.steps:.1f} ms/step")
    ms_pg = None
    if not args.no_pipeline:
        ms_pg, _, _, _, _, _ = timed("pageable")
        log(f"e2e leg, pageable inputs: {ms_pg / args.steps:.1f} ms/step")
    value = world * B * args.steps / (ms_res / 1e3)
    e2e = world * B * args.steps / (ms_e2e / 1e3)

    # roofline of the dominant kernel: gemm_tcgen05_kernel inside the YOLOv9-E forward (233 of its 252 launches,
    # ~95 % of its device time, profiles/); algorithmic FLOPs of the forward / CUDA-event time of the graph replay.
    plan = model._get_io(B, H, W, 640, 300)["plan"]
    for _ in range(3):
        plan.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    reps = 10
    for _ in range(reps):
        plan.run()
    e1.record()
    torch.cuda.synchronize()
    fwd_ms = e0.elapsed_time(e1) / reps
    peak_tf, hbm, how = _peaks()
    achieved = plan.flops / (fwd_ms * 1e-3) / 1e12
    traffic = None
    # measured under ncu for this exact forward (batch 8: dram__bytes_read/write.sum of every launch, caches flushed per
    # kernel), committed per round; not re-measured per run
    for tp, key in ((ROOT / "profiles" / "r2_stage_traffic.json", "detect"), (ROOT / "profiles" / "r1_yolo_b8_traffic.json", None)):
        if tp.is_file() and B == 8 and traffic is None:
            tj = json.loads(tp.read_text())
            tj = tj.get(key, {}) if key else tj
            if "dram_bytes_read" in tj:
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]

    # p50 latency of one screenshot through the public batched entry point (host buffers)
    lat = []
    for i in range(7):
        imgs, ocr = sets[i % N_SETS]
        t0 = time.perf_counter()
        parse_screenshots(imgs[:1], model, cmp_, ocr[:1], BOX_TRESHOLD=args.box_threshold, iou_threshold=0.7, max_new_tokens=args.max_new_tokens)
        torch.cuda.synchronize()
        lat.append(1e3 * (time.perf_counter() - t0))
    lat = sorted(lat[2:])
    log("latency leg done")

    # outside the timed region: the pipelined schedule must return exactly what the one-batch-at-a-time path returns
    verify = None
    if not args.no_pipeline:
        seq_out = [parse_screenshots(sets[i][0], model, cmp_, sets[i][1], BOX_TRESHOLD=args.box_threshold, iou_threshold=0.7,
                                     max_new_tokens=args.max_new_tokens) for i in range(N_SETS)]
        bad = rows = 0
        for rep in range(2):
            for i, out in enumerate(pp.run((sets[j] for j in range(N_SETS)), None)):
                for (_, gi), (_, ri) in zip(out, seq_out[i]):
                    rows += ri.shape[0]
                    bad += ri.shape[0] if gi.shape != ri.shape else int((gi != ri).any(1).sum())
        verify = {"pipelined_vs_sequential_caption_rows": rows, "mismatched_rows": bad}
        log(f"verify: {verify}")

    # per-stage tensor-core figures of the caption path (SURVEY.md §8d: F1/F3 encode, F4 decode step), CUDA events over
    # graph replays of the lane-0 plan; informative only -- a failure here never costs the bench line
    caption_stages = None
    try:
        with torch.inference_mode():
            n_c = counts[0] if not args.no_pipeline else max(1, st["crops"] // max(args.steps, 1))   # a bucket that exists
            cplan = cmp_["model"].plan_for(n_c, args.max_new_tokens, pp.prompt)
            if cplan.use_graph and cplan.warmed or cplan.g_enc is not None:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
                cplan.encode(); torch.cuda.synchronize()
                ev[0].record()
                for _ in range(5):
                    cplan.encode()
                ev[1].record()
                cplan.reset_decode(n_c)
                cplan.decode_step(); torch.cuda.synchronize()
                nd = max(1, args.max_new_tokens - 1)
                ev[2].record()
                for _ in range(nd):
                    cplan.decode_step()
                ev[3].record()
                cplan.join(); torch.cuda.synchronize()
                enc_ms, dec_ms = ev[0].elapsed_time(ev[1]) / 5, ev[2].elapsed_time(ev[3]) / nd
                xk = 3 if cplan.x3 else 1
                caption_stages = {
                    "rows": cplan.K, "precision": "fp16x3" if cplan.x3 else "fp16",
                    "encode": {"ms": enc_ms, "logical_tflops": cplan.flops_enc / enc_ms / 1e9, "executed_tflops": xk * cplan.flops_enc / enc_ms / 1e9,
                               "executed_frac_of_peak": xk * cplan.flops_enc / enc_ms / 1e9 / peak_tf},
                    "decode_step": {"ms": dec_ms, "logical_tflops": cplan.flops_dec / dec_ms / 1e9, "executed_tflops": xk * cplan.flops_dec / dec_ms / 1e9,
                                    "executed_frac_of_peak": xk * cplan.flops_dec / dec_ms / 1e9 / peak_tf,
                                    "note": "~70 launches per step at M = rows: dependency-chain bound (~11 us per launch whatever the tiling), see profiles/r2_notes.md"}}
                log(f"caption stages: encode {enc_ms:.2f} ms, decode step {dec_ms:.3f} ms")
                log(f"device memory: peak allocated {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB, reserved {torch.cuda.memory_reserved() / 2**30:.1f} GiB")
    except Exception as exc:   # noqa: BLE001
        caption_stages = {"error": repr(exc)[:200]}

    # per-stage roofline list (detect / caption encode / decode step): achieved = algorithmic FLOPs (logical: what the
    # reference's fp32 graph computes; the fp16x3 stages execute 3x that on the tensor pipe) / CUDA-event time in THIS run;
    # traffic = DRAM bytes of the stage from the committed ncu launch list of the same kernels (profiles/, per stage).
    stage_traffic = {}
    tpf = ROOT / "profiles" / "r2_stage_traffic.json"
    if tpf.is_file() and B == 8:
        stage_traffic = json.loads(tpf.read_text())
    roofline_stages = [{"stage": "detect: YOLOv9-E forward (gemm_tcgen05_kernel x233 + 27 HBM kernels)", "bound": "tensor", "ms": fwd_ms,
                        "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                        "traffic": (stage_traffic.get("detect") or {}).get("dram_bytes", traffic)}]
    if caption_stages and "encode" in caption_stages:
        for key, label in (("encode", "caption encode: DaViT + projector + BART encoder + cross-KV"), ("decode_step", "caption decode step (6 layers + LM head + pick)")):
            cs = caption_stages[key]
            roofline_stages.append({"stage": label, "bound": "tensor", "ms": cs["ms"], "achieved": cs["logical_tflops"], "executed": cs["executed_tflops"],
                                    "peak": peak_tf, "unit": "TFLOP/s", "frac": cs["logical_tflops"] / peak_tf, "frac_executed": cs["executed_frac_of_peak"],
                                    "traffic": (stage_traffic.get(key) or {}).get("dram_bytes")})

    # the reference's CPU-branch caption semantics (768x768 crops, ref:util/utils.py:123) on the GPU: extra figure, 2 screenshots
    cap768 = None
    if args.with_768:
        try:
            imgs, ocr = sets[0]
            parse_screenshots(imgs[:2], model, cmp_, ocr[:2], BOX_TRESHOLD=args.box_threshold, iou_threshold=0.7,
                              max_new_tokens=args.max_new_tokens, caption_size=768)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out768 = parse_screenshots(imgs[:2], model, cmp_, ocr[:2], BOX_TRESHOLD=args.box_threshold, iou_threshold=0.7,
                                       max_new_tokens=args.max_new_tokens, caption_size=768)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            cap768 = {"screenshots_per_s": 2 / dt, "crops": int(sum(o[1].shape[0] for o in out768)), "note": "768x768 caption mode (the reference's CPU branch), batch of 2 screenshots, one batch at a time, host buffers"}
            log(f"768-mode: {2 / dt:.2f} screenshots/s")
        except Exception as exc:   # noqa: BLE001
            cap768 = {"error": repr(exc)[:200]}

    if rank == 0:
        line = {"metric": "screenshots/sec", "value": value, "unit": "screenshots/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": _config(args, B),
                "e2e": {"value": e2e, "unit": "screenshots/s", "h2d_bytes_per_step": B * H * W * 3 + st["crops"] // max(args.steps, 1) * 20,
                        "d2h_bytes_per_step": B * (4 + 300 * 16) + st["crops"] // max(args.steps, 1) * (args.max_new_tokens + 1) * 8,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": launches, "clocks": clocks,
                "roofline": {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (YOLOv9-E forward, batch %d: 233 GEMM/conv launches + 27 im2col/pooling/upsample/CBFuse launches)" % B,
                             "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic,
                             "traffic_note": "DRAM bytes per forward from the committed ncu launch list (caches flushed per kernel), not from this run",
                             "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({how})", "forward_ms": fwd_ms,
                             "algorithmic_gflop_per_forward": plan.flops / 1e9},
                "roofline_stages": roofline_stages,
                "e2e_pageable": None if ms_pg is None else {"value": world * B * args.steps / (ms_pg / 1e3), "unit": "screenshots/s", "ms_per_step": ms_pg / args.steps,
                                                            "note": "same as e2e but the screenshots are plain pageable numpy arrays (staged through the pipeline's pinned slot)"},
                "caption_768": cap768,
                "verify": verify, "caption_stages": caption_stages, "p50_latency_ms_batch1": lat[len(lat) // 2],
                "stage_ms_per_step": {k: 1e3 * float(np.mean([t[k] for t in tms2])) for k in ("detect_s", "glue_s", "caption_s")},
                "boxes_per_screenshot": st["boxes"] / max(st["n"], 1), "crops_per_screenshot": st["crops"] / max(st["n"], 1)}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args)
        print(json.dumps(line), flush=True)
        if outputs is not None:
            dump_outputs(outputs, args.dump_outputs)
    pipe.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline(args):
    """Oracle port on the host cores, bounded sample (2 screenshots after 1 warm-up, ~10-20 s)."""
    log("cpu baseline (oracle port on the host cores)")
    from omniparser_b200 import synth
    from oracle.pipeline_cpu import OraclePipeline
    torch.set_num_threads(host_threads())
    log(f"host threads: {torch.get_num_threads()} (os.cpu_count {os.cpu_count()})")
    pipe = OraclePipeline()
    ts, crops = [], []
    for i in range(3):
        tm = {}
        t0 = time.perf_counter()
        pipe.parse(synth.screenshot(i), *synth.ocr_boxes(i), BOX_TRESHOLD=args.box_threshold, iou_threshold=0.7,
                   max_new_tokens=args.max_new_tokens, timings=tm)
        if i:
            ts.append(time.perf_counter() - t0)
            crops.append(tm["n_crops"])
    return {"value": len(ts) / sum(ts), "unit": "screenshots/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{len(ts)} screenshots after 1 warm-up, {np.mean(crops):.0f} crops each, 64x64 caption mode (mode-matched), fp32"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--caption-lanes", type=int, default=2, help="caption (groups of) batches in flight, own stream + plan each")
    ap.add_argument("--caption-group", type=int, default=2,
                    help="caption the crops of this many consecutive steps in one Florence-2 pass (PipelinedParser caption_group); measured on one "
                         "B200 box, round 2: lanes 3 / group 1 16.2 ms per step, lanes 4 / group 1 15.1, lanes 2 / group 2 14.6, lanes 3 / group 2 14.5")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="screenshots per GPU per step")
    ap.add_argument("--max-new-tokens", type=int, default=8)
    ap.add_argument("--box-threshold", type=float, default=0.05)
    ap.add_argument("--precision", default="fp16x3", choices=["fp16x3", "fp16"])
    ap.add_argument("--caption-768", action="store_true", help="reference arm only: the reference's CPU branch (768x768 crops)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--with-768", action="store_true", help="B200 arm: also time the 768x768 caption mode (extra key caption_768)")
    ap.add_argument("--no-pipeline", action="store_true", help="one batch at a time (no detect/caption overlap across steps)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="B200 arm: write what the last timed step of the resident leg returned (rank 0's screenshots) as "
                         "DIR/elements.npy and DIR/caption_ids.npy, float64; same arguments, same inputs")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
