"""Shared comparison helpers of the GPU parity tests.

Two near-fp32 evaluations of the detector (the reference's fp32 CPU forward, the fp16x3 tensor-core forward) agree to ~1e-4
on the scores.  Everything downstream of the scores is exact, so the only way the two box LISTS can differ is a "tie-class
event": two boxes whose reference scores are closer than that noise swap places in the score-ordered NMS output (SURVEY.md
8d; DESIGN.md 2).  These helpers match the lists one-to-one, COUNT such events, check each is a genuine near-tie, and bound
them -- reported, never hidden.

The fp32 CPU forward itself sums in an order that depends on the host's instruction set and thread count: on another host
(or with another thread count) the oracle's detector output moves by up to ~4e-4 canvas pixels and ~1e-5 in score from the
bits a golden recorded, with the same boxes in the same order.  :func:`match_cpu_detector` compares it with that margin."""
import torch

CPU_PX_TOL, CPU_SCORE_TOL = 2e-3, 5e-5   # canvas pixels, score: ~5x the spread measured across hosts and thread counts


def px_tolerance(w, h, base=0.05):
    """The detector works on a 640-pixel canvas: a coordinate error of `base` canvas pixels is base * max(w, h) / 640 image pixels."""
    return base * max(1.0, max(w, h) / 640.0)


def match_scored_boxes(gb, gs, rb, rs, px_tol, score_tol=1e-3, max_events=4):
    """ref box i <-> got box j, one to one: same position unless a near-tie swapped them.  Returns the events [(i, j)]."""
    gb, gs, rb, rs = (torch.as_tensor(t, dtype=torch.float32) for t in (gb, gs, rb, rs))
    assert len(gb) == len(rb), (len(gb), len(rb))
    used, events = set(), []
    for i in range(len(rb)):
        d = (gb - rb[i]).abs().amax(1)
        order = [i] + [j for j in torch.argsort(d).tolist() if j != i]
        j = next((j for j in order if j not in used and d[j] <= px_tol and abs(float(gs[j] - rs[i])) <= score_tol), None)
        assert j is not None, f"reference box {i} {rb[i].tolist()} (score {float(rs[i]):.6f}) has no counterpart"
        used.add(j)
        if j != i:
            assert abs(float(rs[i] - rs[j])) <= score_tol, f"boxes {i} and {j} changed places but their reference scores are not tied"
            events.append((i, j))
    assert len(events) <= max_events, f"{len(events)} tie-class events: {events}"
    return events


def match_cpu_detector(kb, ks, gold_xyxy, gold_conf, w, h):
    """The oracle's fp32 CPU detector output vs a golden's boxes and scores: same count, same order up to genuine near-ties
    (at most two), every box and score within the host-to-host noise of the fp32 CPU forward."""
    gb = torch.tensor(gold_xyxy, dtype=torch.float32).reshape(-1, 4)
    return match_scored_boxes(kb, ks, gb, torch.tensor(gold_conf, dtype=torch.float32), px_tolerance(w, h, CPU_PX_TOL),
                              score_tol=CPU_SCORE_TOL, max_events=2)


def golden_scores(g):
    """golden dict with det_xyxy / det_conf -> {ratio bbox tuple: detector score} (the element boxes are det_xyxy / whwh in fp32)."""
    if "det_xyxy" not in g or not g["det_xyxy"]:
        return {}
    w, h = g["case"]["size"]
    ratio = (torch.tensor(g["det_xyxy"], dtype=torch.float32).reshape(-1, 4) / torch.Tensor([w, h, w, h])).tolist()
    return {tuple(r): float(c) for r, c in zip(ratio, g["det_conf"])}


def match_elements(got, ref, size, px_tol, max_shift=3, scores=None, score_tol=1e-3):
    """parsed_content_list vs the golden: same multiset of (type, source, interactivity, box within px_tol); positions may
    differ only by near-tie swaps (|i - j| <= max_shift).  With ``scores`` (golden_scores) every displaced element must be a
    genuine near-tie: its reference score within score_tol of the element whose place it took.  Returns (pairs [(ref index, got
    index)], order events)."""
    w, h = size
    assert len(got) == len(ref), (len(got), len(ref))
    used, pairs, events = set(), [], 0
    for i, b in enumerate(ref):
        cand = [i] + [j for j in range(max(0, i - max_shift), min(len(got), i + max_shift + 1)) if j != i]
        hit = None
        for j in cand:
            a = got[j]
            if j in used or (a["type"], a["source"], a["interactivity"]) != (b["type"], b["source"], b["interactivity"]):
                continue
            if max(abs(x - y) * s for x, y, s in zip(a["bbox"], b["bbox"], (w, h, w, h))) <= px_tol:
                hit = j
                break
        assert hit is not None, f"golden element {i} {b} has no counterpart near its position"
        used.add(hit)
        pairs.append((i, hit))
        if hit != i:
            events += 1
            if scores:
                si, sj = scores.get(tuple(ref[i]["bbox"])), scores.get(tuple(ref[hit]["bbox"]))
                assert si is not None and sj is not None and abs(si - sj) <= score_tol, (
                    f"elements {i} and {hit} changed places but their reference scores ({si}, {sj}) are not tied")
    assert events <= max(2, len(ref) // (10 if scores else 20)), f"{events} order events in {len(ref)} elements"
    return pairs, events
