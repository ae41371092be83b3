"""CPU: host list logic (overlap filter, element construction) of the product vs what the unmodified reference functions
returned on the same cases (tests/golden/reference_remove_overlap_new.json, written by oracle/make_golden.py) and vs the
oracle's independent restatement."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from omniparser_b200 import host_glue
from oracle import pipeline_cpu

W, H = 1920, 1080
THRESHOLDS = (0.7, 0.9)
GOLD = Path(__file__).resolve().parent / "golden"


def case_key(kind, seed, thr):
    return f"{kind}{seed}_iou{thr}"


def decode_elements(enc, icons, oboxes, texts):
    """The reference's element list from its golden encoding: ["o", k] is the OCR element of input box k, ["i", j, content]
    the icon element of input box j (the encoding is checked to round-trip when the golden is written)."""
    out = []
    for e in enc:
        if e[0] == "o":
            out.append({'type': 'text', 'bbox': oboxes[e[1]], 'interactivity': False, 'content': texts[e[1]], 'source': 'box_ocr_content_ocr'})
        else:
            out.append({'type': 'icon', 'bbox': icons[e[1]], 'interactivity': True, 'content': e[2],
                        'source': 'box_yolo_content_ocr' if e[2] is not None else 'box_yolo_content_yolo'})
    return out


def reference_elements(kind, seed, thr, icons, oboxes, texts):
    gold = json.loads((GOLD / "reference_remove_overlap_new.json").read_text())
    return decode_elements(gold[case_key(kind, seed, thr)], icons, oboxes, texts)


def _case(seed, n_icon=70, n_ocr=20):
    n_icon = n_icon + 30 * (seed % 3)
    rng = np.random.default_rng(seed)
    xy = rng.uniform(0, 0.9, size=(n_icon, 2))
    wh = rng.uniform(0.0, 0.08, size=(n_icon, 2))
    icons = torch.tensor(np.concatenate([xy, xy + wh], 1), dtype=torch.float32)
    icons[1] = icons[0]                       # duplicate
    icons[2, 2:] = icons[2, :2]               # zero area
    icons[3, :2] = icons[4, :2] + 0.001       # nested
    icons[3, 2:] = icons[4, 2:] - 0.001
    ob = []
    for i in range(n_ocr):
        x, y = int(rng.integers(0, W - 70)), int(rng.integers(0, H - 30))
        ob.append([x, y, x + 60, y + 20])
    # an OCR box inside an icon and an icon inside an OCR box
    ix = (icons[5] * torch.tensor([W, H, W, H])).tolist()
    ob[0] = [int(ix[0]) + 1, int(ix[1]) + 1, max(int(ix[0]) + 3, int(ix[2]) - 1), max(int(ix[1]) + 3, int(ix[3]) - 1)]
    ox = ob[1]
    icons[6] = torch.tensor([(ox[0] + 5) / W, (ox[1] + 4) / H, (ox[0] + 25) / W, (ox[1] + 14) / H])
    texts = [f"t{i}" for i in range(n_ocr)]
    return icons, ob, texts


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("thr", [0.7, 0.9])
def test_build_elements_matches_oracle_restatement(seed, thr):
    icons, ob, texts = _case(seed)
    whwh = torch.Tensor([W, H, W, H])
    oratio = (torch.tensor(ob) / whwh).tolist()
    a, start = host_glue.build_elements(icons.tolist(), oratio, texts, W, H, thr)
    slow, _ = host_glue.build_elements(icons.tolist(), oratio, texts, W, H, thr, fast=False)
    b = pipeline_cpu.build_elements(icons.tolist(), oratio, texts, W, H, thr)
    assert a == b and a == slow
    assert start == next((i for i, e in enumerate(a) if e["content"] is None), -1)


@pytest.mark.parametrize("seed", range(6))
def test_build_elements_matches_reference(seed):
    icons, ob, texts = _case(seed)
    whwh = torch.Tensor([W, H, W, H])
    for thr in THRESHOLDS:
        # the reference ran ref:util/utils.py:437-451 verbatim on these inputs
        ocr_bbox = (torch.tensor(ob) / whwh).tolist()
        ref = reference_elements("case", seed, thr, icons.tolist(), ocr_bbox, texts)
        got, _ = host_glue.build_elements(icons.tolist(), ocr_bbox, texts, W, H, thr)
        assert got == ref


def _dense_case(seed):
    """Adversarial for the OCR-containment walk (ref:util/utils.py:283-305): big icons holding several OCR boxes, OCR boxes
    holding icons, in random order, so labels are collected, the walk breaks early, and OCR elements get removed."""
    rng = np.random.default_rng(1000 + seed)
    icons, ob = [], []
    for _ in range(12):                                   # big icons
        x, y = rng.uniform(0.02, 0.7, 2)
        icons.append([x, y, x + rng.uniform(0.08, 0.25), y + rng.uniform(0.06, 0.2)])
    for b in list(icons):                                 # OCR boxes inside big icons (pixels)
        for _ in range(int(rng.integers(0, 4))):
            x0 = b[0] * W + rng.uniform(2, 20); y0 = b[1] * H + rng.uniform(2, 15)
            ob.append([int(x0), int(y0), int(x0 + rng.uniform(20, 60)), int(y0 + rng.uniform(8, 18))])
    for _ in range(10):                                   # large OCR boxes with small icons inside them
        x0, y0 = int(rng.integers(0, W - 400)), int(rng.integers(0, H - 120))
        ob.append([x0, y0, x0 + int(rng.integers(150, 380)), y0 + int(rng.integers(40, 100))])
        icons.append([(x0 + 10) / W, (y0 + 8) / H, (x0 + 40) / W, (y0 + 30) / H])
    for _ in range(40):                                   # clutter
        x, y = rng.uniform(0, 0.9, 2)
        icons.append([x, y, x + rng.uniform(0.0, 0.06), y + rng.uniform(0.0, 0.06)])
    order = rng.permutation(len(ob))
    ob = [ob[i] for i in order]
    icons = [icons[i] for i in rng.permutation(len(icons))]
    texts = [f"w{i}" for i in range(len(ob))]
    return torch.tensor(icons, dtype=torch.float32), ob, texts


@pytest.mark.parametrize("seed", range(12))
def test_dense_overlaps_fast_equals_loops_and_reference(seed):
    icons, ob, texts = _dense_case(seed)
    whwh = torch.Tensor([W, H, W, H])
    oratio = (torch.tensor(ob) / whwh).tolist()
    for thr in THRESHOLDS:
        fast, _ = host_glue.build_elements(icons.tolist(), oratio, texts, W, H, thr)
        slow, _ = host_glue.build_elements(icons.tolist(), oratio, texts, W, H, thr, fast=False)
        assert fast == slow
        assert any(e["source"] == "box_yolo_content_ocr" for e in fast), "case does not exercise label collection"
        assert fast == reference_elements("dense", seed, thr, icons.tolist(), oratio, texts)


# ---------------------------------------------------------------------------------------------- device-filter contract
@pytest.mark.parametrize("seed", range(8))
def test_elements_from_flags_equals_build_elements(seed):
    """Host half of the device overlap filter (SURVEY.md 8f-2): the flag contract of b2p_overlap_filter (restated as loops in
    oracle/ref_restate.py::overlap_flags_loops) + host_glue.elements_from_flags rebuild exactly the element list of the
    reference-pinned build_elements, including duplicated OCR elements (list.remove drops the first equal one)."""
    from oracle.ref_restate import overlap_flags_loops
    icons, ob, texts = _dense_case(seed) if seed % 2 else _case(seed)
    if seed == 3:
        ob = ob + [ob[0], ob[0]]                       # equal OCR dicts
        texts = texts + [texts[0], texts[0]]
    whwh = torch.Tensor([W, H, W, H])
    oratio = (torch.tensor(ob) / whwh).tolist()
    ratio = icons.tolist()
    for thr in (0.7, 0.9):
        ref, _ = host_glue.build_elements(ratio, oratio, texts, W, H, thr)
        ocr_elem = host_glue.ocr_elements(oratio, texts, W, H)
        state, mask, removed = overlap_flags_loops(ratio, [e["bbox"] for e in ocr_elem], W, H, thr)
        got = host_glue.elements_from_flags(ratio, state, mask, ocr_elem, removed)
        assert got == ref
