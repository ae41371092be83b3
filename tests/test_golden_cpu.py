"""CPU: the oracle pipeline (oracle/pipeline_cpu.py) reproduces the golden fixtures that the UNMODIFIED reference
(`get_som_labeled_img` + `YOLOv9Detector`, run through oracle/make_golden.py) produced: detector boxes and scores within
the host-to-host noise of the fp32 CPU forward (tests/parity_util.py), in the same order; on the reference's own detector
boxes, parsed_content_list (order, sources, bboxes, OCR-derived content) identical and greedy caption token ids identical."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from omniparser_b200 import synth
from oracle.pipeline_cpu import OraclePipeline
from parity_util import match_cpu_detector

GOLD = Path(__file__).resolve().parent / "golden"


@pytest.fixture(scope="module")
def pipe():
    return OraclePipeline()


# synth_seed5_3240x2160: the geometry of ref:imgs/demo_image.jpg (BASELINE configs[0]: letterbox 640x426 -> canvas 640x448)
@pytest.mark.parametrize("name", ["synth_seed0", "synth_seed3_odd", "synth_seed5_3240x2160"])
def test_oracle_pipeline_equals_reference_golden(pipe, name):
    g = json.loads((GOLD / f"{name}.json").read_text())
    w, h = g["case"]["size"]
    img = synth.screenshot(g["case"]["seed"], w, h)
    texts, boxes = synth.ocr_boxes(g["case"]["seed"], w, h)
    kb, ks = pipe.detect(img, g["box_threshold"], 0.1)
    match_cpu_detector(kb, ks, g["det_xyxy"], g["det_conf"], w, h)
    elems, ids = pipe.parse(img, texts, boxes, BOX_TRESHOLD=g["box_threshold"], iou_threshold=g["iou_threshold"],
                            max_new_tokens=g["max_new_tokens"], det_boxes=g["det_xyxy"])
    assert ids.tolist() == g["caption_ids"]
    assert len(elems) == len(g["parsed_content_list"])
    for a, b in zip(elems, g["parsed_content_list"]):
        assert a["type"] == b["type"] and a["source"] == b["source"] and a["interactivity"] == b["interactivity"]
        assert a["bbox"] == b["bbox"]
        assert a["content"].strip() == b["content"].strip()


# Real screenshots of the reference repo (ref:imgs/*, byte copies under tests/golden/imgs) parsed by the UNMODIFIED reference with
# the ScreenSpot-Pro eval's call-site parameters (ref:eval/ss_pro_gpt4o_omniv2.py:37-51; oracle/make_golden.py real_goldens):
# BASELINE configs[0] (imgs/demo_image.jpg) and the configs[4] call site.  Two of the four cases run here (CPU time); all
# four run against the GPU path in tests/test_boundary_gpu.py.
@pytest.mark.parametrize("name", ["real_header_bar_thin", "real_demo_image"])
def test_oracle_pipeline_equals_reference_golden_on_real_images(pipe, name):
    from PIL import Image
    g = json.loads((GOLD / f"{name}.json").read_text())
    img = np.asarray(Image.open(GOLD / "imgs" / g["case"]["file"]).convert("RGB"))
    assert [img.shape[1], img.shape[0]] == g["case"]["size"]
    kb, ks = pipe.detect(img, g["box_threshold"], 0.1)
    match_cpu_detector(kb, ks, g["det_xyxy"], g["det_conf"], img.shape[1], img.shape[0])
    elems, ids = pipe.parse(img, g["ocr_text"], g["ocr_bbox"], BOX_TRESHOLD=g["box_threshold"], iou_threshold=g["iou_threshold"],
                            max_new_tokens=g["max_new_tokens"], det_boxes=g["det_xyxy"])
    assert ids.tolist() == g["caption_ids"]
    assert len(elems) == len(g["parsed_content_list"])
    for a, b in zip(elems, g["parsed_content_list"]):
        assert a["type"] == b["type"] and a["source"] == b["source"] and a["bbox"] == b["bbox"]
        assert a["content"].strip() == b["content"].strip()
