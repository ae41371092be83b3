"""CPU tests: the oracle restatements against Pillow / OpenCV / torchvision and against what the unmodified reference
wrapper returned (tests/golden/reference_yolov9_predict.json, written by oracle/make_golden.py)."""
import json
from pathlib import Path

import numpy as np
import pytest
import torch

from omniparser_b200 import synth
from oracle import ref_restate as R

GOLD = Path(__file__).resolve().parent / "golden"
PREDICT_SEED, PREDICT_CONF, PREDICT_IOU = 3, 0.05, 0.1


@pytest.mark.parametrize("size,imgsz", [((1920, 1080), 640), ((1919, 1079), 640), ((3240, 2160), 640),
                                        ((300, 200), 640), ((1920, 1080), (1080, 1920)), ((640, 360), 640)])
def test_lanczos_numpy_equals_pillow(size, imgsz):
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, size=(size[1], size[0], 3), dtype=np.uint8)
    a, s1, pl1, pt1 = R.letterbox_pil(img, imgsz)
    b, s2, pl2, pt2 = R.letterbox_numpy(img, imgsz)
    assert (s1, pl1, pt1) == (s2, pl2, pt2)
    assert np.array_equal(a, b)


def test_resize_numpy_equals_cv2():
    import cv2
    rng = np.random.default_rng(2)
    sizes = [(128, 128), (64, 64), (1, 1), (1, 7), (7, 1), (2, 2), (128, 64), (63, 65), (200, 31), (20, 80), (129, 127)]
    sizes += [tuple(int(v) for v in rng.integers(1, 260, size=2)) for _ in range(80)]
    for (h, w) in sizes:
        crop = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        assert np.array_equal(cv2.resize(crop, (64, 64)), R.resize_bilinear_cv2_numpy(crop)), (h, w)


def _rand_boxes(rng, n, ties=True):
    xy = rng.uniform(0, 600, size=(n, 2)).astype(np.float32)
    wh = rng.uniform(0, 120, size=(n, 2)).astype(np.float32)
    boxes = np.concatenate([xy, xy + wh], 1)
    scores = rng.uniform(0.05, 1, size=n).astype(np.float32)
    if ties and n > 4:
        scores[rng.integers(0, n, size=n // 3)] = np.float32(0.5)
        boxes[1] = boxes[0]   # duplicate box, IoU == 1
        boxes[3, 2:] = boxes[3, :2]   # zero-area box
    return boxes, scores


@pytest.mark.parametrize("n,nc", [(0, 1), (1, 1), (7, 1), (300, 1), (999, 3), (1000, 3), (1001, 3), (2500, 1)])
def test_nms_numpy_equals_torchvision(n, nc):
    from torchvision.ops import batched_nms
    rng = np.random.default_rng(n + nc)
    # n > 1000 takes torchvision's per-class path whose final re-sort is NOT stable (tv:ops/boxes.py:107-120):
    # the reference's order among exactly tied scores is implementation-defined there, so no ties in that case.
    boxes, scores = _rand_boxes(rng, n, ties=(n <= 1000))
    cls = rng.integers(0, nc, size=n).astype(np.int64)
    for iou in (0.1, 0.7):
        ref = batched_nms(torch.from_numpy(boxes), torch.from_numpy(scores), torch.from_numpy(cls), iou)[:300].numpy()
        got = R.greedy_nms_numpy(boxes, scores, cls, iou, 300)
        assert np.array_equal(ref, got)


def test_nms_tie_break_and_strictness():
    from torchvision.ops import nms
    # two identical-score overlapping boxes: the lower index wins; IoU == thr keeps both (strict >)
    b = torch.tensor([[0, 0, 10, 10], [0, 0, 10, 10.0]])
    s = torch.tensor([0.5, 0.5])
    assert nms(b, s, 0.5).tolist() == [0]
    assert R.greedy_nms_numpy(b.numpy(), s.numpy(), np.zeros(2, np.int64), 0.5, 300).tolist() == [0]
    b = torch.tensor([[0, 0, 10, 10], [0, 5, 10, 15.0]])   # IoU = 1/3
    thr = float(np.float32(50.0) / np.float32(150.0))
    assert nms(b, s, thr).tolist() == [0, 1]
    assert R.greedy_nms_numpy(b.numpy(), s.numpy(), np.zeros(2, np.int64), thr, 300).tolist() == [0, 1]


def test_restatement_equals_reference_wrapper():
    """End-to-end: unmodified YOLOv9Detector.predict (ref:util/yolov9.py:115-136) on the TorchScript export of the stand-in
    vs the restated pipeline, within the host-to-host noise of the fp32 CPU forward (tests/parity_util.py)."""
    from parity_util import match_cpu_detector
    from standin.yolo_weights import yolo_standin
    g = json.loads((GOLD / "reference_yolov9_predict.json").read_text())
    assert (g["seed"], g["conf"], g["iou"]) == (PREDICT_SEED, PREDICT_CONF, PREDICT_IOU)
    m = yolo_standin(0)
    img = synth.screenshot(PREDICT_SEED)
    canvas, scale, pl, pt = R.letterbox_numpy(img, 640)
    x = torch.from_numpy(canvas.astype(np.float32).transpose(2, 0, 1) / 255.0).unsqueeze(0)
    with torch.no_grad():
        outs = m(x)
    scores, boxes = R.decode_heads(outs)
    b, s, c = R.filter_candidates(scores[0], boxes[0], PREDICT_CONF, scale, pl, pt)
    keep, kb, ks = R.nms_and_clamp(b, s, c, PREDICT_IOU, 300, img.shape[1], img.shape[0])
    assert len(kb) == len(g["xyxy"]) and len(kb) > 5
    match_cpu_detector(kb, ks, g["xyxy"], g["scores"], img.shape[1], img.shape[0])
