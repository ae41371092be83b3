"""CPU: the post-caption part of ``get_som_labeled_img`` (SURVEY.md §8a row G1, §8f-1) -- label coordinates, BoxAnnotator-exact
label placement + drawing, PNG -- against (a) the goldens written by the UNMODIFIED reference (``label_coordinates`` values
and the sha256 of its annotated pixels), (b) torchvision's ``box_convert`` bit for bit, and (c) what the unmodified
``util/box_annotator.py`` + ``util/utils.annotate`` drew on random crowded layouts (sha256 of every pixel and the label
coordinates, tests/golden/reference_annotate_layouts.npz, written by oracle/make_golden.py)."""
import base64
import hashlib
import io
import json
from pathlib import Path

import numpy as np
import pytest
import torch
from PIL import Image

from omniparser_b200 import som_overlay as SO
from omniparser_b200 import synth

GOLD = Path(__file__).resolve().parent / "golden"
CASES = ["synth_seed0", "synth_seed3_odd", "synth_seed5_3240x2160"]


@pytest.mark.parametrize("name", CASES)
def test_label_coordinates_and_overlay_equal_reference_golden(name):
    g = json.loads((GOLD / f"{name}.json").read_text())
    w, h = g["case"]["size"]
    img = synth.screenshot(g["case"]["seed"], w, h)
    boxes = [e["bbox"] for e in g["parsed_content_list"]]
    png_b64, coords, frame = SO.som_outputs(img, boxes, True)          # text_scale 0.4 / padding 5: draw_bbox_config=None
    assert set(coords) == set(g["label_coordinates"])
    for k, v in g["label_coordinates"].items():
        assert [float(x) for x in coords[k]] == v, (k, coords[k], v)
    assert hashlib.sha256(frame.tobytes()).hexdigest() == g["overlay_sha256"]
    back = np.asarray(Image.open(io.BytesIO(base64.b64decode(png_b64))).convert("RGB"))
    assert back.shape == frame.shape and np.array_equal(back, frame)  # the fast PNG decodes to the reference's pixels


@pytest.mark.parametrize("name", ["real_demo_image", "real_omni3", "real_excel_rgba", "real_header_bar_thin"])
def test_real_image_overlay_with_eval_draw_config_equals_reference_golden(name):
    """ref:imgs/* with the eval call site's draw_bbox_config (ref:eval/ss_pro_gpt4o_omniv2.py:38-44): label coordinates and
    every pixel of the annotated image equal what the unmodified reference produced (oracle/make_golden.py real_goldens)."""
    g = json.loads((GOLD / f"{name}.json").read_text())
    img = np.asarray(Image.open(GOLD / "imgs" / g["case"]["file"]).convert("RGB"))
    boxes = [e["bbox"] for e in g["parsed_content_list"]]
    _, coords, frame = SO.som_outputs(img, boxes, True, **g["draw_bbox_config"])
    assert set(coords) == set(g["label_coordinates"])
    for k, v in g["label_coordinates"].items():
        assert [float(x) for x in coords[k]] == v, (k, coords[k], v)
    assert hashlib.sha256(frame.tobytes()).hexdigest() == g["overlay_sha256"]


def test_float32_box_arithmetic_equals_torchvision():
    from torchvision.ops import box_convert
    rng = np.random.default_rng(5)
    xy = rng.random((500, 2), dtype=np.float32)
    wh = rng.random((500, 2), dtype=np.float32) * np.float32(0.2)
    b = np.concatenate([xy, np.minimum(xy + wh, np.float32(1))], 1).astype(np.float32)
    for (w, h) in ((1920, 1080), (3240, 2160), (1919, 1079)):
        t = box_convert(torch.tensor(b.tolist()), "xyxy", "cxcywh")
        c = SO.boxes_cxcywh_f32(b.tolist())
        assert np.array_equal(c, t.numpy())
        tp = t * torch.Tensor([w, h, w, h])
        xyxy, xywh = SO.pixel_boxes_f32(c, w, h)
        assert np.array_equal(xyxy, box_convert(tp, "cxcywh", "xyxy").numpy())
        assert np.array_equal(xywh, box_convert(tp, "cxcywh", "xywh").numpy())


def _layout(seed, n, w, h, crowded):
    rng = np.random.default_rng(seed)
    if crowded:   # a tight grid with little room for labels: every fallback position of get_optimal_label_pos gets used
        side = int(np.ceil(np.sqrt(n)))
        cx = (np.arange(n) % side + 0.5) / side
        cy = (np.arange(n) // side + 0.5) / side
        bw = rng.uniform(0.5, 0.95, n) / side
        bh = rng.uniform(0.5, 0.95, n) / side
    else:
        cx, cy = rng.random(n), rng.random(n)
        bw, bh = rng.uniform(0.01, 0.2, n), rng.uniform(0.01, 0.2, n)
    b = np.stack([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2], 1).clip(0, 1).astype(np.float32)
    return b.tolist()


LAYOUTS = [
    (0, 60, (1920, 1080), dict(text_scale=0.4, text_padding=5)),
    (1, 150, (1920, 1080), dict(text_scale=0.48, text_thickness=1, text_padding=1, thickness=1)),      # util/omniparser.py:21-27 at 1920 px
    (2, 300, (3240, 2160), dict(text_scale=0.81, text_thickness=2, text_padding=3, thickness=3)),
    (3, 40, (640, 480), dict(text_scale=0.8, text_padding=5)),
    (4, 0, (320, 200), dict(text_scale=0.4, text_padding=5)),
]


def layout_key(seed, crowded):
    return f"seed{seed}_{'crowded' if crowded else 'spread'}"


@pytest.mark.parametrize("seed,n,size,cfg", LAYOUTS)
@pytest.mark.parametrize("crowded", [False, True])
def test_overlay_equals_unmodified_box_annotator(seed, n, size, cfg, crowded):
    ref = np.load(GOLD / "reference_annotate_layouts.npz")
    key = layout_key(seed, crowded)
    w, h = size
    img = synth.screenshot(seed, w, h)
    boxes = _layout(seed, n, w, h, crowded)
    _, coords, frame = SO.som_outputs(img, boxes, False, **cfg)
    assert list(frame.shape) == ref[key + "_shape"].tolist()
    assert hashlib.sha256(frame.tobytes()).hexdigest() == str(ref[key + "_sha256"])
    ref_coords = ref[key + "_coords"]
    assert ref_coords.shape == (n, 4)
    assert all(np.array_equal(np.asarray(coords[str(i)]), ref_coords[i]) for i in range(n))


def test_png_levels_decode_identically():
    img = synth.screenshot(9)
    for level in (1, 6):
        back = np.asarray(Image.open(io.BytesIO(SO.encode_png(img, level))).convert("RGB"))
        assert np.array_equal(back, img)
