"""ORACLE (test infrastructure): generate tests/golden/*.json by running the UNMODIFIED reference
(``/root/reference/util/utils.py::get_som_labeled_img`` + ``util/yolov9.py::YOLOv9Detector``) on the seeded stand-ins.
Runs only where /root/reference exists (this container): ``python -m oracle.make_golden``.

The reference's caption branch depends on ``model.device.type`` (ref:util/utils.py:120-123).  The goldens pin the
CUDA-branch semantics (64x64 crops, ``do_resize=False``), executed on the CPU in fp32: the stand-in caption model
reports a ``device`` whose ``.type`` is 'cuda' so the unmodified reference code takes that branch, and the stand-in
processor's ``.to(device, dtype)`` keeps fp32 (the reference's fp16 cast is a precision choice, not semantics).
"""
from __future__ import annotations

import json
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch
from PIL import Image

from omniparser_b200 import synth

from standin import florence as FS
from .shims import import_reference
from standin.yolo_weights import GOLDEN, yolo_standin
from standin.yolov9e import export_torchscript

CASES = [dict(name="synth_seed0", seed=0, size=(1920, 1080)), dict(name="synth_seed3_odd", seed=3, size=(1919, 1079)),
         dict(name="synth_seed5_3240x2160", seed=5, size=(3240, 2160))]   # geometry of ref:imgs/demo_image.jpg (BASELINE configs[0])
BOX_TRESHOLD, IOU = 0.05, 0.7


class _Batch(dict):
    def to(self, device=None, dtype=None):
        return self


class _Processor:
    """What AutoProcessor('microsoft/Florence-2-base') does for ``do_resize=False`` (needs the network, hence restated)."""

    def __call__(self, images, text, return_tensors="pt", do_resize=True):
        assert do_resize is False, "goldens pin the CUDA-branch (64x64) semantics"
        u8 = torch.from_numpy(np.stack([np.asarray(im) for im in images]))
        return _Batch(input_ids=FS.input_ids_for(len(images)), pixel_values=FS.pixel_values_from_u8(u8))

    def batch_decode(self, ids, skip_special_tokens=True):
        return [" ".join(f"<{t}>" for t in row if t not in (0, 1, 2)) for row in ids.tolist()]


class _Model:
    def __init__(self, hf):
        self.hf = hf
        self.config = SimpleNamespace(model_type="florence2", name_or_path="seeded/florence2-standin")
        self.device = SimpleNamespace(type="cuda")
        self.ids = []

    def generate(self, **kw):
        out = self.hf.generate(**kw)
        self.ids.append(out)
        return out


def _overlay_sha(png_b64: str, size) -> str:
    """sha256 of the decoded RGB pixels of the reference's annotated PNG (the PNG byte stream itself is encoder-specific)."""
    import base64, hashlib, io
    im = Image.open(io.BytesIO(base64.b64decode(png_b64))).convert("RGB")
    assert im.size == tuple(size)
    return hashlib.sha256(np.asarray(im).tobytes()).hexdigest()


FACADE = dict(name="facade_seed7", seed=7, size=(1920, 1080))


def facade_golden(path, fl):
    """The reference's own facade, ``util/omniparser.py::Omniparser`` (ref:util/omniparser.py:7-32), run UNMODIFIED: the
    easyocr stand-in returns fixed quads (OCR is outside the hot path), ``get_yolo_model`` loads the TorchScript archive,
    and only ``get_caption_model_processor`` -- which needs the network for microsoft/Florence-2-base, ref:util/utils.py:64 --
    is replaced in the facade's namespace by the seeded stand-in pair."""
    import base64, io, sys
    import easyocr
    ro = __import__("util.omniparser", fromlist=["Omniparser"])
    w, h = FACADE["size"]
    img = synth.screenshot(FACADE["seed"], w, h)
    texts, boxes = synth.ocr_boxes(FACADE["seed"], w, h)
    quads = [([[b[0], b[1]], [b[2], b[1]], [b[2], b[3]], [b[0], b[3]]], t, 0.99) for b, t in zip(boxes, texts)]
    import util.utils as ru
    ru.reader.readtext = lambda image_np, **kw: quads                       # the instance created at ref:util/utils.py:22
    cm = _Model(fl)
    ro.get_caption_model_processor = lambda **kw: {"model": cm, "processor": _Processor()}
    op = ro.Omniparser({"som_model_path": str(path), "caption_model_name": "florence2", "caption_model_path": "seeded/florence2-standin",
                        "BOX_TRESHOLD": BOX_TRESHOLD})
    buf = io.BytesIO()
    Image.fromarray(img).save(buf, format="PNG")
    png, parsed = op.parse(base64.b64encode(buf.getvalue()).decode("ascii"))
    ids = torch.cat(cm.ids, 0) if cm.ids else torch.zeros((0, 1), dtype=torch.long)
    gold = dict(case=FACADE, config=dict(BOX_TRESHOLD=BOX_TRESHOLD), ocr_text=texts, ocr_bbox=boxes, parsed_content_list=parsed,
                caption_ids=ids.tolist(), overlay_sha256=_overlay_sha(png, (w, h)))
    out = GOLDEN / f"{FACADE['name']}.json"
    out.write_text(json.dumps(gold, default=lambda o: float(o) if isinstance(o, (np.floating,)) else o.tolist()))
    print("wrote", out, len(parsed), "elements,", ids.shape[0], "captions")


# Real screenshots shipped with the reference (ref:imgs/*), parsed with the ScreenSpot-Pro eval's call-site parameters
# (ref:eval/ss_pro_gpt4o_omniv2.py:37-51: draw_bbox_config scaled by max(size)/3200, BOX_TRESHOLD 0.05, iou_threshold 0.7,
# output_coord_in_ratio, image passed as a PATH).  BASELINE configs[0] = imgs/demo_image.jpg; configs[4]'s dataset is not
# on disk, so the same call site is replayed on the reference's own images (SURVEY.md 8d).  The images travel as fixtures
# (tests/golden/imgs/, byte copies: /root/reference does not exist on the GPU box); OCR boxes are seeded (OCR is outside the path).
REAL_CASES = [dict(name="real_demo_image", file="demo_image.jpg", seed=11), dict(name="real_omni3", file="omni3.jpg", seed=12),
              dict(name="real_excel_rgba", file="excel.png", seed=13), dict(name="real_header_bar_thin", file="header_bar_thin.png", seed=14)]


def eval_draw_config(size):
    r = max(size) / 3200
    return {"text_scale": 0.8 * r, "text_thickness": max(int(2 * r), 1), "text_padding": max(int(3 * r), 1), "thickness": max(int(3 * r), 1)}


def real_goldens(ru, det, fl):
    import shutil
    (GOLDEN / "imgs").mkdir(exist_ok=True)
    for case in REAL_CASES:
        src = Path("/root/reference/imgs") / case["file"]
        dst = GOLDEN / "imgs" / case["file"]
        if not dst.exists():
            shutil.copyfile(src, dst)
        image = Image.open(dst)
        w, h = image.size
        texts, boxes = synth.ocr_boxes(case["seed"], w, h)
        raw = det.predict(image.convert("RGB"), conf=BOX_TRESHOLD, iou=0.1)[0].boxes
        cm = _Model(fl)
        cfg = eval_draw_config(image.size)
        png, coords, parsed = ru.get_som_labeled_img(str(dst), det, BOX_TRESHOLD=BOX_TRESHOLD, output_coord_in_ratio=True, ocr_bbox=boxes,
                                                   draw_bbox_config=cfg, caption_model_processor={"model": cm, "processor": _Processor()},
                                                   ocr_text=texts, use_local_semantics=True, iou_threshold=IOU, scale_img=False, batch_size=128)
        ids = torch.cat(cm.ids, 0) if cm.ids else torch.zeros((0, 1), dtype=torch.long)
        gold = dict(case=dict(case, size=[w, h], mode=image.mode), box_threshold=BOX_TRESHOLD, iou_threshold=IOU, max_new_tokens=20,
                    draw_bbox_config=cfg, ocr_text=texts, ocr_bbox=boxes,
                    det_xyxy=[[float(np.float32(v)) for v in b] for b in raw.xyxy.tolist()], det_conf=[float(c) for c in raw.conf.tolist()],
                    parsed_content_list=parsed, caption_ids=ids.tolist(), label_coordinates=coords,
                    overlay_sha256=_overlay_sha(png, (w, h)))
        out = GOLDEN / f"{case['name']}.json"
        out.write_text(json.dumps(gold, default=lambda o: float(o) if isinstance(o, (np.floating,)) else o.tolist()))
        print("wrote", out, len(raw.xyxy), "boxes,", ids.shape[0], "captions", flush=True)


# What the CPU tests compare with the reference, beyond the parse goldens above: the reference's own functions run on the
# tests' seeded inputs (the tests' input generators are imported from tests/, so inputs cannot drift apart).
def _tests_module(name):
    import importlib
    import sys
    tests = Path(__file__).resolve().parents[1] / "tests"
    if str(tests) not in sys.path:
        sys.path.insert(0, str(tests))
    return importlib.import_module(name)


def _write_json(name, gold):
    out = GOLDEN / name
    out.write_text(json.dumps(gold, separators=(",", ":")))
    print("wrote", out, out.stat().st_size, "bytes", flush=True)


def facade_calls_golden():
    """ref:util/omniparser.py, unmodified, parses one 160x90 PNG with ``util.utils`` replaced by recorders: the functions
    it calls and the arguments it passes them (tests/test_facade_cpu.py binds them to the drop-in's signatures)."""
    import base64, inspect, io, sys, types
    from .shims import REFERENCE
    calls = []

    def enc(v):
        return {"pil_image": [v.size[0], v.size[1], v.mode]} if isinstance(v, Image.Image) else v

    def rec(name, ret):
        def f(*a, **k):
            calls.append(dict(name=name, args=[enc(v) for v in a], kwargs={kk: enc(v) for kk, v in k.items()}))
            return ret
        return f

    fake = types.ModuleType("util.utils")
    fake.get_yolo_model = rec("get_yolo_model", "som")
    fake.get_caption_model_processor = rec("get_caption_model_processor", {"model": "m", "processor": "p"})
    fake.get_som_labeled_img = rec("get_som_labeled_img", ("b64", {"0": [0, 0, 1, 1]}, [{"type": "icon"}]))
    fake.check_ocr_box = lambda image, **kw: ((["t"], [[1, 2, 30, 40]]), None)
    pkg = types.ModuleType("util")
    pkg.__path__ = [str(REFERENCE / "util")]
    saved = {k: sys.modules.get(k) for k in ("util", "util.utils", "util.omniparser")}
    sys.modules.update({"util": pkg, "util.utils": fake})
    sys.modules.pop("util.omniparser", None)
    try:
        ro = __import__("util.omniparser", fromlist=["Omniparser"])
        config = {"som_model_path": "weights/icon_detect_v3/model.pt", "caption_model_name": "florence2",
                  "caption_model_path": "weights/icon_caption_florence", "BOX_TRESHOLD": 0.05}
        op = ro.Omniparser(config)
        buf = io.BytesIO()
        Image.fromarray(np.zeros((90, 160, 3), np.uint8)).save(buf, format="PNG")
        returned = op.parse(base64.b64encode(buf.getvalue()).decode("ascii"))
        parse_parameters = list(inspect.signature(ro.Omniparser.parse).parameters)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    _write_json("reference_facade_calls.json", dict(config=config, calls=calls, returned=list(returned),
                                                    parse_parameters=parse_parameters))


def overlap_golden(ru):
    """``remove_overlap_new`` (ref:util/utils.py:241-319) behind the ``int_box_area`` filters and the final sort of
    ref:util/utils.py:437-451, on every case of tests/test_host_glue_cpu.py, stored in that test's compact encoding."""
    import copy
    T = _tests_module("test_host_glue_cpu")
    whwh = torch.Tensor([T.W, T.H, T.W, T.H])
    cases = {}
    for kind, make, seeds in (("case", T._case, range(6)), ("dense", T._dense_case, range(12))):
        for seed in seeds:
            icons, ob, texts = make(seed)
            ratio, oratio = icons.tolist(), (torch.tensor(ob) / whwh).tolist()
            for thr in T.THRESHOLDS:
                ocr_elem = [{'type': 'text', 'bbox': box, 'interactivity': False, 'content': txt, 'source': 'box_ocr_content_ocr'}
                            for box, txt in zip(oratio, texts) if ru.int_box_area(box, T.W, T.H) > 0]
                xyxy_elem = [{'type': 'icon', 'bbox': box, 'interactivity': True, 'content': None} for box in ratio
                             if ru.int_box_area(box, T.W, T.H) > 0]
                ref = ru.remove_overlap_new(boxes=xyxy_elem, iou_threshold=thr, ocr_bbox=copy.deepcopy(ocr_elem))
                ref = sorted(ref, key=lambda x: x['content'] is None)
                enc = []
                for e in ref:
                    if e["source"] == "box_ocr_content_ocr":
                        enc.append(["o", next(k for k in range(len(oratio)) if oratio[k] == e["bbox"] and texts[k] == e["content"])])
                    else:
                        enc.append(["i", ratio.index(e["bbox"]), e["content"]])
                assert T.decode_elements(enc, ratio, oratio, texts) == ref
                cases[T.case_key(kind, seed, thr)] = enc
    _write_json("reference_remove_overlap_new.json", cases)


def predict_golden(ry, path):
    """``YOLOv9Detector.predict`` (ref:util/yolov9.py:115-136) on the TorchScript stand-in, tests/test_oracle_cpu.py's case."""
    T = _tests_module("test_oracle_cpu")
    det = ry.YOLOv9Detector(model_path=path, device="cpu")
    ref = det.predict(Image.fromarray(synth.screenshot(T.PREDICT_SEED)), conf=T.PREDICT_CONF, iou=T.PREDICT_IOU)[0].boxes
    _write_json("reference_yolov9_predict.json", dict(seed=T.PREDICT_SEED, conf=T.PREDICT_CONF, iou=T.PREDICT_IOU,
                                                      xyxy=ref.xyxy.tolist(), scores=ref.conf.tolist()))


def check_ocr_box_golden(ru):
    """``check_ocr_box`` (ref:util/utils.py:514-549) driven by tests/test_serving_cpu.py's fake OCR engines; ``repr`` of the
    result, so that tuples, lists and number types are pinned too."""
    T = _tests_module("test_serving_cpu")
    old_r, old_p = ru.reader, ru.paddle_ocr
    ru.reader, ru.paddle_ocr = T._Reader(), T._Paddle()
    try:
        img = T.ocr_golden_image()
        calls = [dict(kwargs=kw, repr=repr(ru.check_ocr_box(img, display_img=False, goal_filtering=None, **kw)))
                 for kw in T.OCR_KWARGS]
    finally:
        ru.reader, ru.paddle_ocr = old_r, old_p
    _write_json("reference_check_ocr_box.json", calls)


def annotate_golden(ru):
    """``annotate`` (ref:util/utils.py:336-366, util/box_annotator.py) on tests/test_overlay_cpu.py's layouts: sha256 of
    the annotated frame and the label coordinates, in one .npz."""
    import hashlib
    from torchvision.ops import box_convert
    T = _tests_module("test_overlay_cpu")
    arrays = {}
    for seed, n, (w, h), cfg in T.LAYOUTS:
        for crowded in (False, True):
            img = synth.screenshot(seed, w, h)
            boxes = T._layout(seed, n, w, h, crowded)
            t = box_convert(torch.tensor(boxes).reshape(-1, 4), "xyxy", "cxcywh")
            frame, coords = ru.annotate(image_source=img, boxes=t, logits=None, phrases=list(range(n)), **cfg)
            key = T.layout_key(seed, crowded)
            arrays[key + "_sha256"] = np.array(hashlib.sha256(frame.tobytes()).hexdigest())
            arrays[key + "_shape"] = np.array(frame.shape, np.int64)
            arrays[key + "_coords"] = np.array([coords[str(i)] for i in range(n)], np.float32).reshape(n, 4)
    out = GOLDEN / "reference_annotate_layouts.npz"
    np.savez_compressed(out, **arrays)
    print("wrote", out, out.stat().st_size, "bytes", flush=True)


def reference_call_goldens(ru, ry, path):
    facade_calls_golden()
    overlap_golden(ru)
    predict_golden(ry, path)
    check_ocr_box_golden(ru)
    annotate_golden(ru)


def main():
    import sys
    ru, ry = import_reference()
    m = yolo_standin(0)
    path = Path("/tmp/b2p_golden/icon_detect_v3/model.pt")
    export_torchscript(m, path, (640, 640))
    det = ru.get_yolo_model(str(path), device="cpu")
    assert type(det).__name__ == "YOLOv9Detector"
    fl = FS.florence_standin(0)
    if "real" in sys.argv[1:]:          # python -m oracle.make_golden real  -> only the real-image goldens
        real_goldens(ru, det, fl)
        return
    if "calls" in sys.argv[1:]:         # python -m oracle.make_golden calls -> only the reference-call goldens
        reference_call_goldens(ru, ry, path)
        return
    for case in CASES:
        w, h = case["size"]
        img = synth.screenshot(case["seed"], w, h)
        texts, boxes = synth.ocr_boxes(case["seed"], w, h)
        raw = det.predict(Image.fromarray(img), conf=BOX_TRESHOLD, iou=0.1)[0].boxes
        cm = _Model(fl)
        png, coords, parsed = ru.get_som_labeled_img(Image.fromarray(img), det, BOX_TRESHOLD=BOX_TRESHOLD, output_coord_in_ratio=True,
                                                   ocr_bbox=boxes, draw_bbox_config=None,
                                                   caption_model_processor={"model": cm, "processor": _Processor()},
                                                   ocr_text=texts, use_local_semantics=True, iou_threshold=IOU, scale_img=False,
                                                   batch_size=128)
        ids = torch.cat(cm.ids, 0) if cm.ids else torch.zeros((0, 1), dtype=torch.long)
        gold = dict(case=case, box_threshold=BOX_TRESHOLD, iou_threshold=IOU, max_new_tokens=20,
                    det_xyxy=[[float(np.float32(v)) for v in b] for b in raw.xyxy.tolist()], det_conf=[float(c) for c in raw.conf.tolist()],
                    parsed_content_list=parsed, caption_ids=ids.tolist(), label_coordinates=coords,
                    overlay_sha256=_overlay_sha(png, (w, h)))
        out = GOLDEN / f"{case['name']}.json"
        out.write_text(json.dumps(gold, default=lambda o: float(o) if isinstance(o, (np.floating,)) else o.tolist()))
        print("wrote", out, len(raw.xyxy), "boxes,", ids.shape[0], "captions")
    facade_golden(path, fl)
    real_goldens(ru, det, fl)
    reference_call_goldens(ru, ry, path)


if __name__ == "__main__":
    main()
