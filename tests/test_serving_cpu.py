"""CPU: the two "next" rows around the hot path that are pure host logic --
* §8f-3 ``omniparser_b200.ocr.check_ocr_box`` (the reference's OCR pre-step adapter, ref:util/utils.py:498-549) against fake
  engines and against what the UNMODIFIED reference function returned when driven by the same fake engines
  (tests/golden/reference_check_ocr_box.json, written by oracle/make_golden.py);
* §8f-4 ``omniparser_b200.server.DynamicBatcher`` / ``create_app`` (cross-request batching behind the reference server's wire
  format, ref:omnitool/omniparserserver/omniparserserver.py:37-48): grouping by key, size and deadline triggers, order,
  error delivery, concurrency."""
import json
import threading
import time
from pathlib import Path

import numpy as np
import pytest
from PIL import Image

from omniparser_b200 import ocr as OCR
from omniparser_b200.server import DynamicBatcher

GOLD = Path(__file__).resolve().parent / "golden"
QUADS = [([[10.7, 20.2], [110.1, 20.2], [110.1, 44.9], [10.7, 44.9]], "File", 0.93),
         ([[300, 400], [420, 400], [420, 431], [300, 431]], "Edit view", 0.41),
         ([[5.5, 600.5], [64.4, 600.5], [64.4, 630.0], [5.5, 630.0]], "x", 0.77)]


class _Reader:
    def __init__(self):
        self.kw = None

    def readtext(self, image_np, **kw):
        assert isinstance(image_np, np.ndarray) and image_np.ndim == 3 and image_np.shape[2] == 3
        self.kw = kw
        return QUADS


class _Paddle:
    def ocr(self, image_np, cls=False):
        assert cls is False
        return [[(q, (t, c)) for q, t, c in QUADS]]


@pytest.fixture()
def engines():
    r, p = _Reader(), _Paddle()
    old = dict(OCR._ENGINES)
    OCR.set_engines(easyocr_reader=r, paddle_ocr=p)
    yield r, p
    OCR._ENGINES.update(old)


@pytest.mark.parametrize("mode", ["RGB", "RGBA"])
def test_check_ocr_box_formats(engines, mode, tmp_path):
    reader, _ = engines
    img = Image.fromarray(np.random.default_rng(0).integers(0, 255, (700, 500, 4 if mode == "RGBA" else 3), dtype=np.uint8), mode)
    (text, bb), goal = OCR.check_ocr_box(img, display_img=False, output_bb_format="xyxy", goal_filtering="g",
                                         easyocr_args={"paragraph": False, "text_threshold": 0.9})
    assert goal == "g" and text == ["File", "Edit view", "x"] and reader.kw == {"paragraph": False, "text_threshold": 0.9}
    assert bb == [(10, 20, 110, 44), (300, 400, 420, 431), (5, 600, 64, 630)]
    (_, bb2), _ = OCR.check_ocr_box(img, display_img=False, output_bb_format="xywh")
    assert bb2 == [(10, 20, 99, 24), (300, 400, 120, 31), (5, 600, 58, 29)]
    # PaddleOCR branch: confidence filter at easyocr_args['text_threshold'] (default 0.5)
    (t3, bb3), _ = OCR.check_ocr_box(img, display_img=False, output_bb_format="xyxy", use_paddleocr=True)
    assert t3 == ["File", "x"] and bb3 == [(10, 20, 110, 44), (5, 600, 64, 630)]
    (t4, _), _ = OCR.check_ocr_box(img, display_img=False, output_bb_format="xyxy", use_paddleocr=True, easyocr_args={"text_threshold": 0.4})
    assert t4 == ["File", "Edit view", "x"]
    path = tmp_path / "shot.png"
    img.save(path)
    (t5, bb5), _ = OCR.check_ocr_box(str(path), display_img=False, output_bb_format="xyxy")
    assert (t5, bb5) == (text, bb)
    assert OCR.get_xywh_yolo([3.9, 4.2, 10.1, 20.9]) == (3, 4, 6, 16)


OCR_KWARGS = [dict(output_bb_format="xyxy"), dict(output_bb_format="xywh"), dict(output_bb_format="xyxy", use_paddleocr=True),
              dict(output_bb_format="xyxy", use_paddleocr=True, easyocr_args={"text_threshold": 0.8}),
              dict(output_bb_format="xyxy", easyocr_args={"text_threshold": 0.8})]


def ocr_golden_image():
    return Image.fromarray(np.zeros((700, 500, 4), np.uint8), "RGBA")


def test_check_ocr_box_equals_unmodified_reference(engines):
    """Same engines, same arguments: the same ``repr`` as the reference's result (tuples vs lists and number types included)."""
    gold = json.loads((GOLD / "reference_check_ocr_box.json").read_text())
    assert [g["kwargs"] for g in gold] == OCR_KWARGS
    img = ocr_golden_image()
    for g in gold:
        assert repr(OCR.check_ocr_box(img, display_img=False, goal_filtering=None, **g["kwargs"])) == g["repr"]


def test_missing_engine_raises_clearly(monkeypatch):
    import sys
    monkeypatch.setitem(sys.modules, "easyocr", None)      # `import easyocr` raises ImportError
    monkeypatch.setitem(sys.modules, "paddleocr", None)
    monkeypatch.setitem(OCR._ENGINES, "easyocr", None)
    monkeypatch.setitem(OCR._ENGINES, "paddle", None)
    with pytest.raises(RuntimeError, match="EasyOCR is not installed"):
        OCR.check_ocr_box(Image.new("RGB", (8, 8)), display_img=False, output_bb_format="xyxy")
    with pytest.raises(RuntimeError, match="PaddleOCR is not installed"):
        OCR.check_ocr_box(Image.new("RGB", (8, 8)), display_img=False, output_bb_format="xyxy", use_paddleocr=True)


# ---------------------------------------------------------------------------------------------- batching
def test_batcher_groups_by_key_size_and_deadline():
    seen = []

    def run(key, items):
        seen.append((key, list(items)))
        time.sleep(0.01)
        return [(key, x * 2) for x in items]

    b = DynamicBatcher(run, max_batch=4, max_wait_s=0.05)
    out = {}

    def call(key, x):
        out[(key, x)] = b.submit(key, x)

    th = [threading.Thread(target=call, args=("a" if i % 3 else "b", i)) for i in range(14)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    b.close()
    assert out == {(k, x): (k, 2 * x) for (k, x) in out} and len(out) == 14
    assert all(len(items) <= 4 for _, items in seen) and all(len({k}) == 1 for k, _ in seen)
    assert sum(len(i) for _, i in seen) == 14 and len(seen) < 14            # requests really shared batches
    assert b.stats["items"] == 14 and b.stats["max_batch_seen"] <= 4
    # a lone request is dispatched after the deadline, not held for a full batch
    b2 = DynamicBatcher(lambda k, it: it, max_batch=8, max_wait_s=0.02)
    t0 = time.monotonic()
    assert b2.submit("k", 5) == 5
    assert 0.015 <= time.monotonic() - t0 < 0.5
    b2.close()


def test_batcher_delivers_errors_and_keeps_serving():
    def run(key, items):
        if key == "bad":
            raise ValueError("boom")
        return items

    b = DynamicBatcher(run, max_batch=2, max_wait_s=0.005)
    with pytest.raises(ValueError, match="boom"):
        b.submit("bad", 1)
    assert b.submit("ok", 2) == 2
    b.close()
    with pytest.raises(RuntimeError):
        b.submit("ok", 3)


def test_app_routes_and_wire_format():
    """The FastAPI app exposes the reference's routes and JSON schema (ref:omnitool/omniparserserver/omniparserserver.py:33-48)."""
    from omniparser_b200.server import create_app, parse_arguments

    class _P:
        def parse(self, b64):
            return "PNG" + b64[:3], [{"type": "icon", "bbox": [0, 0, 1, 1], "interactivity": True, "content": "c", "source": "box_yolo_content_yolo"}]

    app = create_app({}, parser=_P())
    routes = {r.path: r for r in app.routes if hasattr(r, "endpoint")}
    assert "/parse/" in routes and "/probe/" in routes and "POST" in routes["/parse/"].methods and "GET" in routes["/probe/"].methods
    req_model = routes["/parse/"].endpoint.__annotations__["parse_request"]
    body = routes["/parse/"].endpoint(req_model(base64_image="abcdef"))
    assert set(body) == {"som_image_base64", "parsed_content_list", "latency"} and body["som_image_base64"] == "PNGabc"
    assert routes["/probe/"].endpoint() == {"message": "Omniparser API ready"}
    a = parse_arguments(["--BOX_TRESHOLD", "0.1", "--port", "9000"])
    assert a.BOX_TRESHOLD == 0.1 and a.port == 9000 and a.caption_model_name == "florence2" and a.max_batch == 8
