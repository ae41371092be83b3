"""CPU: the reference facade (ref:util/omniparser.py:7-32), UNMODIFIED, calls the three hot functions with arguments that
bind to the drop-in's signatures -- i.e. swapping ``util.utils`` for ``omniparser_b200.utils`` in its import line is the whole
integration.  The calls are the ones the reference file made when it parsed a 160x90 PNG with recorders in place of
``util.utils`` (tests/golden/reference_facade_calls.json, written by oracle/make_golden.py); tests/test_boundary_gpu.py runs
the swapped facade for real on the GPU."""
import inspect
import json
from pathlib import Path

from PIL import Image

from omniparser_b200 import utils as B

GOLD = Path(__file__).resolve().parent / "golden"


def _decode(v):
    if isinstance(v, dict) and set(v) == {"pil_image"}:
        w, h, mode = v["pil_image"]
        return Image.new(mode, (w, h))
    return v


def test_reference_facade_binds_to_the_drop_in_signatures():
    g = json.loads((GOLD / "reference_facade_calls.json").read_text())
    drop_in = {"get_yolo_model": B.get_yolo_model, "get_caption_model_processor": B.get_caption_model_processor,
               "get_som_labeled_img": B.get_som_labeled_img}
    calls = []
    for c in g["calls"]:
        sig = inspect.signature(drop_in[c["name"]])
        # TypeError here = the reference passes something the drop-in does not accept
        ba = sig.bind(*[_decode(v) for v in c["args"]], **{k: _decode(v) for k, v in c["kwargs"].items()})
        calls.append((c["name"], dict(ba.arguments)))
    assert g["returned"] == ["b64", [{"type": "icon"}]]
    names = [c[0] for c in calls]
    assert names == ["get_yolo_model", "get_caption_model_processor", "get_som_labeled_img"]
    kw = calls[2][1]
    assert kw["BOX_TRESHOLD"] == 0.05 and kw["output_coord_in_ratio"] is True and kw["iou_threshold"] == 0.7 and kw["batch_size"] == 128
    assert set(kw["draw_bbox_config"]) == {"text_scale", "text_thickness", "text_padding", "thickness"}
    # the drop-in's own facade is the same file after the import swap: same public surface
    from omniparser_b200.omniparser import Omniparser
    assert list(inspect.signature(Omniparser.parse).parameters) == g["parse_parameters"]
