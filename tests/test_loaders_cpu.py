"""CPU: the loader path real artefacts take (SURVEY.md §8a row D0, §8b) -- a TorchScript archive under
``.../icon_detect_v3/model.pt`` with upstream ``model.N.*`` names (ref:util/utils.py:72-85, ref:util/yolov9.py:32-50) and
a safetensors directory with the microsoft/Florence-2 remote-code names + ``generation_config.json``
(ref:util/utils.py:48-69, ref:README.md:45-46) -- exercised by exporting the seeded stand-ins under those names.
The GPU tests (tests/test_boundary_gpu.py) then run the loaded models end to end."""
import json

import pytest
import torch

from omniparser_b200 import caption
from omniparser_b200.florence_engine import FlorenceWeights
from omniparser_b200.yolo_engine import YoloWeights, rename_upstream
from standin import florence as FS
from standin.yolo_weights import yolo_standin
from standin.yolov9e import UpstreamNamedYOLOv9E, export_torchscript

CPU = torch.device("cpu")


@pytest.fixture(scope="module")
def yolo():
    return yolo_standin(0)


@pytest.fixture(scope="module")
def archive(yolo, tmp_path_factory):
    p = tmp_path_factory.mktemp("w") / "icon_detect_v3" / "model.pt"
    export_torchscript(UpstreamNamedYOLOv9E(yolo).eval(), p, (64, 64))
    return p


def _same_weights(a: YoloWeights, b: YoloWeights):
    assert set(a.W) == set(b.W)
    for k, wa in a.W.items():
        wb = b.W[k]
        if isinstance(wa, int):
            assert wa == wb
            continue
        assert torch.equal(wa.w, wb.w) and torch.equal(wa.b, wb.b), k


def test_torchscript_archive_with_upstream_names(yolo, archive):
    sd = torch.jit.load(str(archive), map_location="cpu").state_dict()
    assert all(k.startswith("model.") for k in sd) and any(k.startswith("model.42.cv2.") for k in sd)
    got = YoloWeights(rename_upstream(sd), CPU)
    _same_weights(got, YoloWeights(yolo.state_dict(), CPU))
    # the traced archive computes what the stand-in computes (it is what the unmodified reference would run)
    x = torch.rand(1, 3, 64, 64)
    with torch.no_grad():
        a, b = torch.jit.load(str(archive))(x), yolo(x)
    assert all(torch.equal(u, v) for u, v in zip(a, b))


def test_archive_with_unknown_or_missing_parameters_is_rejected(yolo):
    sd = {("model.42." + k[len("detect."):] if k.startswith("detect.") else "model." + k[1:]): v for k, v in yolo.state_dict().items()}
    extra = dict(sd)
    extra["model.7.cv9.conv.weight"] = torch.zeros(1)
    with pytest.raises(KeyError, match="does not know"):
        YoloWeights(rename_upstream(extra), CPU)
    missing = {k: v for k, v in sd.items() if not k.startswith("model.5.cv4.")}
    with pytest.raises(KeyError):
        YoloWeights(rename_upstream(missing), CPU)
    with pytest.raises(KeyError, match="outside model"):
        rename_upstream(dict(sd, stray=torch.zeros(1)))


def test_archive_exported_with_fused_conv_bn(yolo):
    """conv+BN already folded by the exporter (no .bn.* keys, conv bias present) loads to the same packed weights."""
    from omniparser_b200.yolo_engine import BN_EPS
    sd = yolo.state_dict()
    fused = {}
    for k, v in sd.items():
        if ".bn." in k:
            continue
        if k.endswith(".conv.weight") and k[:-len(".conv.weight")] + ".bn.weight" in sd:
            p = k[:-len(".conv.weight")]
            s = sd[p + ".bn.weight"] / torch.sqrt(sd[p + ".bn.running_var"] + BN_EPS)
            fused[k] = v * s[:, None, None, None]
            fused[p + ".conv.bias"] = sd[p + ".bn.bias"] - sd[p + ".bn.running_mean"] * s
        else:
            fused[k] = v
    a, b = YoloWeights(fused, CPU), YoloWeights(sd, CPU)
    for k, wa in a.W.items():
        if not isinstance(wa, int):
            assert (wa.w.float() - b.W[k].w.float()).abs().max() <= 1e-3 and torch.allclose(wa.b, b.W[k].b, atol=1e-6), k


def test_detector_loader_needs_cuda(archive):
    """ref:util/yolov9.py:40-41 raises RuntimeError when CUDA is requested but unavailable; there is no CPU fallback.
    With a GPU present, loading on CUDA is covered by tests/test_boundary_gpu.py."""
    from omniparser_b200.utils import get_yolo_model
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            get_yolo_model(str(archive), device="cuda")
    with pytest.raises(RuntimeError):
        get_yolo_model(str(archive), device="cpu")


@pytest.fixture(scope="module")
def florence():
    return FS.florence_standin(0)


def test_safetensors_dir_with_remote_code_names(florence, tmp_path):
    d = tmp_path / "icon_caption_florence"
    FS.export_remote_code_dir(florence, d)
    sd, gen = caption.load_florence_state(d)
    ref = florence.state_dict()
    assert set(sd) == set(ref) | {"final_logits_bias"}
    assert all(torch.equal(sd[k], ref[k]) for k in ref)
    assert gen == {k: FS.GEN[k] for k in gen} and gen["no_repeat_ngram_size"] == 3 and gen["decoder_start_token_id"] == 2
    a, b = FlorenceWeights(sd, CPU, gen, "fp16x3"), FlorenceWeights(ref, CPU, FS.GEN, "fp16x3")
    assert torch.equal(a.E16, b.E16) and torch.equal(a.img_proj.w, b.img_proj.w)
    assert torch.equal(a.blocks[2][4]["channel_block"]["qkv"].w, b.blocks[2][4]["channel_block"]["qkv"].w)
    assert torch.equal(a.dec_layers[5]["ckv"].w, b.dec_layers[5]["ckv"].w)


def test_unknown_florence_parameters_are_rejected(florence):
    remote = FS.to_remote_code_names(florence.state_dict())
    with pytest.raises(KeyError, match="unrecognised"):
        caption.rename_remote_code(dict(remote, some_new_buffer=torch.zeros(1)))
    native = dict(florence.state_dict())
    native["model.language_model.decoder.layers.0.extra.weight"] = torch.zeros(1)
    with pytest.raises(KeyError, match="does not know"):
        FlorenceWeights(native, CPU, FS.GEN, "fp16")
    untied = dict(florence.state_dict())
    untied["lm_head.weight"] = untied["lm_head.weight"] + 1
    with pytest.raises(ValueError, match="not tied"):
        FlorenceWeights(untied, CPU, FS.GEN, "fp16")


# ---- detokeniser (SURVEY.md §8a row F6): BartTokenizer path on a synthetic byte-level BPE vocabulary -------------------
def bytes_to_unicode():
    """GPT-2 / BART byte-level BPE alphabet: printable bytes map to themselves, the rest to 256 + n."""
    bs = list(range(ord("!"), ord("~") + 1)) + list(range(0xA1, 0xAC + 1)) + list(range(0xAE, 0xFF + 1))
    cs, n = bs[:], 0
    for b in range(256):
        if b not in bs:
            bs.append(b)
            cs.append(256 + n)
            n += 1
    return dict(zip(bs, map(chr, cs)))


def _tiny_bpe_dir(d):
    b2u = bytes_to_unicode()
    vocab = {"<s>": 0, "<pad>": 1, "</s>": 2, "<unk>": 3}
    for b in range(256):
        vocab[b2u[b]] = len(vocab)
    merges = []
    for a, b in [("C", "o"), ("Co", "p"), ("Cop", "y"), (b2u[ord(" ")], "F"), (b2u[ord(" ")] + "F", "o"), ("n", "t")]:
        merges.append(f"{a} {b}")
        vocab[a + b] = len(vocab)
    vocab["<mask>"] = len(vocab)
    d.mkdir(parents=True, exist_ok=True)
    (d / "vocab.json").write_text(json.dumps(vocab))
    (d / "merges.txt").write_text("#version: 0.2\n" + "\n".join(merges) + "\n")
    return vocab


def test_processor_batch_decode_through_bart_tokenizer(tmp_path):
    vocab = _tiny_bpe_dir(tmp_path / "Florence-2-base")
    sp = bytes_to_unicode()[ord(" ")]
    assert caption.find_tokenizer_dir(str(tmp_path / "icon_caption_florence")) == tmp_path / "Florence-2-base"   # sibling lookup
    assert caption.find_tokenizer_dir(None, str(tmp_path / "Florence-2-base")) == tmp_path / "Florence-2-base"
    proc = caption.B200Florence2Processor(caption.load_tokenizer(tmp_path / "Florence-2-base"))
    ids = torch.tensor([[2, 0, vocab["Copy"], 2, 1, 1], [2, 0, vocab["Copy"], vocab[sp + "Fo"], vocab["nt"], 2]])
    assert [t.strip() for t in proc.batch_decode(ids, skip_special_tokens=True)] == ["Copy", "Copy Font"]


def test_caption_loader_refuses_id_captions_unless_opted_in(tmp_path, monkeypatch):
    from omniparser_b200.utils import get_caption_model_processor
    monkeypatch.delenv("B2P_FLORENCE_PROCESSOR", raising=False)
    monkeypatch.delenv("B2P_ALLOW_ID_CAPTIONS", raising=False)
    monkeypatch.setenv("HF_HOME", str(tmp_path / "no_cache"))
    (tmp_path / "icon_caption_florence").mkdir()
    with pytest.raises(FileNotFoundError, match="tokenizer"):
        get_caption_model_processor("florence2", str(tmp_path / "icon_caption_florence"), device="cuda")
    with pytest.raises(NotImplementedError):
        get_caption_model_processor("blip2", str(tmp_path))
