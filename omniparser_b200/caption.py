"""Drop-in ``{'model', 'processor'}`` pair for the Florence-2 caption branch of
``get_caption_model_processor`` (ref:util/utils.py:48-69) on the B200 kernels.

Contract kept (SURVEY.md §8b): ``model.config.model_type`` / ``model.config.name_or_path`` (contains 'florence'),
``model.device``, ``model.generate(input_ids=, pixel_values=, max_new_tokens=20, num_beams=1, do_sample=False)`` ->
``LongTensor[K, T]``; ``processor(images=, text=, return_tensors="pt"[, do_resize=False])`` (HF default True: 768x768
bicubic crops, the reference's CPU branch) -> object with
``.to(device=, dtype=)`` and keys ``input_ids`` / ``pixel_values``; ``processor.batch_decode(ids,
skip_special_tokens=True)``.

The processor hands the 64x64 crops to the model as raw u8 HWC (its ``.to(dtype=float16)`` leaves integer tensors
alone, exactly like ``BatchFeature.to``); rescale + ImageNet normalisation is folded into the first kernel's lookup
table.  Float ``pixel_values`` (K,3,64,64) are also accepted and mapped back to the u8 they came from.
"""
from __future__ import annotations

import json
import threading
from pathlib import Path
from types import SimpleNamespace
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from .florence_engine import IMAGENET_MEAN, IMAGENET_STD, FlorencePlan, FlorenceWeights

# "<s>What does the image describe?</s>" in the BART vocabulary (hf:models/florence2/processing_florence2.py:81 maps
# "<CAPTION>" to this question, ref:util/utils.py:109-110)
CAPTION_PROMPT_IDS = [0, 2264, 473, 5, 2274, 6190, 116, 2]
DEFAULT_GEN = dict(forced_bos_token_id=0, forced_eos_token_id=2, no_repeat_ngram_size=3, eos_token_id=2, pad_token_id=1,
                   bos_token_id=0, decoder_start_token_id=2)
BUCKET = 32
BUCKET_768 = 16      # 768x768 mode: 36864 stage-0 tokens per crop -> small chunks (activations ~1.5 GB per crop)


class _Batch(dict):
    """Minimal BatchFeature: attribute access + ``.to`` that only casts floating tensors."""

    def to(self, device=None, dtype=None, **_):
        out = _Batch()
        for k, v in self.items():
            if torch.is_tensor(v):
                v = v.to(device=device, dtype=dtype) if (dtype is not None and v.is_floating_point()) else v.to(device=device)
            out[k] = v
        return out

    __getattr__ = dict.__getitem__


class B200Florence2Processor:
    def __init__(self, tokenizer=None, prompt_ids: Sequence[int] = CAPTION_PROMPT_IDS):
        self.tokenizer = tokenizer
        self.prompt_ids = list(prompt_ids)

    def __call__(self, images=None, text=None, return_tensors="pt", do_resize=True, **kw):
        # Default do_resize=True as in HF's CLIPImageProcessor (what the reference gets when it omits the argument).
        # do_resize=False: the reference's CUDA branch (ref:util/utils.py:121), crops go in as 64x64.
        # do_resize=True (HF default): its CPU branch (:123): CLIP image processor bicubic resize to 768x768 on the u8
        # image (resample=3), done here with Pillow exactly as the HF processor does; the model sees 768x768 u8.
        arr = []
        for im in images:
            pil = im if hasattr(im, "convert") else __import__("PIL.Image", fromlist=["Image"]).fromarray(np.asarray(im, dtype=np.uint8))
            pil = pil.convert("RGB")
            if do_resize:
                from PIL import Image as _I
                pil = pil.resize((768, 768), _I.Resampling.BICUBIC)
            a = np.asarray(pil, dtype=np.uint8)
            if a.shape not in ((64, 64, 3), (768, 768, 3)):
                raise ValueError(f"expected 64x64 RGB crops (or do_resize=True), got {a.shape}")
            arr.append(a)
        side = arr[0].shape[0] if arr else 64
        px = torch.from_numpy(np.stack(arr)) if arr else torch.zeros((0, side, side, 3), dtype=torch.uint8)
        ids = torch.tensor([self.prompt_ids] * len(arr), dtype=torch.long).reshape(len(arr), len(self.prompt_ids))
        return _Batch(input_ids=ids, pixel_values=px)

    def batch_decode(self, ids, skip_special_tokens=True, **kw) -> List[str]:
        ids = ids.tolist() if torch.is_tensor(ids) else ids
        if self.tokenizer is not None:
            return self.tokenizer.batch_decode(ids, skip_special_tokens=skip_special_tokens, **kw)
        special = {0, 1, 2} if skip_special_tokens else set()
        # no BART vocab/merges in this environment: ids are the pinned parity target, strings are id tags
        return [" ".join(f"<{t}>" for t in row if t not in special) for row in ids]


class B200Florence2Model:
    def __init__(self, state_dict: Dict[str, torch.Tensor], device, gen_cfg: Optional[dict] = None,
                 precision: str = "fp16x3", name_or_path: str = "b200/florence2", use_graph: bool = True):
        self.device = torch.device(device)
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise RuntimeError("B200 Florence-2 needs a CUDA device; there is no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.config = SimpleNamespace(model_type="florence2", name_or_path=name_or_path)
        self.gen = dict(DEFAULT_GEN)
        if gen_cfg:
            self.gen.update({k: v for k, v in gen_cfg.items() if k in self.gen or k.endswith("_token_id") or k == "no_repeat_ngram_size"})
        with torch.cuda.device(self.device):
            self.weights = FlorenceWeights(state_dict, self.device, self.gen, precision)
        self.use_graph = use_graph
        self._plans: Dict[tuple, FlorencePlan] = {}
        self._plan_lock = threading.Lock()
        self._lock = threading.RLock()   # generate() uses plan instance 0: one call at a time per handle (see detector._lock)
        inv = np.zeros((3, 256), np.float32)
        for c in range(3):
            inv[c] = (np.arange(256, dtype=np.float32) * np.float32(1 / 255.0) - np.float32(IMAGENET_MEAN[c])) / np.float32(IMAGENET_STD[c])
        self._lut_cpu = torch.from_numpy(inv)

    def to(self, device):
        return self

    def eval(self):
        return self

    def plan_for(self, n: int, max_new_tokens: int, prompt_ids: Sequence[int], size: int = 64, instance: int = 0) -> FlorencePlan:
        """Launch plan (buffers + CUDA graphs) for up to ``n`` crops.  Plans of different ``instance`` share nothing
        mutable, so the pipeline can caption two batches concurrently on two streams."""
        if size == 64:
            K = max(BUCKET, ((n + BUCKET - 1) // BUCKET) * BUCKET)
        else:
            K = BUCKET_768
        key = (K, max_new_tokens, tuple(prompt_ids), size, instance)
        with self._plan_lock:
            if key not in self._plans:
                with torch.cuda.device(self.device):
                    self._plans[key] = FlorencePlan(self.weights, K, max_new_tokens, list(prompt_ids), self.use_graph, size, instance)
            return self._plans[key]

    def plan_ready(self, n: int, max_new_tokens: int, prompt_ids: Sequence[int], size: int = 64, instance: int = 0) -> bool:
        K = max(BUCKET, ((n + BUCKET - 1) // BUCKET) * BUCKET) if size == 64 else BUCKET_768
        p = self._plans.get((K, max_new_tokens, tuple(prompt_ids), size, instance))
        return p is not None and (p.warmed or not p.use_graph)

    @torch.inference_mode()
    def warm_plan(self, n: int, max_new_tokens: int, prompt_ids: Sequence[int], size: int = 64, instance: int = 0, stream=None):
        """Construct the plan for this crop-count bucket and capture its graphs on scratch inputs."""
        with torch.cuda.device(self.device), torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream()):
            self.plan_for(n, max_new_tokens, prompt_ids, size, instance).warm()

    def _to_u8(self, pixel_values: torch.Tensor) -> torch.Tensor:
        if pixel_values.dtype == torch.uint8:
            if pixel_values.dim() == 4 and pixel_values.shape[-1] == 3:
                return pixel_values
            raise ValueError("uint8 pixel_values must be [K,S,S,3]")
        x = pixel_values.float().cpu()   # [K,3,64,64] normalised
        mean = torch.tensor(IMAGENET_MEAN).view(1, 3, 1, 1)
        std = torch.tensor(IMAGENET_STD).view(1, 3, 1, 1)
        return ((x * std + mean) * 255.0).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()

    @torch.inference_mode()
    def generate_from_device_crops(self, plan: FlorencePlan, n: int, sync_every: int = 4, from_resized: bool = False) -> torch.Tensor:
        """Crops already in ``plan.crops[:n]`` (device; ``plan.crops_in`` if from_resized).  Returns LongTensor [n, T] on
        the device, HF layout ``[decoder_start, tokens..., eos, pad...]`` truncated where every row has finished."""
        with plan.lock, torch.cuda.device(self.device):   # a plan instance (buffers + graphs) serves one generation at a time
            if n < plan.K:
                (plan.crops_in if from_resized else plan.crops)[n:].zero_()
            plan.encode(from_resized)
            plan.reset_decode(n)
            steps = 0
            while steps < plan.T:
                plan.decode_step(forced=plan.step_is_forced(steps))
                steps += 1
                if steps % sync_every == 0 and steps < plan.T and plan.unfinished() == 0:
                    break
            plan.join()
            # exact stop length: first step after which no row was unfinished
            seq = plan.seq[:n, :steps + 1]
            if steps > 1:
                done_at = self._first_all_finished(seq)
                if done_at is not None:
                    seq = seq[:, :done_at + 1]
            return seq.long()

    def _first_all_finished(self, seq: torch.Tensor):
        """HF stops right after the first step at which every row has produced EOS (hf:generation/utils.py:2797-2805)."""
        eos = self.gen["eos_token_id"]
        if seq.shape[0] == 0:
            return None
        hit = (seq[:, 1:] == eos)
        first = torch.where(hit.any(1), hit.float().argmax(1) + 1, torch.full((seq.shape[0],), seq.shape[1], device=seq.device))
        last = int(first.max().item())
        return last if last < seq.shape[1] else None

    @torch.inference_mode()
    def generate(self, input_ids=None, pixel_values=None, max_new_tokens=20, num_beams=1, do_sample=False, **kw):
        """ref:util/utils.py:125."""
        if num_beams != 1 or do_sample:
            raise NotImplementedError("only greedy decoding (num_beams=1, do_sample=False) is on the hot path")
        with self._lock:
            return self._generate(input_ids, pixel_values, max_new_tokens)

    def _generate(self, input_ids, pixel_values, max_new_tokens):
        u8 = self._to_u8(pixel_values)
        n = u8.shape[0]
        if n == 0:
            return torch.zeros((0, 1), dtype=torch.long, device=self.device)
        prompt = input_ids[0].tolist() if input_ids is not None else CAPTION_PROMPT_IDS
        if input_ids is not None and not bool((input_ids == input_ids[0:1]).all()):
            raise NotImplementedError("all rows must share one prompt (the reference passes [prompt]*len(batch))")
        side = int(u8.shape[1])
        if side == 64:
            plan = self.plan_for(n, max_new_tokens, prompt)
            plan.crops[:n].copy_(u8.to(self.device, non_blocking=True))
            return self.generate_from_device_crops(plan, n)
        if side != 768:
            raise ValueError("pixel_values must be 64x64 (do_resize=False) or 768x768 (processor default)")
        return self.generate_chunked(u8, max_new_tokens, prompt, from_resized=True)

    @torch.inference_mode()
    def generate_chunked(self, crops_u8: torch.Tensor, max_new_tokens: int, prompt, from_resized: bool) -> torch.Tensor:
        """768x768 mode: run the crops through the (small-K) plan chunk by chunk; HF pads the shorter chunks with pad."""
        n = crops_u8.shape[0]
        plan = self.plan_for(n, max_new_tokens, prompt, 768)
        outs = []
        for c0 in range(0, n, plan.K):
            m = min(plan.K, n - c0)
            dst = plan.crops_in if from_resized else plan.crops
            dst[:m].copy_(crops_u8[c0:c0 + m].to(self.device, non_blocking=True))
            outs.append(self.generate_from_device_crops(plan, m, from_resized=from_resized).clone())
        width = max(o.shape[1] for o in outs)
        pad = self.gen["pad_token_id"]
        outs = [torch.nn.functional.pad(o, (0, width - o.shape[1]), value=pad) for o in outs]
        return torch.cat(outs, 0)


def load_florence_state(path: str | Path):
    """Read ``model.safetensors`` (+ ``generation_config.json`` / ``config.json``) from a local directory
    (ref:README.md:45-46; what ``AutoModelForCausalLM.from_pretrained`` reads at ref:util/utils.py:66-68)."""
    from safetensors.torch import load_file

    p = Path(path)
    if not (p / "model.safetensors").is_file():
        raise FileNotFoundError(f"{p}/model.safetensors not found (no network here: pass a local weights directory)")
    sd = load_file(str(p / "model.safetensors"))
    gen = {}
    for name in ("generation_config.json", "config.json"):
        f = p / name
        if f.is_file():
            cfg = json.loads(f.read_text())
            for src in (cfg, cfg.get("text_config") or {}):
                for k in DEFAULT_GEN:
                    if k in src and src[k] is not None and k not in gen:
                        gen[k] = src[k]
    return rename_remote_code(sd), gen


_VT_LEAF = (   # microsoft/Florence-2 remote-code DaViT leaf names -> transformers-native names
    (".window_attn.norm.", ".norm1."), (".channel_attn.norm.", ".norm1."), (".ffn.norm.", ".norm2."),
    (".window_attn.fn.", ".window_attn."), (".channel_attn.fn.", ".channel_attn."),
    (".conv1.fn.dw.", ".conv1."), (".conv2.fn.dw.", ".conv2."),
    (".ffn.fn.net.fc1.", ".ffn.fc1."), (".ffn.fn.net.fc2.", ".ffn.fc2."),
)


def rename_remote_code(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """microsoft/Florence-2 remote-code parameter names -> transformers-native names (SURVEY.md §8c; recalled layout,
    exercised by exporting the seeded stand-in under those names: tests/test_loaders_cpu.py).  Native names pass
    through.  Every key must be recognised: an unknown key raises instead of loading as a silently different network."""
    if any(k.startswith("model.vision_tower.") for k in sd):
        return dict(sd)
    out = {}
    for k, v in sd.items():
        if k.startswith("vision_tower.convs."):
            nk = "model." + k.replace(".proj.weight", ".conv.weight").replace(".proj.bias", ".conv.bias")
        elif k.startswith("vision_tower.blocks."):
            nk = "model." + k
            for a, b in _VT_LEAF:
                nk = nk.replace(a, b)
        elif k == "image_projection":
            nk, v = "model.multi_modal_projector.image_projection.weight", v.t().contiguous()   # raw (1024, 768) Parameter
        elif k.startswith("image_proj_norm."):
            nk = "model.multi_modal_projector." + k
        elif k.startswith("image_pos_embed."):
            nk = "model.multi_modal_projector.image_position_embed." + k[len("image_pos_embed."):]
        elif k.startswith("visual_temporal_embed."):
            nk = "model.multi_modal_projector." + k
        elif k.startswith("language_model.model."):
            nk = "model.language_model." + k[len("language_model.model."):]
        elif k == "language_model.lm_head.weight":
            nk = "lm_head.weight"
        elif k == "language_model.final_logits_bias":
            nk = "final_logits_bias"
        else:
            raise KeyError(f"unrecognised Florence-2 checkpoint parameter: {k}")
        if nk in out:
            raise KeyError(f"two checkpoint parameters map to {nk}")
        out[nk] = v
    return out


def find_tokenizer_dir(model_name_or_path=None, tokenizer_path=None) -> Optional[Path]:
    """Where the BART byte-level BPE files of the Florence-2 processor can be found offline.  The reference loads the
    processor from the hub id ``microsoft/Florence-2-base`` (ref:util/utils.py:64); ``weights/icon_caption_florence``
    itself holds only config + safetensors.  Search order: explicit ``tokenizer_path`` / $B2P_FLORENCE_PROCESSOR, the
    weights directory, a sibling ``Florence-2-base`` directory, the local Hugging Face hub cache."""
    import os
    cands = []
    for c in (tokenizer_path, os.environ.get("B2P_FLORENCE_PROCESSOR"), model_name_or_path):
        if c:
            cands.append(Path(c))
    if model_name_or_path:
        cands.append(Path(model_name_or_path).parent / "Florence-2-base")
    hub = Path(os.environ.get("HF_HOME", Path.home() / ".cache" / "huggingface")) / "hub" / "models--microsoft--Florence-2-base" / "snapshots"
    try:
        if hub.is_dir():
            cands.extend(sorted(hub.iterdir(), reverse=True))
    except PermissionError:   # a cache this user cannot read holds nothing for it
        pass
    for c in cands:
        if (c / "tokenizer.json").is_file() or ((c / "vocab.json").is_file() and (c / "merges.txt").is_file()):
            return c
    return None


class _FastTokenizer:
    """``tokenizer.json`` through the `tokenizers` library (the added Florence-2 tokens live in that file)."""

    def __init__(self, path: Path):
        from tokenizers import Tokenizer
        self.tk = Tokenizer.from_file(str(path))

    def batch_decode(self, ids, skip_special_tokens=True, **kw):
        return self.tk.decode_batch([list(map(int, r)) for r in ids], skip_special_tokens=skip_special_tokens)


def load_tokenizer(d: Path):
    """BART byte-level BPE detokeniser for ``processor.batch_decode`` (ref:util/utils.py:128)."""
    d = Path(d)
    if (d / "tokenizer.json").is_file():
        return _FastTokenizer(d / "tokenizer.json")
    from transformers import BartTokenizer
    vocab = json.loads((d / "vocab.json").read_text())
    merges = [tuple(ln.split(" ")) for ln in (d / "merges.txt").read_text().splitlines() if ln and not ln.startswith("#version")]
    return BartTokenizer(vocab=vocab, merges=merges)
