"""Query encoders on the device (SURVEY 8f rank 2 / 3) behind the reference's own seams.

The reference embeds a query on whatever torch device is around and brings it back as a Python list
(app/ml/embeddings.py:52-70 `embed_text_batch`, :94-105 `embed_query_for_images`; app/ml/retrieve.py:120-129), then the
store converts it again and copies it to its engine.  Here the three models of the request path are hand-written CUDA
behind the C ABI (csrc/encoder_kernels.cuh: tcgen05 swap-AB GEMMs + fp32 attention / LayerNorm), and their output is a
device tensor that `ResidentIndex.search` consumes directly:

    MiniLM-L6 (sentence-transformers/all-MiniLM-L6-v2)        -> TextQueryEncoder   == embed_text_batch
    CLIP ViT-B/32 text tower (openai/clip-vit-base-patch32)   -> ImageQueryEncoder  == embed_query_for_images
    ms-marco-MiniLM-L-6-v2 cross-encoder                      -> DeviceCrossEncoder == CrossEncoder.predict

and the model of the ingest side, whose output fills the image rows the scan searches:

    CLIP ViT-B/32 vision tower                                -> ImageEncoder       == embed_images_batch

Weights come from the Hugging Face modules the reference loads (`from_hf_bert` / `from_hf_clip` /
`from_hf_clip_vision` read their state_dict); tokenisation and image preprocessing stay on the host (any HF-style
tokenizer, HF's CLIPImageProcessor).  There is no torch / CPU fallback: without the library or an sm_100 device
construction raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N

KINDS = {"minilm": N.MMR_ENC_MINILM, "clip_text": N.MMR_ENC_CLIP_TEXT, "cross": N.MMR_ENC_CROSS}


def hf_bert_weights(model) -> Dict[str, torch.Tensor]:
    """state_dict of a HF BertModel / BertForSequenceClassification -> the C ABI's weight names."""
    sd = {k: v for k, v in model.state_dict().items()}
    pre = "bert." if any(k.startswith("bert.") for k in sd) else ""
    out = {
        "word_emb": sd[pre + "embeddings.word_embeddings.weight"],
        "pos_emb": sd[pre + "embeddings.position_embeddings.weight"],
        "type_emb": sd[pre + "embeddings.token_type_embeddings.weight"],
        "emb_ln_w": sd[pre + "embeddings.LayerNorm.weight"],
        "emb_ln_b": sd[pre + "embeddings.LayerNorm.bias"],
    }
    i = 0
    while f"{pre}encoder.layer.{i}.attention.self.query.weight" in sd:
        p = f"{pre}encoder.layer.{i}."
        out[f"L{i}.qkv_w"] = torch.cat([sd[p + f"attention.self.{n}.weight"] for n in ("query", "key", "value")], dim=0)
        out[f"L{i}.qkv_b"] = torch.cat([sd[p + f"attention.self.{n}.bias"] for n in ("query", "key", "value")], dim=0)
        out[f"L{i}.o_w"], out[f"L{i}.o_b"] = sd[p + "attention.output.dense.weight"], sd[p + "attention.output.dense.bias"]
        out[f"L{i}.ln1_w"], out[f"L{i}.ln1_b"] = sd[p + "attention.output.LayerNorm.weight"], sd[p + "attention.output.LayerNorm.bias"]
        out[f"L{i}.fc1_w"], out[f"L{i}.fc1_b"] = sd[p + "intermediate.dense.weight"], sd[p + "intermediate.dense.bias"]
        out[f"L{i}.fc2_w"], out[f"L{i}.fc2_b"] = sd[p + "output.dense.weight"], sd[p + "output.dense.bias"]
        out[f"L{i}.ln2_w"], out[f"L{i}.ln2_b"] = sd[p + "output.LayerNorm.weight"], sd[p + "output.LayerNorm.bias"]
        i += 1
    if "classifier.weight" in sd:
        out["pooler_w"], out["pooler_b"] = sd[pre + "pooler.dense.weight"], sd[pre + "pooler.dense.bias"]
        out["cls_w"], out["cls_b"] = sd["classifier.weight"].reshape(-1), sd["classifier.bias"].reshape(-1)
    return out


def hf_clip_text_weights(model) -> Dict[str, torch.Tensor]:
    """state_dict of a HF CLIPModel / CLIPTextModelWithProjection -> the C ABI's weight names (text tower only)."""
    sd = model.state_dict()
    t = "text_model."
    out = {
        "word_emb": sd[t + "embeddings.token_embedding.weight"],
        "pos_emb": sd[t + "embeddings.position_embedding.weight"],
        "final_ln_w": sd[t + "final_layer_norm.weight"],
        "final_ln_b": sd[t + "final_layer_norm.bias"],
        "proj_w": sd["text_projection.weight"],
    }
    i = 0
    while f"{t}encoder.layers.{i}.self_attn.q_proj.weight" in sd:
        p = f"{t}encoder.layers.{i}."
        out[f"L{i}.qkv_w"] = torch.cat([sd[p + f"self_attn.{n}_proj.weight"] for n in ("q", "k", "v")], dim=0)
        out[f"L{i}.qkv_b"] = torch.cat([sd[p + f"self_attn.{n}_proj.bias"] for n in ("q", "k", "v")], dim=0)
        out[f"L{i}.o_w"], out[f"L{i}.o_b"] = sd[p + "self_attn.out_proj.weight"], sd[p + "self_attn.out_proj.bias"]
        out[f"L{i}.ln1_w"], out[f"L{i}.ln1_b"] = sd[p + "layer_norm1.weight"], sd[p + "layer_norm1.bias"]
        out[f"L{i}.fc1_w"], out[f"L{i}.fc1_b"] = sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"]
        out[f"L{i}.fc2_w"], out[f"L{i}.fc2_b"] = sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"]
        out[f"L{i}.ln2_w"], out[f"L{i}.ln2_b"] = sd[p + "layer_norm2.weight"], sd[p + "layer_norm2.bias"]
        i += 1
    return out


def hf_clip_vision_weights(model) -> Dict[str, torch.Tensor]:
    """state_dict of a HF CLIPModel / CLIPVisionModelWithProjection -> the C ABI's weight names (vision tower only).
    The patch embedding's Conv2d weight [H, C, P, P] becomes the GEMM weight [H, C * P * P] ((c, kh, kw) column order)."""
    sd = model.state_dict()
    v = "vision_model."
    pw = sd[v + "embeddings.patch_embedding.weight"]
    out = {
        "patch_w": pw.reshape(pw.shape[0], -1),
        "cls_emb": sd[v + "embeddings.class_embedding"],
        "pos_emb": sd[v + "embeddings.position_embedding.weight"],
        "pre_ln_w": sd[v + "pre_layrnorm.weight"],
        "pre_ln_b": sd[v + "pre_layrnorm.bias"],
        "final_ln_w": sd[v + "post_layernorm.weight"],
        "final_ln_b": sd[v + "post_layernorm.bias"],
        "proj_w": sd["visual_projection.weight"],
    }
    i = 0
    while f"{v}encoder.layers.{i}.self_attn.q_proj.weight" in sd:
        p = f"{v}encoder.layers.{i}."
        out[f"L{i}.qkv_w"] = torch.cat([sd[p + f"self_attn.{n}_proj.weight"] for n in ("q", "k", "v")], dim=0)
        out[f"L{i}.qkv_b"] = torch.cat([sd[p + f"self_attn.{n}_proj.bias"] for n in ("q", "k", "v")], dim=0)
        out[f"L{i}.o_w"], out[f"L{i}.o_b"] = sd[p + "self_attn.out_proj.weight"], sd[p + "self_attn.out_proj.bias"]
        out[f"L{i}.ln1_w"], out[f"L{i}.ln1_b"] = sd[p + "layer_norm1.weight"], sd[p + "layer_norm1.bias"]
        out[f"L{i}.fc1_w"], out[f"L{i}.fc1_b"] = sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"]
        out[f"L{i}.fc2_w"], out[f"L{i}.fc2_b"] = sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"]
        out[f"L{i}.ln2_w"], out[f"L{i}.ln2_b"] = sd[p + "layer_norm2.weight"], sd[p + "layer_norm2.bias"]
        i += 1
    return out


def _check_supported(cfg, acts) -> None:
    """The kernels implement erf-GELU (BERT), quick-GELU (CLIP) and absolute position embeddings only: any other model
    would run with the wrong math and no error."""
    act = getattr(cfg, "hidden_act", None)
    if not isinstance(act, str) or act not in acts:
        raise ValueError(f"hidden_act {act!r} is not supported by the device encoders (expected {' or '.join(sorted(acts))})")
    pos = getattr(cfg, "position_embedding_type", "absolute")
    if pos != "absolute":
        raise ValueError(f"position_embedding_type {pos!r} is not supported by the device encoders (expected 'absolute')")


class DeviceEncoder:
    """One transformer (MiniLM / CLIP text / cross-encoder / CLIP vision) resident on a B200, driven through mmr_encoder_*.
    The vision tower is built with `DeviceEncoder.vision(...)` or `from_hf_clip_vision` and run with `forward_pixels`."""

    def __init__(self, kind: str, *, vocab_size: int = 0, hidden: int, layers: int, heads: int, intermediate: int,
                 max_positions: int = 0, type_vocab: int = 2, proj_dim: int = 0, eos_token_id: int = 0, ln_eps: float = 1e-12,
                 image_size: int = 0, patch_size: int = 0, channels: int = 3, device: Any = "cuda:0") -> None:
        lib = N.lib()
        if not torch.cuda.is_available():
            raise N.NativeError("no CUDA device: the device encoders have no CPU fallback")
        self.kind = kind
        self.device = torch.device(device)
        self._handle = C.c_void_p()
        if kind == "clip_vision":
            self.cfg = N.VisionConfig(hidden, layers, heads, intermediate, image_size, patch_size, channels, proj_dim, ln_eps)
            N.check(lib.mmr_encoder_create_vision(self.device.index or 0, C.byref(self.cfg), C.byref(self._handle)))
        else:
            self.cfg = N.EncoderConfig(KINDS[kind], vocab_size, hidden, layers, heads, intermediate, max_positions, type_vocab,
                                       proj_dim, eos_token_id, ln_eps)
            N.check(lib.mmr_encoder_create(self.device.index or 0, C.byref(self.cfg), C.byref(self._handle)))
        self.out_dim = int(lib.mmr_encoder_out_dim(self._handle))
        self._loaded: List[str] = []

    # -- construction from the modules the reference loads ----------------------------------------
    @classmethod
    def from_hf_bert(cls, model, device: Any = "cuda:0", cross: Optional[bool] = None) -> "DeviceEncoder":
        cfg = model.config
        _check_supported(cfg, {"gelu"})
        weights = hf_bert_weights(model)
        cross = ("cls_w" in weights) if cross is None else cross
        enc = cls("cross" if cross else "minilm", vocab_size=cfg.vocab_size, hidden=cfg.hidden_size,
                  layers=cfg.num_hidden_layers, heads=cfg.num_attention_heads, intermediate=cfg.intermediate_size,
                  max_positions=cfg.max_position_embeddings, type_vocab=cfg.type_vocab_size, ln_eps=cfg.layer_norm_eps,
                  device=device)
        enc.load(weights)
        return enc

    @classmethod
    def from_hf_clip(cls, model, device: Any = "cuda:0") -> "DeviceEncoder":
        cfg = getattr(model.config, "text_config", model.config)
        _check_supported(cfg, {"quick_gelu"})
        weights = hf_clip_text_weights(model)
        enc = cls("clip_text", vocab_size=cfg.vocab_size, hidden=cfg.hidden_size, layers=cfg.num_hidden_layers,
                  heads=cfg.num_attention_heads, intermediate=cfg.intermediate_size,
                  max_positions=cfg.max_position_embeddings, proj_dim=int(weights["proj_w"].shape[0]),
                  eos_token_id=int(cfg.eos_token_id), ln_eps=cfg.layer_norm_eps, device=device)
        enc.load(weights)
        return enc

    @classmethod
    def from_hf_clip_vision(cls, model, device: Any = "cuda:0") -> "DeviceEncoder":
        """CLIP vision tower of a HF CLIPModel or CLIPVisionModelWithProjection (the model `embed_images_batch` runs)."""
        cfg = getattr(model.config, "vision_config", model.config)
        _check_supported(cfg, {"quick_gelu"})
        weights = hf_clip_vision_weights(model)
        enc = cls("clip_vision", hidden=cfg.hidden_size, layers=cfg.num_hidden_layers, heads=cfg.num_attention_heads,
                  intermediate=cfg.intermediate_size, proj_dim=int(weights["proj_w"].shape[0]), ln_eps=cfg.layer_norm_eps,
                  image_size=cfg.image_size, patch_size=cfg.patch_size, channels=cfg.num_channels, device=device)
        enc.load(weights)
        return enc

    def load(self, weights: Dict[str, torch.Tensor]) -> None:
        lib = N.lib()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            for name, w in weights.items():
                t = w.detach().to(device=self.device, dtype=torch.float32).contiguous()
                N.check(lib.mmr_encoder_set_weight(self._handle, name.encode(), t.data_ptr(), t.numel(), stream))
                self._loaded.append(name)
            torch.cuda.synchronize(self.device)

    # -- forward ----------------------------------------------------------------------------------
    def forward_ids(self, input_ids, attention_mask=None, token_type_ids=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Token ids [B, S] (host) -> [B, out_dim] fp32 on the device (unit-norm embeddings; [B] logits for "cross")."""
        ids = np.ascontiguousarray(np.atleast_2d(np.asarray(input_ids)), dtype=np.int32)
        b, s = ids.shape
        mask = None if attention_mask is None else np.ascontiguousarray(np.atleast_2d(np.asarray(attention_mask)), dtype=np.int32)
        types = None if token_type_ids is None else np.ascontiguousarray(np.atleast_2d(np.asarray(token_type_ids)), dtype=np.int32)
        for name, a in (("attention_mask", mask), ("token_type_ids", types)):
            if a is not None and a.shape != ids.shape:
                raise ValueError(f"{name} must have the shape of input_ids")
        if out is None:
            out = torch.empty((b, self.out_dim) if self.kind != "cross" else (b,), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.lib().mmr_encoder_forward(self._handle, ids.ctypes.data, None if mask is None else mask.ctypes.data,
                                                None if types is None else types.ctypes.data, b, s, out.data_ptr(),
                                                torch.cuda.current_stream(self.device).cuda_stream))
        return out

    def forward_pixels(self, pixel_values: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Pixel values [B, C, S, S] (what CLIPImageProcessor returns; any device / dtype) -> [B, proj] fp32 unit-norm image
        embeddings on the device."""
        if self.kind != "clip_vision":
            raise ValueError(f"forward_pixels needs a CLIP vision encoder, not {self.kind!r}")
        c = self.cfg
        px = torch.as_tensor(pixel_values).to(device=self.device, dtype=torch.float32).contiguous()
        if px.dim() != 4 or tuple(px.shape[1:]) != (c.channels, c.image_size, c.image_size):
            raise ValueError(f"pixel_values must be [B, {c.channels}, {c.image_size}, {c.image_size}], got {tuple(px.shape)}")
        b = px.shape[0]
        if out is None:
            out = torch.empty((b, self.out_dim), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.lib().mmr_encoder_forward_pixels(self._handle, px.data_ptr(), b, out.data_ptr(),
                                                       torch.cuda.current_stream(self.device).cuda_stream))
        return out

    def close(self) -> None:
        if self._handle:
            N.lib().mmr_encoder_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _tokenize(tokenizer: Callable, texts, **kw) -> Tuple[np.ndarray, Optional[np.ndarray], Optional[np.ndarray]]:
    enc = tokenizer(texts, padding=True, truncation=True, return_tensors="np", **kw)
    get = enc.get if hasattr(enc, "get") else (lambda k, d=None: getattr(enc, k, d))
    return np.asarray(get("input_ids")), get("attention_mask"), get("token_type_ids")


class TextQueryEncoder:
    """`embed_text_batch` (app/ml/embeddings.py:52-70) with MiniLM on the device: texts -> unit-norm f32 [n, 384]."""

    def __init__(self, tokenizer: Callable, encoder: DeviceEncoder, max_length: int = 256) -> None:
        self.tokenizer, self.encoder, self.max_length = tokenizer, encoder, max_length

    def encode_device(self, texts: Sequence[str]) -> torch.Tensor:
        ids, mask, types = _tokenize(self.tokenizer, list(texts), max_length=self.max_length)
        return self.encoder.forward_ids(ids, mask, types)

    def __call__(self, texts: Sequence[str], batch_size: int = 32) -> np.ndarray:
        if not texts:
            return np.empty((0, self.encoder.out_dim), dtype=np.float32)
        return self.encode_device(texts).cpu().numpy()


class ImageQueryEncoder:
    """`embed_query_for_images` (app/ml/embeddings.py:94-105) with the CLIP text tower on the device."""

    def __init__(self, tokenizer: Callable, encoder: DeviceEncoder, max_length: int = 77) -> None:
        self.tokenizer, self.encoder, self.max_length = tokenizer, encoder, max_length

    def encode_device(self, queries: Sequence[str]) -> torch.Tensor:
        ids, mask, _ = _tokenize(self.tokenizer, list(queries), max_length=self.max_length)
        out = self.encoder.forward_ids(ids, mask)
        blank = [i for i, q in enumerate(queries) if not q.strip()]
        if blank:                                  # `if not query.strip(): return zeros(512)` (:96-97)
            out[torch.as_tensor(blank, device=out.device)] = 0.0
        return out

    def __call__(self, query: str) -> np.ndarray:
        if not query.strip():
            return np.zeros((self.encoder.out_dim,), dtype=np.float32)
        return self.encode_device([query])[0].cpu().numpy()


class DeviceCrossEncoder:
    """`CrossEncoder.predict(pairs)` (app/ml/retrieve.py:146) on the device: raw logits, one per (query, passage) pair
    (ms-marco-MiniLM-L-6-v2 ships `Identity` as its activation).  Pairs from several requests can share one forward pass."""

    def __init__(self, tokenizer: Callable, encoder: DeviceEncoder, max_length: int = 512) -> None:
        self.tokenizer, self.encoder, self.max_length = tokenizer, encoder, max_length

    def predict_device(self, pairs: Sequence[Tuple[str, str]]) -> torch.Tensor:
        enc = self.tokenizer([p[0] for p in pairs], [p[1] for p in pairs], padding=True, truncation=True,
                             max_length=self.max_length, return_tensors="np")
        return self.encoder.forward_ids(enc["input_ids"], enc.get("attention_mask"), enc.get("token_type_ids"))

    def predict(self, pairs: Sequence[Tuple[str, str]]) -> np.ndarray:
        if not pairs:
            return np.empty((0,), dtype=np.float32)
        return self.predict_device(pairs).cpu().numpy()


class ImageEncoder:
    """`embed_images_batch` (app/ml/embeddings.py:73-91) with the CLIP vision tower on the device: images -> unit-norm f32
    [n, proj].  `processor` is the caller's HF CLIPImageProcessor (resize, centre crop, normalise stay on the host, as
    tokenisation does for the text encoders); any callable returning {"pixel_values": [n, C, S, S]} works."""

    def __init__(self, processor: Callable, encoder: DeviceEncoder) -> None:
        self.processor, self.encoder = processor, encoder

    def encode_device(self, images: Sequence[Any]) -> torch.Tensor:
        px = self.processor(images=list(images), return_tensors="pt")["pixel_values"]
        return self.encoder.forward_pixels(px)

    def __call__(self, images: Sequence[Any], batch_size: int = 32) -> np.ndarray:
        images = list(images)
        if not images:
            return np.empty((0, self.encoder.out_dim), dtype=np.float32)
        parts = [self.encode_device(images[i:i + batch_size]).cpu().numpy() for i in range(0, len(images), batch_size)]
        return np.concatenate(parts, axis=0)


__all__ = ["DeviceEncoder", "TextQueryEncoder", "ImageQueryEncoder", "ImageEncoder", "DeviceCrossEncoder", "hf_bert_weights",
           "hf_clip_text_weights", "hf_clip_vision_weights"]
