#!/usr/bin/env python
"""Outputs of the text-side encoders from two builds of the library, compared bit for bit.

    python benchmarks/encoder_outputs_ab.py dump OUT.npz [TREE]     # the package (binding + built library) of TREE,
                                                                    # default: this checkout
    python benchmarks/encoder_outputs_ab.py compare A.npz B.npz

Seeded HF modules of the three shipped text-side models (MiniLM-L6, CLIP text tower, ms-marco cross-encoder; linear weights
rounded to bf16 values) at the shapes the serving path runs: MiniLM 1 x 16 and 128 x 16, CLIP 40 x 77, cross-encoder
8 x 128 and 72 x 64.  A change that must not alter these encoders dumps with the parent's library and with its own."""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _round(model):
    with torch.no_grad():
        for name, p in model.named_parameters():
            if p.dim() == 2 and "embedding" not in name.lower():
                p.mul_(2.0)
                p.copy_(p.to(torch.bfloat16).to(torch.float32))
            elif p.dim() == 1 and "bias" in name:
                p.normal_(0.0, 0.05)
            elif p.dim() == 1 and "weight" in name:
                p.normal_(1.0, 0.1)
    return model.eval()


def dump(path, tree=ROOT):
    sys.path.insert(0, os.path.abspath(tree))
    from transformers import BertConfig, BertForSequenceClassification, BertModel, CLIPTextConfig, CLIPTextModelWithProjection
    enc_mod = importlib.import_module("multimodal-rag-for-image-text-search_b200.encoders")
    bcfg = dict(vocab_size=30522, hidden_size=384, num_hidden_layers=6, num_attention_heads=12, intermediate_size=1536)
    torch.manual_seed(0)
    minilm = enc_mod.DeviceEncoder.from_hf_bert(_round(BertModel(BertConfig(**bcfg), add_pooling_layer=False)))
    torch.manual_seed(1)
    clip = enc_mod.DeviceEncoder.from_hf_clip(_round(CLIPTextModelWithProjection(CLIPTextConfig())))
    torch.manual_seed(2)
    cross = enc_mod.DeviceEncoder.from_hf_bert(_round(BertForSequenceClassification(BertConfig(**bcfg, num_labels=1))))
    out = {}
    for name, enc, b, s in (("minilm_1x16", minilm, 1, 16), ("minilm_128x16", minilm, 128, 16), ("clip_40x77", clip, 40, 77),
                            ("cross_8x128", cross, 8, 128), ("cross_72x64", cross, 72, 64)):
        rng = np.random.default_rng(b * 1000 + s)
        ids = rng.integers(1000, 30000, size=(b, s))
        lens = rng.integers(max(2, s // 3), s + 1, size=b)
        lens[0] = s
        mask = (np.arange(s)[None, :] < lens[:, None]).astype(np.int64)
        if name.startswith("clip"):
            ids[:, 0] = 49406
            for i in range(b):
                ids[i, lens[i] - 1:] = 49407
        types = (np.arange(s)[None, :] >= lens[:, None] // 3).astype(np.int64) * mask if name.startswith("cross") else None
        out[name] = enc.forward_ids(ids, mask, types).cpu().numpy()
    np.savez(path, **out)
    print("dumped", sorted(out), "from", importlib.import_module("multimodal-rag-for-image-text-search_b200._native").LIB_PATH)


def compare(a_path, b_path):
    a, b = np.load(a_path), np.load(b_path)
    ok = sorted(a.files) == sorted(b.files)
    for k in sorted(a.files):
        same = a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes()
        diff = float(np.abs(a[k].astype(np.float64) - b[k]).max()) if a[k].shape == b[k].shape else float("nan")
        print(f"{k:16s} bit-identical={same} max|diff|={diff:g}")
        ok &= same
    print("ALL BIT-IDENTICAL" if ok else "OUTPUTS DIFFER")
    return 0 if ok else 1


if __name__ == "__main__":
    if sys.argv[1] == "dump":
        dump(*sys.argv[2:4])
    else:
        sys.exit(compare(sys.argv[2], sys.argv[3]))
