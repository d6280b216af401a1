#!/usr/bin/env python
"""Throughput of the CLIP vision tower on the device (mmr_encoder_forward_pixels) next to the same HF module run by
PyTorch on the same GPU: what `embed_images_batch` (reference app/ml/embeddings.py:73-91) costs at ingest.

    python benchmarks/vision_encoder_bench.py > vision_encoder_bench.json

ViT-B/32 (12 layers, hidden 768, 224 px, patch 32, projection 512) with seeded random weights (no checkpoints offline).
Pixels are already on the device for every arm (image decoding and CLIPImageProcessor stay on the host and are not timed).
Times are CUDA-event means per forward pass after warm-up.  `hf_fp32_ms` is HF eager in fp32 with torch's default
settings (the reference's path), `hf_bf16_ms` the same module cast to bf16.  FLOPs are the algorithm's multiply-adds x 2
from shapes (patch GEMM, QKV, attention scores and context, out-projection, MLP, projection head); LayerNorms, softmax and
activations are not counted."""
import copy
import importlib
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
enc_mod = importlib.import_module("multimodal-rag-for-image-text-search_b200.encoders")
native = importlib.import_module("multimodal-rag-for-image-text-search_b200._native")

BATCHES = (1, 32, 256, 1024)


def timed(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def flops_per_image(c):
    H, L, I, P, S, C = c.hidden_size, c.num_hidden_layers, c.intermediate_size, c.patch_size, c.image_size, c.num_channels
    NP = (S // P) ** 2
    T = NP + 1
    layer = 2 * T * H * 3 * H + 2 * 2 * T * T * H + 2 * T * H * H + 2 * 2 * T * H * I
    return 2 * NP * C * P * P * H + L * layer + 2 * H * c.projection_dim


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as exc:                                  # the JSON still says where the card facts are missing
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({exc})"}


def main():
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    torch.manual_seed(0)
    model = CLIPVisionModelWithProjection(CLIPVisionConfig()).eval()
    cfg = model.config
    dev = enc_mod.DeviceEncoder.from_hf_clip_vision(model)
    hf32 = model.cuda()
    hf16 = copy.deepcopy(model).to(torch.bfloat16)
    fpi = flops_per_image(cfg)
    out = []
    for b in BATCHES:
        px = (torch.randn(b, 3, cfg.image_size, cfg.image_size, generator=torch.Generator().manual_seed(b)) * 0.8).cuda()
        px16 = px.to(torch.bfloat16)
        res = torch.empty(b, dev.out_dim, device="cuda")
        n0 = native.lib().mmr_launch_count()
        dev.forward_pixels(px, out=res)
        launches = native.lib().mmr_launch_count() - n0
        reps = max(5, 200 // b)
        ours = timed(lambda: dev.forward_pixels(px, out=res), reps)
        with torch.no_grad():
            t32 = timed(lambda: hf32(pixel_values=px), max(3, reps // 4))
            t16 = timed(lambda: hf16(pixel_values=px16), max(3, reps // 4))
        out.append({"batch": b, "device_encoder_ms": ours, "images_per_s": b / ours * 1e3, "kernel_launches": int(launches),
                    "gflop": fpi * b / 1e9, "device_tflops": fpi * b / ours / 1e9,
                    "hf_fp32_ms": t32, "hf_bf16_ms": t16, "hf_fp32_tflops": fpi * b / t32 / 1e9, "hf_bf16_tflops": fpi * b / t16 / 1e9,
                    "speedup_vs_hf_fp32": t32 / ours, "speedup_vs_hf_bf16": t16 / ours})
    print(json.dumps({"what": "CLIP ViT-B/32 image tower, ms per forward pass (CUDA events, pixels resident on the device)",
                      "card": card(), "model": {"hidden": cfg.hidden_size, "layers": cfg.num_hidden_layers,
                                                "image_size": cfg.image_size, "patch_size": cfg.patch_size,
                                                "tokens_per_image": (cfg.image_size // cfg.patch_size) ** 2 + 1,
                                                "flops_per_image": fpi},
                      "results": out}, indent=1))
    dev.close()


if __name__ == "__main__":
    main()
