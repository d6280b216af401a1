#!/usr/bin/env python
"""CLIP image preprocessing per image: HF's two host processors next to the device path (DeviceImageProcessor ->
mmr_image_preprocess), and what each gives the ingest path end to end (ImageEncoder images/s with the ViT-B/32 tower).

    python benchmarks/image_preprocess_bench.py > image_preprocess_bench.json

Input: a seeded synthetic mix of decoded RGB PIL images, 224x224, 500x375, 640x480, 1280x720 and 1920x1080 in turn, at
batches of 32 and 256.  Arms, in ms per image:
  host_torchvision / host_pil   CLIPImageProcessor() / CLIPImageProcessorPil() on the host CPU (wall clock, one batch call)
  device_call                   DeviceImageProcessor.__call__ end to end (pack into pinned memory, upload, kernel), wall
                                clock to a device synchronise
  h2d                           the upload alone: the packed uint8 bytes from pinned memory (CUDA events)
  kernel                        mmr_image_preprocess alone on resident bytes (CUDA events, mean over repeats).  `kernel_gbps`
                                counts the source bytes the crop windows need (the input rows and columns under each crop's
                                bicubic windows) plus the fp32 output.  The 32-image batch's source fits the 126 MB L2 and
                                is read from there on repeats; the 256-image batch's does not.
ImageEncoder images/s: the whole embed_images_batch call (preprocess, tower, copy back) at batch_size = the batch, with
each processor.  The device output is checked bit for bit against CLIPImageProcessorPil on every batch."""
import ctypes as C
import importlib
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
from vision_encoder_bench import card, timed  # noqa: E402

enc_mod = importlib.import_module("multimodal-rag-for-image-text-search_b200.encoders")
native = importlib.import_module("multimodal-rag-for-image-text-search_b200._native")

MIX = [(224, 224), (500, 375), (640, 480), (1280, 720), (1920, 1080)]
BATCHES = (32, 256)


def images(n, seed):
    from PIL import Image
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        w, h = MIX[i % len(MIX)]
        base = rng.integers(0, 256, size=(1, 1, 3))
        out.append(Image.fromarray(np.clip(base + rng.integers(-60, 60, size=(h, w, 3)), 0, 255).astype(np.uint8), "RGB"))
    return out


def window(in_size, out_size, lo, n):
    """Input indices [first, end) that Pillow's bicubic windows of outputs lo .. lo + n - 1 cover."""
    if in_size == out_size:
        return lo, lo + n
    scale = in_size / out_size
    support = 2.0 * max(scale, 1.0)
    first = max(int((lo + 0.5) * scale - support + 0.5), 0)
    end = min(int((lo + n - 1 + 0.5) * scale + support + 0.5), in_size)
    return first, end


def wall(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / reps


def main():
    from transformers import CLIPImageProcessor, CLIPImageProcessorPil, CLIPVisionConfig, CLIPVisionModelWithProjection
    tv, pil = CLIPImageProcessor(), CLIPImageProcessorPil()
    dev = enc_mod.DeviceImageProcessor.from_hf(pil)
    torch.manual_seed(0)
    tower = enc_mod.DeviceEncoder.from_hf_clip_vision(CLIPVisionModelWithProjection(CLIPVisionConfig()).eval())
    lib = native.lib()
    results = []
    for b in BATCHES:
        ims = images(b, seed=b)
        host_reps = 2 if b <= 32 else 1
        t_tv = wall(lambda: tv(images=ims, return_tensors="pt"), host_reps)
        t_pil = wall(lambda: pil(images=ims, return_tensors="pt"), host_reps)
        want = pil(images=ims, return_tensors="pt")["pixel_values"]
        got = dev(images=ims)["pixel_values"]
        identical = bool(torch.equal(got.cpu().view(torch.int32), want.view(torch.int32)))
        t_call = wall(lambda: dev(images=ims), 10)

        # the upload and the kernel alone, on the packing DeviceImageProcessor makes
        arrays = [np.asarray(im) for im in ims]
        geom = np.empty((b, 7), dtype=np.int64)
        off, need = 0, 0
        for i, a in enumerate(arrays):
            h, w = a.shape[:2]
            oh, ow, top, left = enc_mod.clip_resize_geometry(h, w, 224, 224, 224)
            geom[i] = (off, h, w, oh, ow, top, left)
            y0, y1 = window(h, oh, top, 224)
            x0, x1 = window(w, ow, left, 224)
            need += (y1 - y0) * (x1 - x0) * 3
            off += (a.nbytes + 15) & ~15
        host = torch.empty(off, dtype=torch.uint8, pin_memory=True)
        hv = host.numpy()
        for a, (o, h, w) in zip(arrays, geom[:, :3]):
            hv[o:o + h * w * 3] = a.reshape(-1)
        src = torch.empty(off, dtype=torch.uint8, device="cuda")
        out = torch.empty(b, 3, 224, 224, device="cuda")
        t_h2d = timed(lambda: src.copy_(host, non_blocking=True), 20)
        stream = torch.cuda.current_stream().cuda_stream

        def kernel():
            native.check(lib.mmr_image_preprocess(0, C.byref(dev.cfg), src.data_ptr(), off, geom.ctypes.data, b, out.data_ptr(), stream))

        t_kernel = timed(kernel, 50)
        assert torch.equal(out.cpu().view(torch.int32), want.view(torch.int32))
        out_bytes = b * 3 * 224 * 224 * 4

        enc_host = enc_mod.ImageEncoder(tv, tower)
        enc_pil = enc_mod.ImageEncoder(pil, tower)
        enc_dev = enc_mod.ImageEncoder(dev, tower)
        t_e2e_tv = wall(lambda: enc_host(ims, batch_size=b), host_reps)
        t_e2e_pil = wall(lambda: enc_pil(ims, batch_size=b), host_reps)
        t_e2e_dev = wall(lambda: enc_dev(ims, batch_size=b), 5)
        results.append({
            "batch": b, "bit_identical_to_pil": identical,
            "source_mb_packed": off / 1e6, "source_mb_crop_windows": need / 1e6, "output_mb": out_bytes / 1e6,
            "ms_per_image": {"host_torchvision": t_tv / b, "host_pil": t_pil / b, "device_call": t_call / b,
                             "h2d": t_h2d / b, "kernel": t_kernel / b},
            "h2d_gbps": off / t_h2d / 1e6, "kernel_ms": t_kernel, "kernel_gbps": (need + out_bytes) / t_kernel / 1e6,
            "image_encoder_images_per_s": {"host_torchvision": b / t_e2e_tv * 1e3, "host_pil": b / t_e2e_pil * 1e3,
                                           "device": b / t_e2e_dev * 1e3},
        })
    print(json.dumps({"what": "CLIP image preprocessing, ms per image (mix " + ", ".join(f"{w}x{h}" for w, h in MIX) + ")",
                      "card": card(), "host_cpus": os.cpu_count(), "results": results}, indent=1))
    tower.close()


if __name__ == "__main__":
    main()
