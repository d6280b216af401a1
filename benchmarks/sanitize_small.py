#!/usr/bin/env python
"""Small shapes through every kernel, for `compute-sanitizer --tool {memcheck,racecheck,synccheck} python ...`."""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import util  # noqa: E402

pkg = importlib.import_module("multimodal-rag-for-image-text-search_b200")


def main():
    rows = util.unit_rows(6000, 512, seed=1)
    seg = np.array([0, 100, 100, 3000, 6000], dtype=np.int64)
    for dtype in ("bf16", "f32"):
        ix = pkg.ResidentIndex.from_f32(rows, seg_offsets=seg, dtype=dtype)
        for b in (1, 2, 4):
            q = torch.from_numpy(util.queries(b, 512)).cuda()
            ix.search(q, 10)
            ix.search(q, 50, [2] * b)
        q = torch.from_numpy(util.queries(4, 512)).cuda()
        ix.search(q, 10, [0, 1, 2, 3])            # varlen
        ix.search_ranges(q, 10, [[(0, 50), (200, 900)], [(10, 20)], [], [(0, 6000)]])
        ix.close()
    ix = pkg.ResidentIndex.from_f32(rows, dtype="bf16")
    for b in (5, 130):                             # K2: one query tile (single CTAs), two (CTA pairs)
        q = torch.from_numpy(util.queries(b, 512)).cuda()
        s, r = ix.search(q, 10)
        ix.debug_umma_scores(q, 0, 6000)
    parts_s = torch.stack([s, s]); parts_r = torch.stack([r, r + 100000])
    pkg.merge_topk(parts_s, parts_r)
    pkg.fuse((s, r), (s[:, :5].contiguous(), r[:, :5].contiguous()), 4, 0.25)
    # image preprocessing: a ragged batch with a downscale, an upscale, one-pass and no-resize images and a partial tile
    enc_mod = importlib.import_module("multimodal-rag-for-image-text-search_b200.encoders")
    table = np.tile(np.arange(256, dtype=np.float32), (3, 1))
    prep = enc_mod.DeviceImageProcessor(40, 40, 37, table)
    rng = np.random.default_rng(0)
    prep(images=[rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in ((300, 170), (13, 29), (40, 41), (40, 40))])
    torch.cuda.synchronize()
    print("sanitize_small: done")


if __name__ == "__main__":
    main()
