"""CLIP image preprocessing on the device (DeviceImageProcessor -> mmr_image_preprocess) against HF's processors: bit-identical
to CLIPImageProcessorPil (Pillow's bicubic resize, centre crop, rescale, normalise) for every size, content and input kind
below; within two uint8 steps of the default torchvision-backed CLIPImageProcessor; and through the CLIP vision tower."""
import importlib

import numpy as np
import pytest
import torch

from tests.test_gpu_vision_encoder import TOL, _pil_images, _reference, _vision_model

pytestmark = pytest.mark.gpu
PKG = "multimodal-rag-for-image-text-search_b200"

# (width, height): square at the target, one pixel off it (one pass only), landscape and portrait downscales, pure upscales,
# extreme aspect ratios, and a 6000 x 4000 photo (73-tap windows)
SIZES = [(224, 224), (224, 225), (640, 480), (1920, 1080), (100, 300), (33, 33), (1000, 57), (57, 1000), (6000, 4000)]


def _content(kind, w, h, seed):
    """smooth gradients; uniform noise; a one-pixel checkerboard of 0 / 255 (the bicubic lobes ring past both ends, so the
    clip to [0, 255] decides many bytes)."""
    if kind == "smooth":
        y, x = np.mgrid[0:h, 0:w].astype(np.float64)
        a = np.stack([255 * x / max(w - 1, 1), 255 * y / max(h - 1, 1), 127.5 + 127.5 * np.sin((x + 2 * y) / 37.0)], -1)
        return np.round(a).astype(np.uint8)
    if kind == "noise":
        return np.random.default_rng(seed).integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    y, x = np.mgrid[0:h, 0:w]
    board = (((x + y) & 1) * 255).astype(np.uint8)
    return np.stack([board, 255 - board, board], -1)


def _images(kinds=("smooth", "noise", "checker"), sizes=SIZES):
    from PIL import Image
    return [Image.fromarray(_content(k, w, h, seed=w * 7 + h), "RGB") for w, h in sizes for k in kinds]


@pytest.fixture(scope="module")
def enc_mod():
    return importlib.import_module(PKG + ".encoders")


@pytest.fixture(scope="module")
def pil_proc():
    from transformers import CLIPImageProcessorPil
    return CLIPImageProcessorPil()


@pytest.fixture(scope="module")
def dev_proc(enc_mod, pil_proc):
    return enc_mod.DeviceImageProcessor.from_hf(pil_proc)


def _bits_equal(got, want):
    assert got.is_cuda and got.dtype == torch.float32 and got.shape == want.shape, (got.shape, want.shape)
    got = got.cpu()
    diff = got.view(torch.int32) != want.to(torch.float32).view(torch.int32)
    assert not bool(diff.any()), f"{int(diff.sum())} of {diff.numel()} values differ; first at {diff.nonzero()[0].tolist()}"


def test_bit_identical_to_the_pil_backend(pil_proc, dev_proc):
    """Every size x content in one ragged batch, then each image alone: both equal CLIPImageProcessorPil bit for bit."""
    images = _images()
    want = pil_proc(images=images, return_tensors="pt")["pixel_values"]
    batch = dev_proc(images=images, return_tensors="pt")["pixel_values"]
    _bits_equal(batch, want)
    for i, im in enumerate(images):
        alone = dev_proc(images=[im], return_tensors="pt")["pixel_values"]
        assert torch.equal(alone[0], batch[i]), (i, im.size)


def test_other_crops_and_sizes(enc_mod):
    """shortest_edge 256 with a 224 crop (every image resized, then cropped on both axes), and a 223 x 201 crop whose
    offsets are odd and whose width is not a multiple of the kernel's 32-column tile."""
    from transformers import CLIPImageProcessorPil
    images = _images(kinds=("noise", "checker"))
    for kw in (dict(size={"shortest_edge": 256}), dict(crop_size={"height": 223, "width": 201}),
               dict(image_mean=[0.5, 0.5, 0.5], image_std=[0.5, 0.5, 0.5])):
        proc = CLIPImageProcessorPil(**kw)
        dev = enc_mod.DeviceImageProcessor.from_hf(proc)
        _bits_equal(dev(images=images)["pixel_values"], proc(images=images, return_tensors="pt")["pixel_values"])


def test_image_modes_and_arrays(pil_proc, dev_proc):
    """Grayscale, RGBA and palette PIL images are converted to RGB as the processor converts them; uint8 [H, W, 3] arrays
    (also non-contiguous views) give what their PIL image gives."""
    from PIL import Image
    base = _images(kinds=("smooth", "noise"), sizes=[(640, 480), (100, 300), (224, 225)])
    rgba = []
    for im in base:
        a = np.asarray(im.convert("RGBA")).copy()
        a[..., 3] = np.arange(a.shape[1], dtype=np.uint8)[None, :]
        rgba.append(Image.fromarray(a, "RGBA"))
    modes = [im.convert("L") for im in base] + rgba + [im.convert("P", palette=Image.Palette.ADAPTIVE, colors=64) for im in base]
    _bits_equal(dev_proc(images=modes)["pixel_values"], pil_proc(images=modes, return_tensors="pt")["pixel_values"])
    arrays = [np.asarray(im) for im in base] + [np.asarray(base[0])[::2, ::3]]
    want = pil_proc(images=base + [Image.fromarray(np.ascontiguousarray(arrays[-1]))], return_tensors="pt")["pixel_values"]
    _bits_equal(dev_proc(images=arrays)["pixel_values"], want)
    with pytest.raises(TypeError):
        dev_proc(images=[np.zeros((8, 8, 3), np.float32)])
    with pytest.raises(TypeError):
        dev_proc(images=[np.zeros((8, 8), np.uint8)])


def test_repeated_calls_reuse_the_staging_buffer(pil_proc, dev_proc):
    """Calls back to back without a synchronise: a later call's packing must not overwrite bytes an earlier upload still
    reads."""
    base = _images(kinds=("noise",), sizes=[(1920, 1080), (640, 480)] * 2)
    sets = [base, [im.transpose(0) for im in base], [im.rotate(90, expand=True) for im in base]]
    outs = [dev_proc(images=s)["pixel_values"] for s in sets]
    for s, o in zip(sets, outs):
        _bits_equal(o, pil_proc(images=s, return_tensors="pt")["pixel_values"])


def test_close_to_the_torchvision_backend():
    """The default CLIPImageProcessor resizes with torch's uint8 bicubic, which differs from Pillow's in a few bytes by one
    or two steps; through the tower the embeddings stay within TOL of the default processor's."""
    from transformers import CLIPImageProcessor
    enc_mod = importlib.import_module(PKG + ".encoders")
    proc = CLIPImageProcessor()
    dev = enc_mod.DeviceImageProcessor.from_hf(proc)
    images = _images(kinds=("smooth", "noise"), sizes=SIZES[:-1])
    got = dev(images=images)["pixel_values"].cpu()
    want = proc(images=images, return_tensors="pt")["pixel_values"]
    std = torch.tensor(proc.image_std).view(1, 3, 1, 1)
    steps = (got - want).abs() * std * 255.0
    assert float(steps.max()) <= 2.0 + 1e-3, float(steps.max())
    frac = float((steps > 0.5).float().mean())
    assert frac <= 0.02, frac
    model = _vision_model(11)
    enc = enc_mod.DeviceEncoder.from_hf_clip_vision(model)
    emb = enc.forward_pixels(dev(images=images)["pixel_values"])
    ref = _reference(model.cuda(), want)
    assert (emb - ref).abs().max().item() <= TOL
    enc.close()


def test_image_encoder_with_the_device_processor(enc_mod, pil_proc, dev_proc):
    """ImageEncoder(DeviceImageProcessor, enc) = ImageEncoder(CLIPImageProcessorPil, enc) bit for bit, and ingest then
    search: 600 images of mixed sizes embedded through the device processor are each their own top hit."""
    model = _vision_model(11)
    enc = enc_mod.DeviceEncoder.from_hf_clip_vision(model)
    images = _pil_images([(224, 224), (640, 480), (100, 300), (1000, 57), (33, 33), (224, 225), (512, 512)], seed=3)
    got = enc_mod.ImageEncoder(dev_proc, enc)(images)
    want = enc_mod.ImageEncoder(pil_proc, enc)(images)
    assert np.array_equal(got, want)

    mmr = importlib.import_module(PKG)
    store_mod = importlib.import_module(PKG + ".store")
    n = 600
    sizes = [(224, 224), (500, 375), (640, 480), (375, 500), (300, 100), (1280, 720)]
    ingest = _pil_images([sizes[i % len(sizes)] for i in range(n)], seed=77)
    emb = enc_mod.ImageEncoder(dev_proc, enc)(ingest, batch_size=128)
    assert emb.shape == (n, 512)
    store = mmr.B200Store()
    store.upsert_image_vectors([store_mod.VectorRow(chunk_id=f"img{i}", user_id="u", document_id="d", modality="image",
                                                    embedding=emb[i], meta={}) for i in range(n)])
    for i in np.random.default_rng(5).choice(n, 16, replace=False):
        hits = store.search_image("u", emb[i], 5)
        assert hits[0]["chunk_id"] == f"img{i}", (i, hits[:2])
        assert hits[0]["score"] >= 1 - 1e-3, (i, hits[0]["score"])
    enc.close()
