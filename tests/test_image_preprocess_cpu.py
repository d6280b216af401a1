"""Host side of the device image preprocessing (no GPU needed): the argument checks of mmr_image_preprocess, which all run
before any CUDA call; the resize / crop geometry against transformers' own functions; DeviceImageProcessor.from_hf's
refusals; and the rescale / normalise table against the PIL backend, bit for bit."""
import ctypes as C
import importlib

import numpy as np
import pytest
import torch

PKG = "multimodal-rag-for-image-text-search_b200"
enc_mod = importlib.import_module(PKG + ".encoders")
native = importlib.import_module(PKG + "._native")
INVALID, CUDA = 1, 2


def _pil_processor(**kw):
    from transformers import CLIPImageProcessorPil
    return CLIPImageProcessorPil(**kw)


class _Call:
    """One mmr_image_preprocess call on fake (never dereferenced) 16-byte aligned pointers; geometry rows as keyword edits."""

    def __init__(self):
        self.buf = (C.c_uint8 * 64)()
        self.p = (C.addressof(self.buf) + 15) & ~15

    def __call__(self, crop=(224, 224), B=None, geom=((0, 480, 640, 224, 298, 0, 37),), src_bytes=640 * 480 * 3, src=0, out=0,
                 cfg=True, geom_ptr=True):
        c = native.ImagePrep(*crop)
        g = np.ascontiguousarray(np.asarray(geom, dtype=np.int64).reshape(-1, 7))
        src = self.p if src == 0 else src
        out = self.p if out == 0 else out
        return native.lib().mmr_image_preprocess(0, C.byref(c) if cfg else None, src, src_bytes, g.ctypes.data if geom_ptr else None,
                                                 len(g) if B is None else B, out, None)


def test_preprocess_rejects_bad_arguments_before_any_cuda_call():
    lib = native.lib()
    call = _Call()
    good = (0, 480, 640, 224, 298, 0, 37)
    cases = [
        (dict(cfg=False), b"NULL"), (dict(geom_ptr=False), b"NULL"), (dict(src=None), b"NULL"), (dict(out=None), b"NULL"),
        (dict(B=0), b"B = 0"), (dict(B=-2), b"B = -2"),
        (dict(crop=(0, 224)), b"crop 0 x 224"), (dict(crop=(224, 4097)), b"crop 224 x 4097"),
        (dict(src=call.p + 4), b"16-byte aligned"), (dict(out=call.p + 2), b"4-byte aligned"),
        (dict(src_bytes=8), b"src_bytes = 8"),
        (dict(geom=(0, 0, 640, 224, 298, 0, 37)), b"image 0: 0 x 640"),
        (dict(geom=(0, 480, 65536, 224, 30583, 0, 37)), b"image 0: 480 x 65536"),
        (dict(geom=(0, 480, 640, 0, 298, 0, 37)), b"resized to 0 x 298"),
        (dict(geom=(0, 480, 640, 224, (1 << 24) + 1, 0, 37)), b"resized to 224 x 16777217"),
        (dict(geom=(0, 480, 640, 224, 298, -1, 37)), b"not inside"),
        (dict(geom=(0, 480, 640, 224, 298, 0, -1)), b"not inside"),
        (dict(geom=(0, 480, 640, 224, 298, 1, 37)), b"not inside"),          # top + crop_h > out_h
        (dict(geom=(0, 480, 640, 224, 298, 0, 75)), b"not inside"),          # left + crop_w > out_w
        (dict(crop=(224, 300)), b"not inside"),
        (dict(geom=(0, 480, 64000, 224, 298, 0, 37), src_bytes=480 * 64000 * 3), b"63.5x"),   # 214x along the width
        (dict(geom=(0, 20000, 640, 224, 298, 0, 37), src_bytes=20000 * 640 * 3), b"63.5x"),
        (dict(geom=(0, 14225, 640, 224, 640, 0, 0), src_bytes=14225 * 640 * 3), b"63.5x"),   # 257 taps
        (dict(geom=(16, 480, 640, 224, 298, 0, 37)), b"offset 16"),          # runs past src_bytes
        (dict(geom=(8, 480, 640, 224, 298, 0, 37), src_bytes=10 ** 7), b"offset 8"),   # not a multiple of 16
        (dict(geom=(-16, 480, 640, 224, 298, 0, 37)), b"offset -16"),
        (dict(geom=(0, 7, 7, 224, 224, 0, 0), src_bytes=147), b"offset 0"),   # 147 bytes round up to 160
        (dict(geom=(good, (921600, 480, 640, 224, 298, 0, 37))), b"image 1"),  # the second image runs past src_bytes
    ]
    for kw, words in cases:
        assert call(**kw) == INVALID, (kw, lib.mmr_last_error())
        assert words in lib.mmr_last_error(), (kw, lib.mmr_last_error())


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_device_no_preprocessing():
    """Valid arguments (a 63.5x downscale included) reach the device and fail there: no fallback."""
    call = _Call()
    assert call() == CUDA
    assert call(geom=(0, 14224, 640, 224, 640, 0, 0), src_bytes=14224 * 640 * 3) == CUDA   # 255 taps
    with pytest.raises(native.NativeError):
        enc_mod.DeviceImageProcessor.from_hf(_pil_processor())


def _hf_geometry(h, w, se, ch, cw):
    from transformers.image_transforms import center_crop, get_resize_output_image_size
    from transformers.image_utils import ChannelDimension
    first = ChannelDimension.FIRST
    out_h, out_w = get_resize_output_image_size(np.broadcast_to(np.uint8(0), (3, h, w)), size=se, default_to_square=False,
                                                input_data_format=first)
    rows = np.broadcast_to(np.arange(out_h, dtype=np.int64)[None, :, None], (1, out_h, out_w))
    cols = np.broadcast_to(np.arange(out_w, dtype=np.int64)[None, None, :], (1, out_h, out_w))
    top = int(center_crop(rows, (ch, cw), input_data_format=first)[0, 0, 0])
    left = int(center_crop(cols, (ch, cw), input_data_format=first)[0, 0, 0])
    return out_h, out_w, top, left


def test_geometry_matches_transformers():
    sizes = [(h, w) for h in range(1, 400, 13) for w in range(1, 400, 11)]
    sizes += [(1, 1000), (1000, 1), (1, 224), (224, 1), (57, 1000), (1000, 57), (6000, 4000), (4000, 6000), (1080, 1920),
              (224, 224), (224, 225), (225, 224), (3, 65535)]
    for se, ch, cw in ((224, 224, 224), (256, 224, 224), (224, 200, 150)):
        for h, w in sizes:
            assert enc_mod.clip_resize_geometry(h, w, se, ch, cw) == _hf_geometry(h, w, se, ch, cw), (h, w, se, ch, cw)


def test_table_equals_the_pil_backend_on_a_ramp():
    """A 1 x 256 image whose every channel is the ramp 0..255, through CLIPImageProcessorPil without resize and crop, is the
    [3, 256] table itself."""
    from PIL import Image
    ramp = Image.fromarray(np.repeat(np.arange(256, dtype=np.uint8)[None, :, None], 3, axis=2), "RGB")
    cases = [dict(), dict(image_mean=[0.5, 0.4, 0.3], image_std=[0.2, 0.25, 0.3]), dict(rescale_factor=1 / 127.5),
             dict(do_normalize=False), dict(do_rescale=False), dict(image_mean=0.5, image_std=0.5)]
    for kw in cases:
        proc = _pil_processor(**kw)
        want = proc(images=[ramp], do_resize=False, do_center_crop=False, return_tensors="np")["pixel_values"][0]
        got = enc_mod.clip_value_table(proc.do_rescale, proc.rescale_factor, proc.do_normalize, proc.image_mean, proc.image_std)
        assert got.dtype == np.float32 and got.shape == (3, 256)
        assert np.array_equal(got.view(np.int32), want.reshape(3, 256).astype(np.float32).view(np.int32)), kw


def test_from_hf_refuses_what_it_cannot_reproduce():
    from PIL import Image
    from transformers import CLIPImageProcessor
    for proc in (_pil_processor(), CLIPImageProcessor()):
        assert enc_mod.DeviceImageProcessor._hf_fields(proc) == (224, 224, 224)
    assert enc_mod.DeviceImageProcessor._hf_fields(_pil_processor(size={"shortest_edge": 256})) == (256, 224, 224)
    cases = [
        (dict(resample=Image.Resampling.BILINEAR), "resample"),
        (dict(resample=Image.Resampling.LANCZOS), "resample"),
        (dict(size={"height": 224, "width": 224}), "size"),
        (dict(do_center_crop=False), "do_center_crop"),
        (dict(crop_size={"height": 256, "width": 256}), "crop_size"),
        (dict(size={"shortest_edge": 200}), "crop_size"),
        (dict(do_resize=False), "do_resize"),
        (dict(do_convert_rgb=False), "do_convert_rgb"),
    ]
    for backend in (_pil_processor, CLIPImageProcessor):
        for kw, field in cases:
            with pytest.raises(ValueError, match=field):
                enc_mod.DeviceImageProcessor.from_hf(backend(**kw))
