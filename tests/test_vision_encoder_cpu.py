"""Host side of the CLIP vision tower (no GPU needed): HF state_dict -> C-ABI weight names, the activation check, and the
argument checks of mmr_encoder_create_vision / mmr_encoder_forward_pixels / mmr_debug_enc_patch_embed, which all run
before any CUDA call."""
import ctypes as C
import importlib

import pytest
import torch

PKG = "multimodal-rag-for-image-text-search_b200"
enc_mod = importlib.import_module(PKG + ".encoders")
native = importlib.import_module(PKG + "._native")
INVALID, CUDA, UNSUPPORTED = 1, 2, 3
B32 = dict(hidden=768, layers=12, heads=12, intermediate=3072, image_size=224, patch_size=32, channels=3, proj_dim=512, ln_eps=1e-5)


def _check_weights(w, layers, H=768, C_=3, P=32, NP=49, proj=512):
    assert w["patch_w"].shape == (H, C_ * P * P)
    assert w["cls_emb"].shape == (H,) and w["pos_emb"].shape == (NP + 1, H)
    assert w["pre_ln_w"].shape == (H,) and w["pre_ln_b"].shape == (H,)
    assert w["final_ln_w"].shape == (H,) and w["final_ln_b"].shape == (H,) and w["proj_w"].shape == (proj, H)
    assert w[f"L{layers - 1}.qkv_w"].shape == (3 * H, H) and w["L0.qkv_b"].shape == (3 * H,)
    assert w["L0.o_w"].shape == (H, H) and w["L0.fc1_w"].shape == (4 * H, H) and w["L0.fc2_w"].shape == (H, 4 * H)
    assert f"L{layers}.qkv_w" not in w
    assert len(w) == 8 + 12 * layers


def test_clip_vision_weight_names_and_shapes():
    from transformers import CLIPConfig, CLIPModel, CLIPVisionConfig, CLIPVisionModelWithProjection
    model = CLIPVisionModelWithProjection(CLIPVisionConfig(num_hidden_layers=2))
    w = enc_mod.hf_clip_vision_weights(model)
    _check_weights(w, 2)
    sd = model.state_dict()
    pw = sd["vision_model.embeddings.patch_embedding.weight"]
    assert torch.equal(w["patch_w"], pw.reshape(768, -1))
    assert torch.equal(w["patch_w"][5, 2 * 1024 + 3 * 32 + 7], pw[5, 2, 3, 7])          # column order (c, kh, kw)
    assert torch.equal(w["L1.qkv_w"][768:1536], sd["vision_model.encoder.layers.1.self_attn.k_proj.weight"])   # q | k | v
    # a CLIPModel: the vision tower only, the text tower's weights stay out
    full = CLIPModel(CLIPConfig(text_config=dict(num_hidden_layers=1, vocab_size=100),
                                vision_config=dict(num_hidden_layers=2, image_size=64, patch_size=16), projection_dim=256))
    w = enc_mod.hf_clip_vision_weights(full)
    _check_weights(w, 2, P=16, NP=16, proj=256)
    assert torch.equal(w["proj_w"], full.state_dict()["visual_projection.weight"])


def test_from_hf_clip_vision_refuses_other_activations_before_the_library():
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    for act in ("gelu", "gelu_new"):
        with pytest.raises(ValueError, match="hidden_act"):
            enc_mod.DeviceEncoder.from_hf_clip_vision(CLIPVisionModelWithProjection(CLIPVisionConfig(num_hidden_layers=1,
                                                                                                    hidden_act=act)))
    enc_mod._check_supported(CLIPVisionConfig(num_hidden_layers=1), {"quick_gelu"})


def _create(**kw):
    cfg = native.VisionConfig(**{**B32, **kw})
    out = C.c_void_p()
    rc = native.lib().mmr_encoder_create_vision(0, C.byref(cfg), C.byref(out))
    return rc, native.lib().mmr_last_error()


def test_create_vision_rejects_bad_configs_before_any_cuda_call():
    lib = native.lib()
    out = C.c_void_p()
    assert lib.mmr_encoder_create_vision(0, None, C.byref(out)) == INVALID and b"NULL" in lib.mmr_last_error()
    cfg = native.VisionConfig(**B32)
    assert lib.mmr_encoder_create_vision(0, C.byref(cfg), None) == INVALID and b"NULL" in lib.mmr_last_error()
    cases = [
        (dict(hidden=512, heads=8), UNSUPPORTED, b"hidden 512"),           # not 768
        (dict(hidden=1024, heads=16), UNSUPPORTED, b"hidden 1024"),        # ViT-L
        (dict(heads=24), UNSUPPORTED, b"heads 24"),                        # head dim 32
        (dict(heads=0), UNSUPPORTED, b"heads 0"),
        (dict(heads=5), UNSUPPORTED, b"heads 5"),
        (dict(layers=0), INVALID, b"layers = 0"),
        (dict(channels=0), INVALID, b"channels 0"),
        (dict(patch_size=0), INVALID, b"patch_size 0"),
        (dict(image_size=0), INVALID, b"image_size 0"),
        (dict(image_size=225), INVALID, b"not a multiple of patch_size"),
        (dict(channels=1, patch_size=4, image_size=32), UNSUPPORTED, b"multiple of 64"),    # C P^2 = 16
        (dict(channels=3, patch_size=14), UNSUPPORTED, b"multiple of 64"),                  # 588
        (dict(intermediate=3000), UNSUPPORTED, b"intermediate"),
        (dict(intermediate=0), UNSUPPORTED, b"intermediate"),
        (dict(patch_size=8), UNSUPPORTED, b"785 tokens"),                  # 28^2 + 1 > 330
        (dict(image_size=608, patch_size=32), UNSUPPORTED, b"362 tokens"),
        (dict(proj_dim=0), INVALID, b"proj_dim 0"),
        (dict(proj_dim=769), INVALID, b"proj_dim 769"),
    ]
    for kw, code, words in cases:
        rc, msg = _create(**kw)
        assert rc == code, (kw, rc, msg)
        assert words in msg, (kw, msg)


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_device_no_vision_encoder():
    """A valid config (ViT-B/32, and ViT-B/16 at 197 tokens) reaches the device check and fails there: no fallback."""
    assert _create()[0] == CUDA
    assert _create(patch_size=16)[0] == CUDA
    with pytest.raises(native.NativeError):
        enc_mod.DeviceEncoder("clip_vision", **B32)


def test_forward_pixels_rejects_bad_arguments():
    lib = native.lib()
    buf = (C.c_float * 64)()
    p = C.addressof(buf)
    for args, words in (((None, p, 1, p), b"NULL"), ((p, None, 1, p), b"NULL"), ((p, p, 1, None), b"NULL"),
                        ((p, p, 0, p), b"B = 0"), ((p, p, -3, p), b"B = -3"), ((p, p, 65536, p), b"B = 65536")):
        e = None if args[0] is None else C.c_void_p(0)
        assert lib.mmr_encoder_forward_pixels(e, args[1], args[2], args[3], None) == INVALID, args
        assert words in lib.mmr_last_error(), (args, lib.mmr_last_error())


def test_patch_embed_hook_rejects_bad_arguments():
    """mmr_debug_enc_patch_embed checks everything before any CUDA call (the buffers below are never dereferenced)."""
    lib = native.lib()
    buf = (C.c_float * 64)()
    p = C.addressof(buf)
    odd = p + 2

    def hook(H=768, C_=3, S=224, P=32, B=1, px=p, w=p, cls=p, pos=p, g=p, b=p, p16=p, pout=p, x=p):
        return lib.mmr_debug_enc_patch_embed(H, C_, S, P, B, px, w, cls, pos, g, b, 1e-5, p16, pout, x, None)

    cases = [
        (dict(H=512), b"H = 512"), (dict(H=1024), b"H = 1024"),
        (dict(C_=0), b"C = 0"), (dict(P=0), b"patch = 0"), (dict(S=0), b"image_size = 0"),
        (dict(S=100), b"not a multiple of patch"),
        (dict(C_=1, P=4, S=32), b"multiple of 64"),
        (dict(B=0), b"B = 0"), (dict(B=65536), b"B = 65536"),
        (dict(B=30000, P=16), b"2^22"),                                   # 30000 x 197 tokens
        (dict(px=None), b"NULL"), (dict(cls=None), b"NULL"), (dict(pos=None), b"NULL"), (dict(g=None), b"NULL"),
        (dict(b=None), b"NULL"), (dict(pout=None), b"NULL"), (dict(x=None), b"NULL"),
        (dict(w=None), b"patch_w and patch16"), (dict(w=odd), b"patch_w and patch16"),
        (dict(p16=None), b"patch_w and patch16"), (dict(p16=odd), b"patch_w and patch16"),
    ]
    for kw, words in cases:
        assert hook(**kw) == INVALID, kw
        assert words in lib.mmr_last_error(), (kw, lib.mmr_last_error())
