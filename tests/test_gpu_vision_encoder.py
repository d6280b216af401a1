"""CLIP vision tower on the device (mmr_encoder_create_vision / mmr_encoder_forward_pixels) against plain fp32 PyTorch on the
SAME weights, its front end against a float64 reference, and its batch invariance.

As in tests/test_gpu_encoders.py, the HF modules are built from their configs with seeded random weights (no checkpoint
files offline), spread so that softmax / GELU / LayerNorm see spread, and the linear and patch-embedding weights are rounded
to bf16-representable values first: both sides hold identical weights and only the activation precision differs (bf16 GEMM
inputs on the device, fp32 in torch).  Tolerance: |delta| <= 1e-3 per component of the unit-norm embedding (DESIGN §2).
The torch references run with TF32 off (cuDNN would otherwise run the patch-embedding convolution in TF32)."""
import contextlib
import ctypes as C
import importlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
PKG = "multimodal-rag-for-image-text-search_b200"
TOL = 1e-3
U = 2.0 ** -24


def _round_linear_weights(model):
    """Linear weights and the patch embedding's Conv2d weight -> bf16-representable values (the device keeps both as bf16)."""
    with torch.no_grad():
        for name, p in model.named_parameters():
            if (p.dim() == 2 and "embedding" not in name.lower()) or name.endswith("patch_embedding.weight"):
                p.copy_(p.to(torch.bfloat16).to(torch.float32))
    return model.eval()


def _spread(model, scale=2.0):
    """Random init (std 0.02) gives near-uniform attention; scale the projections up so softmax / GELU / LN see spread."""
    with torch.no_grad():
        for name, p in model.named_parameters():
            if p.dim() == 2 and "embedding" not in name.lower():
                p.mul_(scale)
            elif p.dim() == 1 and "bias" in name:
                p.normal_(0.0, 0.05)
            elif p.dim() == 1 and "weight" in name:
                p.normal_(1.0, 0.1)
    return model


@contextlib.contextmanager
def _no_tf32():
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


def _reference(model_gpu, px):
    with torch.no_grad(), _no_tf32():
        return F.normalize(model_gpu(pixel_values=px.cuda()).image_embeds, dim=1)


def _pixels(b, size, seed):
    """Roughly what CLIPImageProcessor yields: per-channel normalised values within about [-2, 2]."""
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(b, 3, size, size, generator=g) * 0.8).clamp(-1.8, 2.1)


def _vision_model(seed, **cfg):
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection
    torch.manual_seed(seed)
    return _round_linear_weights(_spread(CLIPVisionModelWithProjection(CLIPVisionConfig(**cfg))))


@pytest.fixture(scope="module")
def enc_mod():
    return importlib.import_module(PKG + ".encoders")


@pytest.fixture(scope="module")
def native():
    n = importlib.import_module(PKG + "._native")
    n.lib()
    return n


@pytest.fixture(scope="module")
def vit_b32():
    """ViT-B/32 as openai/clip-vit-base-patch32 ships it: 12 layers, hidden 768, 224 px, patch 32, projection 512."""
    return _vision_model(11)


@pytest.fixture(scope="module")
def vit_b32_gpu(vit_b32):
    import copy
    return copy.deepcopy(vit_b32).cuda()


@pytest.fixture(scope="module")
def b32_enc(enc_mod, vit_b32):
    enc = enc_mod.DeviceEncoder.from_hf_clip_vision(vit_b32)
    yield enc
    enc.close()


def test_vit_b32_matches_fp32_torch(enc_mod, native, vit_b32, vit_b32_gpu, b32_enc):
    assert b32_enc.kind == "clip_vision" and b32_enc.out_dim == 512
    for b in (1, 8, 64):
        px = _pixels(b, 224, seed=b)
        want = _reference(vit_b32_gpu, px)
        got = b32_enc.forward_pixels(px)
        assert got.shape == (b, 512) and got.is_cuda and got.dtype == torch.float32
        err = (got - want).abs().max().item()
        assert err <= TOL, (b, err)
        assert torch.allclose(got.norm(dim=1), torch.ones(b, device="cuda"), atol=1e-5)
    # the other entry point / kind combinations are refused with a message
    ids = np.ones((1, 4), np.int32)
    out = torch.empty(1, 512, device="cuda")
    rc = native.lib().mmr_encoder_forward(b32_enc._handle, ids.ctypes.data, None, None, 1, 4, out.data_ptr(), None)
    assert rc == 1 and b"mmr_encoder_forward_pixels" in native.lib().mmr_last_error()


def test_vit_b32_from_a_clip_model(enc_mod, native, vit_b32, vit_b32_gpu, b32_enc):
    """from_hf_clip_vision on a CLIPModel (the module the reference loads) takes the vision tower and visual_projection:
    the same weights as the CLIPVisionModelWithProjection give bit-identical embeddings, within TOL of torch.  A text
    encoder refuses pixels."""
    from transformers import CLIPConfig, CLIPModel, CLIPTextConfig, CLIPTextModelWithProjection
    clip = CLIPModel(CLIPConfig(text_config=dict(num_hidden_layers=1), vision_config=vit_b32.config.to_dict()))
    clip.vision_model.load_state_dict(vit_b32.vision_model.state_dict())
    clip.visual_projection.load_state_dict(vit_b32.visual_projection.state_dict())
    enc = enc_mod.DeviceEncoder.from_hf_clip_vision(clip.eval())
    px = _pixels(8, 224, seed=80)
    got = enc.forward_pixels(px)
    assert torch.equal(got, b32_enc.forward_pixels(px))
    with torch.no_grad(), _no_tf32():
        feats = clip.cuda().get_image_features(pixel_values=px.cuda())
        feats = feats if torch.is_tensor(feats) else feats.pooler_output      # transformers 5 returns the projected output here
        want = F.normalize(feats, dim=1)
    assert (got - want).abs().max().item() <= TOL
    enc.close()
    text = enc_mod.DeviceEncoder.from_hf_clip(CLIPTextModelWithProjection(CLIPTextConfig(num_hidden_layers=1)))
    out = torch.empty(1, 512, device="cuda")
    rc = native.lib().mmr_encoder_forward_pixels(text._handle, px.cuda().data_ptr(), 1, out.data_ptr(), None)
    assert rc == 1 and b"takes token ids" in native.lib().mmr_last_error()
    text.close()


def test_vit_b16_shape_matches_fp32_torch(enc_mod):
    """ViT-B/16: 197 tokens per image (attention_kernel<64> near its 330-token limit) and a patch GEMM with K = 768."""
    model = _vision_model(12, patch_size=16)
    enc = enc_mod.DeviceEncoder.from_hf_clip_vision(model)
    px = _pixels(2, 224, seed=16)
    got = enc.forward_pixels(px)
    want = _reference(model.cuda(), px)
    assert (got - want).abs().max().item() <= TOL
    enc.close()


@pytest.mark.parametrize("P,S,B", ((32, 224, 3), (16, 224, 2), (16, 64, 37)))
def test_patch_front_end_matches_fp64(native, P, S, B):
    """mmr_debug_enc_patch_embed: patchify -> patch GEMM -> class token + positions + pre-LayerNorm, the forward pass's
    launches.  The patch matrix is bf16(F.unfold(pixels)) in (c, kh, kw) column order, bit for bit.  The GEMM output
    against float64 on the bf16 operands: products of bf16 values are exact in fp32, so only the K-term fp32 sum errs,
        |e - e_ref| <= d_e = 2 (K + 2) u |X| |W|^T                                     (DESIGN §2, no bias).
    The LayerNorm input v = e + pos adds one rounding: |v - v_ref| <= d = d_e + u |v_ref| (row 0, the class token: u |v_ref|).
    To first order LayerNorm moves by rstd (d_c - mean(d) - x^_c mean(x^ d)) under an input error d, and mean|x^| <= 1, so
    the propagated error is at most |g_c| rstd (d_c + max(d) (1 + |x^_c|)); with the kernel's own LayerNorm bound (DESIGN §2)
        |x - x_ref| <= 1.01 |g| rstd (d + max(d) (1 + |x^|)) + |g| rstd (H/32 + 6) u mean|v| + (H/32 + 16) u |g x^| + 2 u |b|."""
    H, Cc = 768, 3
    np_ = (S // P) ** 2
    T, K = np_ + 1, Cc * P * P
    g = torch.Generator(device="cuda").manual_seed(P * 1000 + B)
    px = torch.randn(B, Cc, S, S, generator=g, device="cuda") * 1.5
    w16 = (torch.randn(H, K, generator=g, device="cuda") * 0.05).to(torch.bfloat16)
    cls = torch.randn(H, generator=g, device="cuda") * 0.5
    pos = torch.randn(T, H, generator=g, device="cuda") * 0.3
    lg = 1.0 + 0.1 * torch.randn(H, generator=g, device="cuda")
    lb = 0.05 * torch.randn(H, generator=g, device="cuda")
    eps = 1e-5
    p16 = torch.full((B * np_, K), float("nan"), device="cuda", dtype=torch.bfloat16)
    pout = torch.full((B * np_, H), float("nan"), device="cuda")
    x = torch.full((B * T, H), float("nan"), device="cuda")
    native.check(native.lib().mmr_debug_enc_patch_embed(H, Cc, S, P, B, px.data_ptr(), w16.data_ptr(), cls.data_ptr(), pos.data_ptr(),
                                                        lg.data_ptr(), lb.data_ptr(), eps, p16.data_ptr(), pout.data_ptr(),
                                                        x.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    want16 = F.unfold(px, P, stride=P).transpose(1, 2).reshape(B * np_, K).to(torch.bfloat16)
    assert torch.equal(p16.view(torch.int16), want16.view(torch.int16)), "patch matrix != bf16(unfold(pixels))"

    # fp64 reference from the convolution itself on the bf16 pixels and weights
    conv = F.conv2d(px.to(torch.bfloat16).double(), w16.double().reshape(H, Cc, P, P), stride=P)       # [B, H, gh, gw]
    e_ref = conv.flatten(2).transpose(1, 2).reshape(B * np_, H)
    d_e = 2 * (K + 2) * U * (want16.double().abs() @ w16.double().abs().t())
    assert not bool(((pout.double() - e_ref).abs() > d_e).any()), float(((pout.double() - e_ref).abs() - d_e).max())

    v_ref = torch.cat([cls.double().expand(B, 1, H), e_ref.reshape(B, np_, H)], 1) + pos.double()        # [B, T, H]
    d = torch.cat([torch.zeros(B, 1, H, device="cuda", dtype=torch.float64), d_e.reshape(B, np_, H)], 1) + U * v_ref.abs()
    mean = v_ref.mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(((v_ref - mean) ** 2).mean(-1, keepdim=True) + eps)
    xh = (v_ref - mean) * rstd
    ref = xh * lg.double() + lb.double()
    ga = lg.double().abs()
    bound = (1.01 * ga * rstd * (d + d.amax(-1, keepdim=True) * (1 + xh.abs()))
             + ga * rstd * (H / 32 + 6) * U * v_ref.abs().mean(-1, keepdim=True) + (H / 32 + 16) * U * (lg.double() * xh).abs()
             + 2 * U * lb.double().abs())
    err = (x.double().reshape(B, T, H) - ref).abs()
    assert not bool((err > bound).any()), float((err - bound).max())


def _token_tile(M, N, sms):
    """enc_token_tile_for (csrc/mmr_encoder.cu): the tile by token count, halved while the grid would leave SMs idle."""
    nt = 64 if M <= 1024 else (128 if M <= 4096 else 256)
    while nt > 64 and (N // 128) * ((M + nt - 1) // nt) < (1 if nt == 256 else 2) * sms:
        nt //= 2
    return nt


def test_image_embedding_does_not_depend_on_its_batch(native, b32_enc):
    """An image's embedding is bit-identical alone and inside batches of 7, 48 and 200 images, whose QKV / FFN1 GEMMs run on
    the 64-, 128- and 256-token tiles (50 tokens per image; the tiles come from the library's rule and the device's SM
    count, and the test requires each of the three to occur)."""
    n = C.c_int(0)
    native.check(native.lib().mmr_device_sm_count(0, C.byref(n)))
    tiles = {b: _token_tile(b * 50, min(3 * 768, 3072), n.value) for b in (7, 48, 200)}
    assert sorted(tiles.values()) == [64, 128, 256], tiles
    img = _pixels(1, 224, seed=4242)
    alone = b32_enc.forward_pixels(img).cpu()
    for b in (7, 48, 200):
        px = _pixels(b, 224, seed=b + 1)
        px[b // 3] = img[0]
        batch = b32_enc.forward_pixels(px).cpu()
        assert torch.equal(batch[b // 3], alone[0]), (b, tiles[b], float((batch[b // 3] - alone[0]).abs().max()))


def _pil_images(sizes, seed):
    from PIL import Image
    rng = np.random.default_rng(seed)
    out = []
    for w, h in sizes:
        base = rng.integers(0, 256, size=(1, 1, 3))
        noise = rng.integers(-80, 80, size=(h, w, 3))
        out.append(Image.fromarray(np.clip(base + noise, 0, 255).astype(np.uint8), "RGB"))
    return out


def test_image_encoder_matches_processor_and_torch(enc_mod, vit_b32_gpu, b32_enc):
    """ImageEncoder = embed_images_batch: the caller's CLIPImageProcessor (resize, centre crop, normalise) on the host, the
    tower on the device; PIL images of several sizes and aspect ratios.  Micro-batching does not change a row."""
    from transformers import CLIPImageProcessor
    proc = CLIPImageProcessor()
    enc = enc_mod.ImageEncoder(proc, b32_enc)
    images = _pil_images([(224, 224), (640, 480), (100, 300), (1000, 57), (33, 33), (224, 225), (512, 512)], seed=3)
    got = enc(images)
    assert isinstance(got, np.ndarray) and got.dtype == np.float32 and got.shape == (7, 512)
    want = _reference(vit_b32_gpu, proc(images=images, return_tensors="pt")["pixel_values"]).cpu().numpy()
    assert np.abs(got - want).max() <= TOL, np.abs(got - want).max()
    np.testing.assert_allclose(np.linalg.norm(got, axis=1), 1.0, atol=1e-5)
    assert np.array_equal(enc(images, batch_size=3), got)
    dev = enc.encode_device(images[:2])
    assert dev.is_cuda and torch.equal(dev.cpu(), torch.from_numpy(got[:2]))
    assert enc([]).shape == (0, 512) and enc([]).dtype == np.float32


def test_ingest_then_search_finds_each_image(enc_mod, b32_enc):
    """The ingest path end to end: 2,000 images -> ImageEncoder -> B200Store.upsert_image_vectors; the embeddings of 16 of
    them, searched with search_image, return each image as its own top hit with score >= 1 - 1e-3."""
    from transformers import CLIPImageProcessor
    mmr = importlib.import_module(PKG)
    store_mod = importlib.import_module(PKG + ".store")
    enc = enc_mod.ImageEncoder(CLIPImageProcessor(), b32_enc)
    n = 2000
    images = _pil_images([(224, 224)] * n, seed=99)
    emb = enc(images, batch_size=256)
    assert emb.shape == (n, 512)
    store = mmr.B200Store()
    store.upsert_image_vectors([store_mod.VectorRow(chunk_id=f"img{i}", user_id="u", document_id="d", modality="image",
                                                    embedding=emb[i], meta={}) for i in range(n)])
    for i in np.random.default_rng(5).choice(n, 16, replace=False):
        hits = store.search_image("u", emb[i], 5)
        assert hits[0]["chunk_id"] == f"img{i}", (i, hits[:2])
        assert hits[0]["score"] >= 1 - 1e-3, (i, hits[0]["score"])
