"""Host side of the device encoders: HF state_dict -> C-ABI weight names (no GPU needed)."""
import importlib

import torch

PKG = "multimodal-rag-for-image-text-search_b200"
enc_mod = importlib.import_module(PKG + ".encoders")


def test_bert_and_cross_encoder_weight_names_and_shapes():
    from transformers import BertConfig, BertForSequenceClassification, BertModel
    cfg = BertConfig(vocab_size=100, hidden_size=384, num_hidden_layers=2, num_attention_heads=12, intermediate_size=1536,
                     max_position_embeddings=64, num_labels=1)
    w = enc_mod.hf_bert_weights(BertModel(cfg, add_pooling_layer=False))
    assert w["word_emb"].shape == (100, 384) and w["pos_emb"].shape == (64, 384) and w["type_emb"].shape == (2, 384)
    assert w["L1.qkv_w"].shape == (1152, 384) and w["L1.qkv_b"].shape == (1152,)
    assert w["L0.fc1_w"].shape == (1536, 384) and w["L0.fc2_w"].shape == (384, 1536) and "cls_w" not in w
    assert len(w) == 5 + 2 * 12
    model = BertForSequenceClassification(cfg)
    w = enc_mod.hf_bert_weights(model)
    assert w["pooler_w"].shape == (384, 384) and w["cls_w"].shape == (384,) and w["cls_b"].shape == (1,)
    q = model.state_dict()["bert.encoder.layer.0.attention.self.key.weight"]
    assert torch.equal(w["L0.qkv_w"][384:768], q)              # stacked q | k | v


def test_clip_text_weight_names_and_shapes():
    from transformers import CLIPTextConfig, CLIPTextModelWithProjection
    cfg = CLIPTextConfig(num_hidden_layers=2, vocab_size=500)
    w = enc_mod.hf_clip_text_weights(CLIPTextModelWithProjection(cfg))
    assert w["word_emb"].shape == (500, 512) and w["pos_emb"].shape == (77, 512) and w["proj_w"].shape == (512, 512)
    assert w["L1.qkv_w"].shape == (1536, 512) and w["L0.fc1_w"].shape == (2048, 512) and w["final_ln_w"].shape == (512,)
    assert len(w) == 5 + 2 * 12


def test_no_device_no_encoder():
    import pytest
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(Exception):
        enc_mod.DeviceEncoder("minilm", vocab_size=10, hidden=384, layers=1, heads=12, intermediate=1536, max_positions=8)


def test_unsupported_activation_or_position_type_is_refused_before_the_library():
    """The kernels implement erf-GELU (BERT), quick-GELU (CLIP) and absolute positions only; another model must be refused
    with ValueError before any library call (no GPU needed: the check runs first)."""
    import pytest
    from transformers import BertConfig, BertModel, CLIPTextConfig, CLIPTextModelWithProjection
    small = dict(vocab_size=100, hidden_size=384, num_hidden_layers=1, num_attention_heads=12, intermediate_size=1536,
                 max_position_embeddings=64)
    for kw, words in ((dict(hidden_act="gelu_new"), "hidden_act"), (dict(hidden_act="relu"), "hidden_act"),
                      (dict(position_embedding_type="relative_key"), "position_embedding_type"),
                      (dict(position_embedding_type="relative_key_query"), "position_embedding_type")):
        with pytest.raises(ValueError, match=words):
            enc_mod.DeviceEncoder.from_hf_bert(BertModel(BertConfig(**small, **kw), add_pooling_layer=False))
    for act in ("gelu", "gelu_new"):
        with pytest.raises(ValueError, match="hidden_act"):
            enc_mod.DeviceEncoder.from_hf_clip(CLIPTextModelWithProjection(CLIPTextConfig(num_hidden_layers=1, vocab_size=100,
                                                                                           hidden_act=act)))
    # the supported configs pass the check (and then need the library and a device)
    enc_mod._check_supported(BertConfig(**small), {"gelu"})
    enc_mod._check_supported(CLIPTextConfig(num_hidden_layers=1), {"quick_gelu"})
