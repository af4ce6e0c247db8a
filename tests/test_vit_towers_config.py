"""The OpenAI CLIP tower presets (`EngineConfig.for_clip`) and checkpoint shape inference for the large towers; no GPU."""
import pytest
import torch

# The published OpenAI towers (openai/CLIP clip/model.py build_model; HF openai/clip-vit-* configs):
# (image, patch, vision width, vision layers, projection dim, text width, text layers, text heads)
PUBLISHED = {
    "ViT-B/32": (224, 32, 768, 12, 512, 512, 12, 8),
    "ViT-B/16": (224, 16, 768, 12, 512, 512, 12, 8),
    "ViT-L/14": (224, 14, 1024, 24, 768, 768, 12, 12),
    "ViT-L/14@336px": (336, 14, 1024, 24, 768, 768, 12, 12),
}


@pytest.mark.parametrize("name", sorted(PUBLISHED))
def test_presets_match_the_published_towers(name):
    import clipcap_b200 as cc
    transformers = pytest.importorskip("transformers")
    image, patch, width, layers, proj, t_width, t_layers, t_heads = PUBLISHED[name]
    hf = transformers.CLIPVisionConfig(hidden_size=width, intermediate_size=4 * width, num_hidden_layers=layers,
                                       num_attention_heads=width // 64, image_size=image, patch_size=patch, projection_dim=proj)
    cfg = cc.EngineConfig.for_clip(name)
    assert (cfg.vit_image, cfg.vit_patch, cfg.vit_width, cfg.vit_layers, cfg.vit_heads, cfg.vit_out) == (
        hf.image_size, hf.patch_size, hf.hidden_size, hf.num_hidden_layers, hf.num_attention_heads, hf.projection_dim)
    assert (cfg.text_width, cfg.text_layers, cfg.text_heads, cfg.text_out) == (t_width, t_layers, t_heads, proj)
    assert cfg.map_dim_clip == proj
    n_tok = (image // patch) ** 2 + 1
    assert cc.EngineConfig.for_clip(name, map_kind="transformer_all").map_clip_len == n_tok
    assert cc.EngineConfig.for_clip(name, map_kind="transformer_all", map_clip_len=7).map_clip_len == 7
    assert cc.EngineConfig.for_clip(name).map_clip_len == cc.EngineConfig.map_clip_len


def test_unknown_tower_name():
    import clipcap_b200 as cc
    with pytest.raises(ValueError, match="RN50"):
        cc.EngineConfig.for_clip("RN50")


def _shaped(*shape):
    return torch.zeros(()).expand(*shape)   # shapes are all config_from_checkpoint reads: no storage


def test_config_from_l14_336_all_features_checkpoint():
    """The names and shapes synthetic.vit_state_dict / mapper_state_dict produce for ViT-L/14@336px + an all-features
    mapper on GPT-2 small."""
    import clipcap_b200 as cc
    w, L, S, out, d = 1024, 24, 577, 768, 768
    sd = {"visual.conv1.weight": _shaped(w, 3, 14, 14), "visual.class_embedding": _shaped(w),
          "visual.positional_embedding": _shaped(S, w), "visual.proj": _shaped(w, out)}
    for l in range(L):
        p = "visual.transformer.resblocks.%d." % l
        sd.update({p + "attn.in_proj_weight": _shaped(3 * w, w), p + "mlp.c_fc.weight": _shaped(4 * w, w)})
    sd.update({"clip_project.linear.weight": _shaped(d, out), "clip_project.pos_embeddings": _shaped(S, d),
               "clip_project.prefix_const": _shaped(10, d)})
    sd.update({"language_model.transformer.wte.weight": _shaped(50257, d), "language_model.transformer.wpe.weight": _shaped(1024, d),
               "language_model.transformer.h.0.ln_1.weight": _shaped(d)})
    hp = dict(prefix_size=out, prefix_length=10, clip_prefix_length=10, num_attention_heads=8, num_layers=8,
              use_all_vit_features=True, pos_embeddings=True)
    cfg = cc.model.CLIPCaptionModel.config_from_checkpoint(sd, hp, lm_heads=12)
    assert (cfg.vit_patch, cfg.vit_image, cfg.vit_width, cfg.vit_layers, cfg.vit_heads, cfg.vit_out) == (14, 336, 1024, 24, 16, 768)
    assert (cfg.map_kind, cfg.map_clip_len, cfg.map_dim_clip, cfg.map_prefix_len) == ("transformer_all", 577, 768, 10)
    # without the (optional) pos_embeddings the token count comes from the tower
    del sd["clip_project.pos_embeddings"]
    hp["pos_embeddings"] = False
    assert cc.model.CLIPCaptionModel.config_from_checkpoint(sd, hp, lm_heads=12).map_clip_len == 577
