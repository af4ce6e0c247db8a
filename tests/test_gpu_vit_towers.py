"""The large OpenAI CLIP towers (ViT-L/14: 257 tokens, ViT-L/14@336px: 577) and the all-features mapper over them: the
long-sequence tcgen05 attention kernel (S > 256) against fp32 torch, the towers against the fp32 oracle and HF
CLIPVisionModelWithProjection, the mappers at 577 + P tokens, captions end to end, and the shapes that stay rejected."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import clipcap_oracle as orc  # noqa: E402

pytestmark = pytest.mark.gpu
TOL = 2e-2


def rel(a, b):
    return (a.float() - b.float()).abs().max().item() / max(b.float().abs().max().item(), 1e-9)


def _ref_attention(qkv, B, S, H, hd):
    q, k, v = qkv.float().view(B, S, 3, H, hd).unbind(2)
    att = (torch.einsum("bnhd,bmhd->bhnm", q, k) * hd ** -0.5).softmax(-1)
    return torch.einsum("bhnm,bmhd->bnhd", att, v).reshape(B * S, H * hd)


# (B, S, H, hd): ViT-L/14, ViT-L/14@336px, several key tiles, a ragged last tile, the mapper head dims (GPT2-XL all-features
# 617 tokens / 200, GPT-2 small 267 / 96) and every accumulator width the kernel is built for
LONG_CASES = [(2, 257, 16, 64), (3, 577, 16, 64), (1, 1024, 2, 64), (2, 300, 3, 64), (2, 617, 8, 200), (2, 267, 8, 96),
              (1, 297, 8, 128), (1, 337, 8, 160), (1, 300, 4, 256), (1, 400, 2, 8), (1, 333, 2, 72)]


@pytest.mark.parametrize("B,S,H,hd", LONG_CASES)
def test_long_attention_matches_torch(tiny_engine, B, S, H, hd):
    g = torch.Generator().manual_seed(S * hd + B)
    qkv = torch.randn(B * S, 3 * H * hd, generator=g).bfloat16().cuda()
    out = tiny_engine.op_attention(qkv, B, S, H, hd)
    ref = _ref_attention(qkv, B, S, H, hd)
    assert (out.float() - ref).abs().max().item() <= 1.5e-2 * ref.abs().max().item() + 1e-3


def test_long_attention_rescales_when_the_largest_scores_come_last(tiny_engine):
    """Queries aligned with keys of the last tile: the running maximum grows there and the accumulated O is rescaled."""
    B, S, H, hd = 2, 577, 4, 64
    g = torch.Generator().manual_seed(3)
    qkv = torch.randn(B, S, 3, H, hd, generator=g)
    u = torch.randn(H, hd, generator=g)
    qkv[:, :, 0] = 0.25 * qkv[:, :, 0] + u            # every query leans towards u
    qkv[:, S - 20:, 1] = 3.0 * u                      # ... and the keys of the last tile are u, scaled: the largest scores
    qkv = qkv.reshape(B * S, -1).bfloat16().cuda()
    out = tiny_engine.op_attention(qkv, B, S, H, hd)
    ref = _ref_attention(qkv, B, S, H, hd)
    assert (out.float() - ref).abs().max().item() <= 1.5e-2 * ref.abs().max().item() + 1e-3


def test_long_attention_is_deterministic(tiny_engine):
    g = torch.Generator().manual_seed(11)
    qkv = torch.randn(3 * 577, 3 * 16 * 64, generator=g).bfloat16().cuda()
    a = tiny_engine.op_attention(qkv, 3, 577, 16, 64)
    b = tiny_engine.op_attention(qkv, 3, 577, 16, 64)
    assert torch.equal(a, b)


def test_long_sequences_outside_the_kernel_are_rejected(tiny_engine):
    qkv = torch.randn(300, 3 * 2 * 64).bfloat16().cuda()
    with pytest.raises(RuntimeError, match="attention_prefill"):
        tiny_engine.op_attention(qkv, 1, 300, 2, 64, causal=True)
    qkv512 = torch.randn(300, 3 * 512).bfloat16().cuda()
    with pytest.raises(RuntimeError, match="attention_prefill"):
        tiny_engine.op_attention(qkv512, 1, 300, 1, 512)
    # the context is still usable
    out = tiny_engine.op_attention(qkv, 1, 300, 2, 64)
    assert (out.float() - _ref_attention(qkv, 1, 300, 2, 64)).abs().max().item() <= 2e-2


def test_gptj_all_features_mapper_over_256_tokens_is_rejected_at_creation(tiny_engine):
    import clipcap_b200 as cc
    cfg = cc.EngineConfig.for_clip("ViT-L/14", lm_arch="gptj", lm_d=4096, lm_layers=1, lm_heads=16, lm_vocab=512, lm_n_pos=64,
                                   lm_rotary_dim=64, map_kind="transformer_all", map_prefix_len=40, map_layers=1, max_images=2,
                                   max_ctx=48)
    with pytest.raises(RuntimeError, match="head_dim 512"):
        cc.Engine(cfg)
    qkv = torch.randn(40, 3 * 2 * 64).bfloat16().cuda()
    assert tiny_engine.op_attention(qkv, 1, 40, 2, 64).shape == (40, 128)


@pytest.fixture(scope="module", params=["ViT-L/14", "ViT-L/14@336px"])
def tower(request):
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    cfg = cc.EngineConfig.for_clip(request.param, lm_d=128, lm_layers=1, lm_heads=2, lm_vocab=503, lm_n_pos=64, map_kind="none",
                                   max_images=4, max_ctx=32)
    eng = cc.Engine(cfg)
    sd = synthetic.vit_state_dict(cfg, 1236, "cuda")
    eng.load_state_dict(synthetic.lm_state_dict(cfg, 1234, "cuda"), prefix="language_model.")
    eng.load_state_dict(sd, prefix="visual.")
    eng.check_weights()
    yield request.param, cfg, eng, sd
    eng.close()


def test_tower_matches_oracle(tower):
    from clipcap_b200 import synthetic
    name, cfg, eng, sd = tower
    images = synthetic.synthetic_images(4, cfg, device="cuda")
    n = (cfg.vit_image // cfg.vit_patch) ** 2 + 1
    feat = eng.vit_encode(images)
    ref = orc.vit_forward(sd, images, cfg.vit_heads, cfg.vit_patch)
    assert feat.shape == ref.shape == (4, 768)
    assert rel(feat, ref) <= TOL, name
    toks = eng.vit_encode(images, all_tokens=True)
    ref_toks = orc.vit_forward(sd, images, cfg.vit_heads, cfg.vit_patch, all_tokens=True)
    assert toks.shape == ref_toks.shape == (4, n, 768)
    assert rel(toks, ref_toks) <= TOL, name


def test_l14_336_matches_hf_clip_vision():
    transformers = pytest.importorskip("transformers")
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from make_golden import bf16_round_, export_clip_vision
    hf_cfg = transformers.CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16,
                                           image_size=336, patch_size=14, projection_dim=768, hidden_act="quick_gelu")
    torch.manual_seed(0)
    with torch.device("cuda"):
        hf = bf16_round_(transformers.CLIPVisionModelWithProjection(hf_cfg).float().eval())
    cfg = cc.EngineConfig.for_clip("ViT-L/14@336px", lm_d=128, lm_layers=1, lm_heads=2, lm_vocab=503, lm_n_pos=64, map_kind="none",
                                   max_images=4, max_ctx=32)
    eng = cc.Engine(cfg)
    eng.load_state_dict(synthetic.lm_state_dict(cfg, 1234, "cuda"), prefix="language_model.")
    assert not eng.load_state_dict(export_clip_vision(hf), prefix="visual.")
    eng.check_weights()
    images = synthetic.synthetic_images(4, cfg, device="cuda")
    with torch.no_grad():
        ref = hf(pixel_values=images).image_embeds.float()
    assert rel(eng.vit_encode(images), ref) <= TOL
    eng.close()


@pytest.mark.parametrize("lm_d,P", [(1600, 40), (768, 10)])
def test_all_features_mapper_over_577_tokens(lm_d, P):
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    cfg = cc.EngineConfig.for_clip("ViT-L/14@336px", vit=False, lm_d=lm_d, lm_layers=1, lm_heads=lm_d // 64, lm_vocab=503,
                                   lm_n_pos=128, map_kind="transformer_all", map_prefix_len=P, map_layers=2, max_images=4,
                                   max_ctx=P + 8)
    assert cfg.map_clip_len == 577 and cfg.map_dim_clip == 768
    eng = cc.Engine(cfg)
    sd = synthetic.mapper_state_dict(cfg, 1235, "cuda")
    eng.load_state_dict(synthetic.lm_state_dict(cfg, 1234, "cuda"), prefix="language_model.")
    eng.load_state_dict(sd, prefix="clip_project.")
    eng.check_weights()
    feats = torch.randn(4, 577, 768, generator=torch.Generator().manual_seed(4)).cuda()
    out = eng.map_prefix(feats)
    ref = orc.mapper_all_forward(sd, feats, cfg.map_heads, "relu")
    assert out.shape == ref.shape == (4, P, lm_d)
    assert rel(out, ref) <= TOL
    eng.close()


def test_l14_336_all_features_captions_end_to_end(tmp_path):
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    cfg = cc.EngineConfig.for_clip("ViT-L/14@336px", lm_d=768, lm_layers=2, lm_heads=12, lm_vocab=2048, lm_n_pos=128,
                                   map_kind="transformer_all", map_prefix_len=10, map_layers=2, max_images=4, max_ctx=32)
    eng = cc.Engine(cfg)
    sds = synthetic.load_synthetic(eng)
    images = synthetic.synthetic_images(4, cfg, device="cuda")
    p = eng.gen_params("greedy", 12, stop_token=-1, max_stops=0)
    tokens, _, _ = eng.caption_images(images, p)
    tokens = tokens.cpu()
    step, _, _ = eng.generate(eng.map_prefix(eng.vit_encode(images)), p)
    assert torch.equal(tokens, step.cpu())

    sd = {"language_model." + k: v.cpu() for k, v in sds["lm"].items()}
    sd.update({"clip_project." + k: v.cpu() for k, v in sds["mapper"].items()})
    sd.update({"visual_encoder." + k: v.cpu() for k, v in sds["vit"].items()})
    hp = dict(prefix_size=768, prefix_length=10, clip_prefix_length=10, num_attention_heads=8, num_layers=2, mlp_ratio=4.0,
              act_fn_name="relu", use_all_vit_features=True, pos_embeddings=True)
    path = str(tmp_path / "l14_336_all.ckpt")
    torch.save({"state_dict": sd, "hyper_parameters": hp}, path)
    eng.close()
    model = cc.CLIPCaptionModel.load_from_checkpoint(path, strict=True, lm_heads=12, max_images=4, max_ctx=32)
    c = model.engine.cfg
    assert (c.vit_image, c.vit_patch, c.vit_width, c.vit_layers, c.vit_heads, c.vit_out, c.map_clip_len) == (336, 14, 1024, 24, 16, 768, 577)
    again, _, _ = model.engine.caption_images(images, p)
    assert torch.equal(again.cpu(), tokens)
    model.engine.close()


def test_preprocess_at_336_matches_pil_pipeline(tiny_engine):
    import numpy as np
    from PIL import Image
    from torchvision import transforms
    from torchvision.transforms import InterpolationMode
    tf = transforms.Compose([transforms.Resize(336, interpolation=InterpolationMode.BICUBIC), transforms.CenterCrop(336),
                             transforms.ToTensor(),
                             transforms.Normalize((0.48145466, 0.4578275, 0.40821073), (0.26862954, 0.26130258, 0.27577711))])
    rng = np.random.default_rng(9)
    imgs = [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for h, w in [(480, 640), (640, 480), (336, 336), (1000, 333)]]
    want = torch.stack([tf(Image.fromarray(a)) for a in imgs])
    got = tiny_engine.preprocess_images([torch.from_numpy(a) for a in imgs], n_px=336).cpu()
    assert torch.equal(got, want)
