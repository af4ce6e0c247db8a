"""The persistent decode-step kernel (csrc/decode_mega.cu) against the operator-per-kernel decode chain and the
reference-generated golden captions, through the C ABI.

Both paths round activations to bf16 at the same points and accumulate in fp32; they differ only in the order of the
fp32 split-K sums, so intermediate buffers agree to a few bf16 ulps (tolerance 2e-2 * max|ref|, the north-star
tolerance) and greedy / beam token sequences on the fixtures are identical.
"""
import ctypes as C
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
TOL = 2e-2


def tiny_engine(max_images=32, page_tokens=4):
    import clipcap_b200 as cc
    fx = torch.load(os.path.join(GOLDEN, "tiny_gpt2.pt"), weights_only=False)
    cfg = cc.EngineConfig(
        lm_arch="gpt2", lm_d=fx["d"], lm_layers=2, lm_heads=fx["heads"], lm_vocab=fx["V"], lm_n_pos=64,
        map_dim_clip=fx["dim_clip"], map_clip_len=fx["CL"], map_prefix_len=fx["P"], map_heads=fx["map_heads"],
        map_layers=2, vit_image=fx["vit_image"], vit_patch=fx["vit_patch"], vit_width=fx["vit_width"],
        vit_layers=fx["vit_layers"], vit_heads=fx["vit_heads"], vit_out=fx["dim_clip"], max_images=max_images, max_beam=5,
        max_ctx=32, page_tokens=page_tokens)
    eng = cc.Engine(cfg)
    eng.load_state_dict(fx["sd_lm"], prefix="language_model.")
    eng.load_state_dict(fx["sd_mapper"], prefix="clip_project.")
    eng.load_state_dict(fx["sd_vit"], prefix="visual.")
    eng.check_weights()
    return eng, fx


def set_mega(eng, on):
    return eng.lib.ccb_debug_set_mega(eng._h, 1 if on else 0)


def grab(eng, which, numel, dtype):
    out = torch.empty(numel, dtype=dtype, device="cuda")
    assert eng.lib.ccb_debug_copy_buffer(eng._h, which, C.c_void_p(out.data_ptr()), out.numel() * out.element_size(), None) == 0
    torch.cuda.synchronize()
    return out.float().cpu()


def test_first_call_of_a_fresh_engine_matches_golden_greedy():
    """The very first generate call (graph capture + cold caches; idle CTAs race ahead of the busy ones on a model this
    small) must already be right: regression test for the barrier protocol."""
    eng, fx = tiny_engine()
    assert set_mega(eng, True) == 1
    p = eng.gen_params("greedy", 10, stop_token=fx["stop_id"], max_stops=1)
    tokens, lengths, _ = eng.generate(fx["prefix"].cuda(), p)
    tokens, lengths = tokens.cpu(), lengths.cpu()
    for i, want in enumerate(fx["greedy"]):
        assert tokens[i, :int(lengths[i])].tolist() == want
    eng.close()


@pytest.mark.parametrize("mode,kw", [("greedy", {}), ("beam", {"beam_size": 5}), ("beam", {"beam_size": 3}),
                                     ("sample", {"top_p": 0.9, "seed": 7})])
@pytest.mark.parametrize("n_images", [1, 3, 32])
def test_tokens_identical_to_operator_chain(mode, kw, n_images):
    eng, fx = tiny_engine()
    prefix = fx["prefix"].cuda()
    prefix = prefix.repeat((n_images + 2) // 3, 1, 1)[:n_images].contiguous()
    prefix = prefix + 0.05 * torch.arange(n_images, device="cuda").view(-1, 1, 1)   # distinct rows
    p = eng.gen_params(mode, 12, stop_token=-1, max_stops=0, **kw)
    out = {}
    for on in (True, False):
        set_mega(eng, on)
        t, l, s = eng.generate(prefix, p)
        torch.cuda.synchronize()
        out[on] = (t.cpu(), l.cpu())
    if mode == "sample":
        # identical noise, but the logits of the two paths differ in the last fp32 / bf16 bits (order of the split-K
        # sums): argmax(p / q) flips on near-ties and the row then continues differently.  Bit-exactness of the sampler
        # itself given identical logits is pinned in test_gpu_parity.py; here most rows must agree.
        same = (out[True][0] == out[False][0]).all(dim=-1).float().mean().item()
        assert same >= 0.75, same
    else:
        assert torch.equal(out[True][0], out[False][0])
        assert torch.equal(out[True][1], out[False][1])
    eng.close()


@pytest.mark.parametrize("page_tokens", [1, 4, 16])
def test_activations_after_one_step_match_operator_chain(page_tokens):
    eng, fx = tiny_engine(page_tokens=page_tokens)
    prefix = fx["prefix"].cuda()
    R, d = prefix.shape[0], fx["d"]
    p = eng.gen_params("greedy", 2, stop_token=-1, max_stops=0)   # prefill + exactly one decode step
    bufs = {}
    for on in (True, False):
        set_mega(eng, on)
        eng.generate(prefix, p)
        torch.cuda.synchronize()
        bufs[on] = {"h": grab(eng, 0, R * d, torch.float32), "x": grab(eng, 1, R * d, torch.bfloat16),
                    "att": grab(eng, 2, R * d, torch.bfloat16), "mlp": grab(eng, 3, R * 4 * d, torch.bfloat16),
                    "logits": grab(eng, 4, R * ((fx["V"] + 63) // 64 * 64), torch.float32).view(R, -1)[:, :fx["V"]]}
    for name in bufs[True]:
        a, b = bufs[True][name], bufs[False][name]
        assert (a - b).abs().max().item() <= TOL * max(b.abs().max().item(), 1e-6), name
    eng.close()


def test_gpt2_xl_shaped_layers_match_operator_chain():
    """d = 1600, 25 heads (every CTA owns units of every GEMM, 13 split-K slots for c_proj), 2 layers, 64 + 1 rows."""
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    cfg = cc.EngineConfig(lm_layers=2, map_kind="none", vit=False, max_images=80, max_beam=1, max_ctx=64, lm_vocab=2048)
    eng = cc.Engine(cfg)
    eng.load_state_dict(synthetic.lm_state_dict(cfg, 1234, "cuda"), prefix="language_model.")
    eng.check_weights()
    torch.manual_seed(3)
    for rows in (64, 65, 7):
        embeds = (0.5 * torch.randn(rows, 9, cfg.lm_d, device="cuda")).contiguous()
        # activations after exactly one decode step (before any near-tie can send a row down another path)
        p1 = eng.gen_params("greedy", 2, stop_token=-1, max_stops=0)
        buf = {}
        for on in (True, False):
            assert set_mega(eng, on) == 1
            eng.generate(embeds, p1)
            torch.cuda.synchronize()
            buf[on] = (grab(eng, 1, rows * cfg.lm_d, torch.bfloat16), grab(eng, 0, rows * cfg.lm_d, torch.float32))
        for k in range(2):
            assert (buf[True][k] - buf[False][k]).abs().max().item() <= TOL * buf[False][k].abs().max().item(), (rows, k)
        # tokens over several steps: random-init logits have near-ties (top-2 margins below the bf16 noise of the
        # activations, BASELINE.md section 2), so a row may flip and then continues differently
        p6 = eng.gen_params("greedy", 6, stop_token=-1, max_stops=0)
        tok = {}
        for on in (True, False):
            set_mega(eng, on)
            t, l, _ = eng.generate(embeds, p6)
            torch.cuda.synchronize()
            tok[on] = t.cpu()
        same = (tok[True] == tok[False]).all(dim=-1).float().mean().item()
        assert same >= 0.95, (rows, same)
    eng.close()


@pytest.mark.parametrize("rows", [16, 33, 100, 128, 129, 160, 176, 208, 255, 256])
def test_row_counts_across_the_ring_configurations(rows):
    """GPT2-XL-shaped layers at row counts that switch the kernel's shared-memory plan: X ring of 8 / 4 / 3 tiles, slot
    pairs vs single slots (> 128 rows), helper-warp staging behind vs inside the ring (> ~170 rows).  Activations after one
    decode step against the operator chain, twice (the second pass must reproduce the first bit for bit)."""
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    cfg = cc.EngineConfig(lm_layers=3, map_kind="none", vit=False, max_images=256, max_beam=1, max_ctx=64, lm_vocab=2048)
    eng = cc.Engine(cfg)
    eng.load_state_dict(synthetic.lm_state_dict(cfg, 1234, "cuda"), prefix="language_model.")
    eng.check_weights()
    torch.manual_seed(rows)
    embeds = (0.5 * torch.randn(rows, 21, cfg.lm_d, device="cuda")).contiguous()
    p1 = eng.gen_params("greedy", 2, stop_token=-1, max_stops=0)
    buf = {}
    for tag, on in (("mega", True), ("chain", False), ("mega_again", True)):
        assert set_mega(eng, on) == 1
        eng.generate(embeds, p1)
        torch.cuda.synchronize()
        buf[tag] = (grab(eng, 1, rows * cfg.lm_d, torch.bfloat16), grab(eng, 0, rows * cfg.lm_d, torch.float32))
    for k in range(2):
        assert (buf["mega"][k] - buf["chain"][k]).abs().max().item() <= TOL * buf["chain"][k].abs().max().item(), (rows, k)
        assert torch.equal(buf["mega"][k], buf["mega_again"][k]), (rows, k)
    eng.close()


def test_gptj_is_served_by_the_operator_chain():
    import clipcap_b200 as cc
    fx = torch.load(os.path.join(GOLDEN, "tiny_gptj.pt"), weights_only=False)
    cfg = cc.EngineConfig(lm_arch="gptj", lm_d=fx["d"], lm_layers=2, lm_heads=fx["heads"], lm_vocab=fx["V"], lm_n_pos=64,
                          lm_rotary_dim=fx["rotary_dim"], map_kind="none", vit=False, max_images=4, max_ctx=32)
    eng = cc.Engine(cfg)
    assert set_mega(eng, True) == 0     # parallel-block / rotary layers are not covered by the persistent kernel
    eng.close()
