"""Operator-level parity of the CUDA kernels (through the C ABI) against plain PyTorch fp32 references."""
import pytest
import torch

pytestmark = pytest.mark.gpu

ACTS = {
    "none": lambda x: x,
    "relu": torch.relu,
    "quick_gelu": lambda x: x * torch.sigmoid(1.702 * x),
    "gelu_new": lambda x: 0.5 * x * (1.0 + torch.tanh(0.7978845608028654 * (x + 0.044715 * x ** 3))),
    "gelu": torch.nn.functional.gelu,
    "tanh": torch.tanh,
}


def _ref_linear(x, w, bias, act, residual):
    y = x.float() @ w.float().t()
    if bias is not None:
        y = y + bias
    y = ACTS[act](y)
    if residual is not None:
        y = y + residual
    return y


# (tokens, features, K, orientation, bn, split_k)
LINEAR_CASES = [
    (128, 256, 64, 1, 0, 0),
    (128, 128, 128, 1, 128, 0),
    (2560, 4800, 1600, 1, 256, 0),   # GPT2-XL prefill c_attn
    (2560, 1600, 6400, 1, 0, 0),     # c_proj of the MLP, auto split
    (64, 4800, 1600, 2, 64, 1),      # decode, swapped orientation
    (64, 4800, 1600, 0, 0, 0),       # decode, auto
    (64, 1600, 6400, 2, 64, 4),      # split-K, swapped
    (1, 768, 768, 0, 0, 0),          # batch 1
    (5, 2304, 768, 2, 32, 3),
    (256, 50257, 128, 2, 256, 1),    # lm_head shape, swapped with odd vocab
    (200, 1000, 512, 1, 128, 0),
    (49, 768, 3072, 0, 0, 0),        # ViT patch embed at batch 1
    # persistent kernel (normal orientation): auto and forced tile widths, ragged edges, many tiles per CTA
    (300, 520, 256, 1, 0, 0),        # ragged rows / features
    (300, 520, 256, 1, 64, 0),
    (1000, 100, 128, 1, 96, 0),
    (130, 96, 64, 1, 0, 0),
    (2560, 4800, 1600, 1, 0, 0),     # GPT2-XL prefill c_attn
    (3200, 768, 768, 1, 0, 0),       # ViT attention projection at batch 64
    (5120, 6400, 1600, 1, 224, 0),   # mapper MLP, 5 stages
    (20000, 512, 192, 4, 32, 0),     # 2512 tiles: 17 per CTA, both accumulator buffers, ring wrap-around
    # CTA-pair kernel (cta_group::2, 256-token tiles)
    (300, 520, 256, 3, 64, 0),
    (2560, 4800, 1600, 3, 256, 0),
    (3200, 768, 768, 3, 96, 0),      # 12.5 pair tiles: the last peer CTA is entirely out of range
    (1000, 100, 128, 3, 128, 0),
    (20000, 512, 192, 3, 32, 0),
    (5120, 6400, 1600, 3, 224, 0),
]


@pytest.mark.parametrize("tokens,features,K,orientation,bn,split_k", LINEAR_CASES)
def test_linear_matches_torch(tiny_engine, tokens, features, K, orientation, bn, split_k):
    g = torch.Generator().manual_seed(tokens * 131 + features)
    x = torch.randn(tokens, K, generator=g).bfloat16()
    w = (torch.randn(features, K, generator=g) * 0.05).bfloat16()
    bias = torch.randn(features, generator=g)
    res = torch.randn(tokens, features, generator=g)
    for act, use_res, out_dtype in (("none", False, torch.float32), ("gelu_new", True, torch.float32),
                                    ("relu", False, torch.bfloat16)):
        out = tiny_engine.op_linear(x, w, bias, act, res if use_res else None, out_dtype, orientation, bn, split_k)
        ref = _ref_linear(x.cuda(), w.cuda(), bias.cuda(), act, res.cuda() if use_res else None)
        tol = 2e-2 if out_dtype == torch.bfloat16 else 2e-3
        err = (out.float() - ref).abs().max().item()
        scale = ref.abs().max().item()
        assert err <= tol * scale + 1e-5, (act, err, scale)


def test_linear_split_k_needs_the_swapped_orientation(tiny_engine):
    """Split-K exists only in the one-tile kernel (weights on the 128-row side): asked for with tokens on that side, it is
    rejected, not run some other way, and the context keeps working."""
    g = torch.Generator().manual_seed(7)
    x = torch.randn(300, 256, generator=g).bfloat16()
    w = (torch.randn(520, 256, generator=g) * 0.05).bfloat16()
    with pytest.raises(RuntimeError, match="split-K"):
        tiny_engine.op_linear(x[:64], w, orientation=1, split_k=2)
    with pytest.raises(RuntimeError, match="split-K"):
        tiny_engine.op_linear(x, w, orientation=0, split_k=2)     # 300 tokens: normal orientation
    out = tiny_engine.op_linear(x, w)
    ref = _ref_linear(x.cuda(), w.cuda(), None, "none", None)
    assert (out - ref).abs().max().item() <= 2e-3 * ref.abs().max().item()


def test_linear_no_bias_in_place_residual(tiny_engine):
    g = torch.Generator().manual_seed(5)
    x = torch.randn(96, 192, generator=g).bfloat16()
    w = (torch.randn(320, 192, generator=g) * 0.05).bfloat16()
    res = torch.randn(96, 320, generator=g)
    out = tiny_engine.op_linear(x, w, None, "none", res)
    ref = _ref_linear(x.cuda(), w.cuda(), None, "none", res.cuda())
    assert (out - ref).abs().max().item() < 2e-3 * ref.abs().max().item()


@pytest.mark.parametrize("rows,d", [(1, 128), (77, 768), (300, 1600), (64, 4096)])
def test_layernorm(tiny_engine, rows, d):
    g = torch.Generator().manual_seed(d)
    x = torch.randn(rows, d, generator=g) * 3 + 0.5
    gamma, beta = torch.randn(d, generator=g), torch.randn(d, generator=g)
    y = tiny_engine.op_layernorm(x, gamma, beta, 1e-5)
    ref = torch.nn.functional.layer_norm(x, (d,), gamma, beta, 1e-5).cuda()
    assert (y.float() - ref).abs().max().item() <= 2e-2 * ref.abs().max().item()


def _ref_attention(qkv, B, S, H, hd, causal):
    d = H * hd
    q, k, v = qkv.float().view(B, S, 3, H, hd).unbind(2)
    att = torch.einsum("bnhd,bmhd->bhnm", q, k) * hd ** -0.5
    if causal:
        m = torch.ones(S, S, dtype=torch.bool, device=qkv.device).tril()
        att = att.masked_fill(~m, float("-inf"))
    att = att.softmax(-1)
    return torch.einsum("bhnm,bmhd->bnhd", att, v).reshape(B * S, d)


@pytest.mark.parametrize("B,S,H,hd,causal", [(2, 50, 12, 64, False), (3, 80, 8, 200, False), (2, 20, 8, 96, False),
                                             (4, 40, 25, 64, True), (1, 80, 8, 512, False), (2, 41, 4, 256, True),
                                             # head_dim above 256 (the 4096-wide mapper): Q fragments streamed, ragged S / head_dim, causal
                                             (2, 33, 4, 512, True), (1, 80, 2, 320, False), (3, 7, 2, 512, False),
                                             # head_dim 64, S <= 64: the tcgen05 / TMEM kernel (full tile, one row, ragged)
                                             (1, 64, 3, 64, True), (3, 1, 2, 64, True), (2, 17, 5, 64, False), (2, 64, 2, 64, False)])
def test_attention(tiny_engine, B, S, H, hd, causal):
    g = torch.Generator().manual_seed(S * hd)
    qkv = torch.randn(B * S, 3 * H * hd, generator=g).bfloat16().cuda()
    out = tiny_engine.op_attention(qkv, B, S, H, hd, causal)
    ref = _ref_attention(qkv, B, S, H, hd, causal)
    assert (out.float() - ref).abs().max().item() <= 1.5e-2 * ref.abs().max().item() + 1e-3


def test_argmax_lowest_index_on_ties(tiny_engine):
    g = torch.Generator().manual_seed(0)
    logits = torch.randn(7, 50257, generator=g)
    logits[3, 100] = logits[3, 40000] = 99.0
    nxt = tiny_engine.argmax(logits)
    ref = logits.argmax(-1)
    ref[3] = 100
    assert nxt.cpu().tolist() == ref.tolist()


def test_argmax_strided_and_unaligned_rows(tiny_engine):
    """Rows that start on a 16-byte boundary take the float4 path, others the scalar one; ties inside one float4 and the
    scalar tail (V % 4) follow the same lowest-index rule."""
    g = torch.Generator().manual_seed(1)
    for V, ld in ((50257, 50257), (50257, 50264), (50400, 50400), (1027, 1031)):
        buf = torch.randn(9, ld, generator=g).cuda()
        logits = buf[:, :V]
        logits[2, 5] = logits[2, 6] = 50.0          # tie inside one float4
        logits[4, V - 1] = 60.0                     # scalar tail
        logits[6, 17] = logits[6, V - 2] = 70.0
        nxt = tiny_engine.argmax(logits)
        ref = logits.argmax(-1)
        ref[2], ref[4], ref[6] = 5, V - 1, 17
        assert nxt.cpu().tolist() == ref.cpu().tolist()


def test_cross_entropy_at_full_vocabulary(tiny_engine):
    """ccb_cross_entropy against torch's F.cross_entropy (what the reference calls, model.py:210) at V = 50257 on 64 x 20
    target rows: mean within 1e-5 relative, per-row within 1e-4 absolute; ignored rows, a row map, all rows ignored (NaN)."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(2)
    V, rows = 50257, 1280
    logits = (3.0 * torch.randn(rows + 64, V, generator=g)).cuda()
    targets = torch.randint(0, V, (rows,), generator=g).cuda()
    targets[::7] = 0
    row_map = torch.randperm(rows + 64, generator=g)[:rows].cuda()
    loss, row_loss, n = tiny_engine.cross_entropy(logits, targets, ignore_index=0, row_map=row_map)
    picked = logits[row_map]
    want = F.cross_entropy(picked, targets, ignore_index=0)
    want_rows = F.cross_entropy(picked, targets, ignore_index=0, reduction="none")
    assert abs(float(loss) - float(want)) <= 1e-5 * abs(float(want))
    assert (row_loss - want_rows).abs().max().item() <= 1e-4
    assert int(n) == int((targets != 0).sum())
    loss2, _, _ = tiny_engine.cross_entropy(logits[:rows], targets, ignore_index=0)
    assert abs(float(loss2) - float(F.cross_entropy(logits[:rows], targets, ignore_index=0))) <= 1e-5 * abs(float(want))
    loss3, _, n3 = tiny_engine.cross_entropy(logits[:4], torch.zeros(4, dtype=torch.int64), ignore_index=0)
    assert torch.isnan(loss3).item() and int(n3) == 0
    # bit-identical run to run (row-order sum by one CTA)
    again, _, _ = tiny_engine.cross_entropy(logits, targets, ignore_index=0, row_map=row_map)
    assert float(again) == float(loss)
