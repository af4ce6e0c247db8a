"""Every GEMM route and epilogue against a float64 reference, through the pitches, row remap and in-place residuals the
engine uses.

Three kernels run every linear layer: `gemm_bf16_tn_kernel<BN>` (one 128-feature x BN-token tile per CTA, tokens <= 256,
split-K as one cluster reducing over distributed shared memory), `gemm_persist_kernel` (persistent, 128-token tiles) and
`gemm_pair_kernel` (cta_group::2, 256-token tiles).  All three end in the fused epilogue bias -> activation -> residual ->
f32 / bf16 store.  The tests here
  * check the float64 reference and its per-element error bound on the CPU against fp32 matmuls, and that the bound is
    tight enough to see split-K partials staged in bf16;
  * run a covering matrix of forced routes (every tile width and split, persistent and pair widths) x the eight epilogue
    activations x residual none / separate / aliased with out x f32 / bf16 output x pitch variants (lda > K, ldw > K at a
    column offset, ldo > features, an out base 16 but not 32 bytes aligned, ldo % 8 != 0, odd ldo), plus the row remap
    of the all-features mapper, through `op_linear(out=, residual_is_out=, row_remap=)` (ccb_op_linear_ex);
  * run the engine's own GEMM shapes with automatic routing (GPT-2 / GPT2-XL / GPT-J prefill and decode, lm_head, ViT-L/14,
    the MLP and all-features mappers);
  * place every operand and output inside NaN-filled buffers (guard rows, pitch padding, the other column range of a shared
    weight matrix): a stray read turns an output into NaN, every element a call must not write keeps its exact bits,
    rows a remap leaves alone keep their pre-filled values, and the inputs are never written;
  * check two calls are bit-identical, and under torch.profiler which kernel ran with which grid (tiles x splits);
  * probe with exact inputs: small integers (every sum exact in fp32: the output must equal the reference bit for bit),
    one-hot x rows and one-hot w rows at k-block, UMMA-slice and split boundaries, and saturating biases;
  * check that every out-of-range pitch, remap and activation code is refused with a message and launches nothing.

Bound, per output element, from the exact bf16 / f32 inputs:
  e_pre = 2^-18 (sum_k |x_k w_k| + |b|)                       fp32 accumulation, margin for the MMA adder order
  e_y   = L_act e_pre + 2^-20 (|pre| + |act(pre)|)            L_act the activation's Lipschitz constant; __expf / __fdividef
  f32 out adds 2^-23 (|act(pre)| + |r|); bf16 out adds one bf16 ulp of |y|.
"""
import json
import math
import os
import re
import sys
import tempfile
from typing import NamedTuple, Optional

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

gpu = pytest.mark.gpu

ACTS = ("none", "relu", "quick_gelu", "gelu_new", "gelu", "elu", "selu", "tanh")   # epilogue codes 0..7
LIPSCHITZ = {"none": 1.0, "relu": 1.0, "elu": 1.0, "tanh": 1.0, "quick_gelu": 1.13, "gelu_new": 1.13, "gelu": 1.13,
             "selu": 1.76}
SELU_ALPHA, SELU_SCALE = 1.6732632423543772848170429916717, 1.0507009873554804934193349852946
E_ACC = 2.0 ** -18    # fp32 accumulation, relative to sum |x w| + |b|
E_FAST = 2.0 ** -20   # fast exp / divide of the epilogue, relative to |pre| + |act(pre)|
E_F32 = 2.0 ** -23    # the f32 adds of the residual and the stored value
G = 8                 # NaN guard rows above and below every operand / output (keeps every view 16-byte aligned)
NAN = float("nan")
DEV = "cuda"


# ------------------------------------------------------------------------------------------------ float64 reference
def act64(name, z):
    """The epilogue activations in closed form (float64 in, float64 out)."""
    if name == "none":
        return z
    if name == "relu":
        return z.clamp_min(0)
    if name == "quick_gelu":
        return z * torch.sigmoid(1.702 * z)
    if name == "gelu_new":
        return 0.5 * z * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (z + 0.044715 * z ** 3)))
    if name == "gelu":
        return 0.5 * z * (1.0 + torch.erf(z / math.sqrt(2.0)))
    if name == "elu":
        return torch.where(z > 0, z, torch.expm1(z))
    if name == "selu":
        return SELU_SCALE * torch.where(z > 0, z, SELU_ALPHA * torch.expm1(z))
    if name == "tanh":
        return torch.tanh(z)
    raise ValueError(name)


def bf16_ulp(v):
    """One bf16 ulp of v >= 0 (8 significant bits): 2^(e - 8) for v in [2^(e-1), 2^e); 0 for v = 0."""
    _, e = torch.frexp(v)
    return torch.where(v > 0, torch.ldexp(torch.ones_like(v), e - 8), torch.zeros_like(v))


def reference(x, w, bias, act, r, out_bf16):
    """y = act(x w^T + b) + r in float64 from the exact inputs, and the per-element bound of the module docstring.
    x [T, K] bf16, w [F, K] bf16, bias [F] f32 or None, r [T, F] f32 or None (the residual each token row reads)."""
    x64, w64 = x.double(), w.double()
    pre = x64 @ w64.t()
    mag = x64.abs() @ w64.abs().t()
    if bias is not None:
        pre += bias.double()
        mag += bias.double().abs()
    a = act64(act, pre)
    y = a if r is None else a + r.double()
    bound = LIPSCHITZ[act] * E_ACC * mag + E_FAST * (pre.abs() + a.abs())
    bound += E_F32 * (a.abs() + (r.double().abs() if r is not None else 0.0))
    if out_bf16:
        bound += bf16_ulp(y.abs() + bound)
    return y, bound


def remap_rows(T, remap):
    """Output row of every token row: (t // rg_in) * rg_out + rg_off + t % rg_in (identity without a remap)."""
    t = torch.arange(T)
    if not remap:
        return t
    rg_in, rg_out, rg_off = remap
    return (t // rg_in) * rg_out + rg_off + t % rg_in


def ratio(got, y, bound):
    """max |got - y| / bound (an error where the bound is 0 counts as infinite)."""
    err = (got.double() - y).abs()
    r = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
    return float(r.max())


# ------------------------------------------------------------------------------------------------ CPU self-tests
@pytest.mark.parametrize("T,F,K", [(7, 33, 64), (50, 130, 640), (3, 20, 4096), (64, 96, 1600)])
def test_bound_covers_an_fp32_matmul(T, F, K):
    """The bound holds for what a correct fp32 GEMM + fp32 epilogue computes (torch on the CPU, every activation, f32 and
    bf16 output), yet a split-K whose partials were staged in bf16 breaks it."""
    g = torch.Generator().manual_seed(T * 1000 + K)
    x = torch.randn(T, K, generator=g).bfloat16()
    w = (torch.randn(F, K, generator=g) / math.sqrt(K)).bfloat16()
    b = torch.randn(F, generator=g) * 0.5
    r = torch.randn(T, F, generator=g)
    pre32 = x.float() @ w.float().t() + b
    worst = 0.0
    for act in ACTS:
        y32 = act64(act, pre32) + r
        y, bound = reference(x, w, b, act, r, False)
        worst = max(worst, ratio(y32, y, bound))
        y, bound = reference(x, w, b, act, r, True)
        worst = max(worst, ratio(y32.bfloat16(), y, bound))
    assert worst <= 1.0, worst
    if K >= 640:
        half = K // 2
        p0 = (x.float()[:, :half] @ w.float()[:, :half].t()).bfloat16().float()
        p1 = (x.float()[:, half:] @ w.float()[:, half:].t()).bfloat16().float()
        y, bound = reference(x, w, b, "none", None, False)
        assert ratio(p0 + p1 + b, y, bound) > 3.0


def test_reference_activations_and_remap():
    z = torch.tensor([-100.0, -3.0, -0.5, 0.0, 0.5, 3.0, 100.0], dtype=torch.float64)
    F = torch.nn.functional
    assert torch.allclose(act64("gelu", z), F.gelu(z))
    assert torch.allclose(act64("gelu_new", z), F.gelu(z, approximate="tanh"))
    assert torch.allclose(act64("elu", z), F.elu(z))
    assert torch.allclose(act64("selu", z), F.selu(z))
    assert torch.allclose(act64("quick_gelu", z), z * torch.sigmoid(1.702 * z))
    assert remap_rows(7, (3, 5, 1)).tolist() == [1, 2, 3, 6, 7, 8, 11]
    assert bf16_ulp(torch.tensor([1.0, 1.5, 0.75, 0.0], dtype=torch.float64)).tolist() == [2 ** -7, 2 ** -7, 2 ** -8, 0.0]


# ------------------------------------------------------------------------------------------------ cases
class Case(NamedTuple):
    T: int
    F: int
    K: int
    route: tuple              # (orientation, bn, split): 2 = one-tile kernel, 4 = persistent, 3 = pair, 0 = auto
    act: str = "none"
    res: str = "none"         # none | sep (own buffer, ldr != ldo) | alias (read from out, as the residual stream)
    out: str = "f32"          # f32 | bf16
    lda: int = 0              # 0: K
    ldw: int = 0              # 0: K
    woff: int = 0             # column of w inside its [F, ldw] buffer
    ldo: int = 0              # 0: F
    ocol: int = 0             # column of out inside its [rows, ldo] buffer
    ldr: int = 0              # separate residual pitch (0: ldo + 4)
    remap: Optional[tuple] = None
    data: str = "randn"       # randn | int | onehot_x | onehot_w | sat
    bias: bool = True
    tag: str = ""
    expect: Optional[tuple] = None   # literal (kernel, grid) of an auto-routed engine shape


def _r8(n):
    return (n + 7) // 8 * 8


def pitched(T, F, K, route, act="none", res="none", out="f32", pitch="base", **kw):
    """A case with one of the pitch variants laid out."""
    lay = {}
    if pitch == "lda":
        lay = dict(lda=K + 72)
    elif pitch == "ldw":
        lay = dict(ldw=K + 128, woff=64)
    elif pitch == "ldo":
        lay = dict(ldo=_r8(F) + 16)
    elif pitch == "out16":   # base 16 B past a 32-byte boundary on every row (f32: ldo % 8 == 0; bf16: ldo % 16 == 0)
        oc = 4 if out == "f32" else 8
        lay = dict(ocol=oc, ldo=(F + oc + 15) // 16 * 16)
    elif pitch == "scalar":  # ldo % 8 == 4: the persistent epilogue's scalar stores
        lay = dict(ldo=_r8(F) + 4)
    elif pitch == "odd":
        lay = dict(ldo=F + 1 if F % 2 == 0 else F + 2)
    lay.update(kw)
    return Case(T, F, K, route, act, res, out, **lay)


TILE_ROUTES = [(2, bn, s) for bn in (32, 64, 128, 256) for s in (1, 2, 3, 5, 8)]
PERSIST_ROUTES = [(4, bn, 0) for bn in (32, 96, 224, 256)]
PAIR_ROUTES = [(3, bn, 0) for bn in (64, 128, 256)]
ROUTES = TILE_ROUTES + PERSIST_ROUTES + PAIR_ROUTES

TILE_T = {32: [1, 7, 17, 32], 64: [33, 64, 50, 1], 128: [65, 128, 100, 97], 256: [129, 256, 200, 255]}
TILE_F = [20, 128, 129, 257, 300, 1, 384, 200]
# per split: K values whose k-blocks split as forced (never clamped), with uneven last splits (25 = 9+9+7, 23 = 5*4+3,
# 60 = 8*7+4) and one k-block per split (5, 8)
SPLIT_K = {1: [64, 640, 192, 1600], 2: [512, 1600], 3: [1600, 768], 5: [1472, 320], 8: [3840, 512, 4096]}
PERSIST_T = [300, 129, 1000, 50, 257, 128, 1, 640]
PAIR_T = [300, 600, 400, 50, 513, 256, 1000, 129]   # 300 / 600 / 129 / 50: the last pair tile's peer CTA has no rows
PERSIST_F = [520, 100, 33, 256, 1000, 224, 20, 96]
PERSIST_K = [64, 256, 640, 128]
RES_OUT = [("none", "f32"), ("none", "bf16"), ("sep", "f32"), ("sep", "bf16"), ("alias", "f32")]
PITCHES = ["base", "lda", "ldw", "ldo", "out16", "scalar", "odd"]


def _route_label(route):
    o, bn, s = route
    return {2: "tile<%d>/s%d" % (bn, s), 4: "persist<%d>" % bn, 3: "pair<%d>" % bn}.get(o, "auto")


def _matrix():
    cases = []
    for ri, route in enumerate(ROUTES):
        o, bn, s = route
        for ai, act in enumerate(ACTS):
            res, out = RES_OUT[(ri + ai) % len(RES_OUT)]
            n = ai + ri
            if o == 2:
                T, F, K = TILE_T[bn][n % 4], TILE_F[(ai + 3 * ri) % 8], SPLIT_K[s][n % len(SPLIT_K[s])]
                pitch = PITCHES[(ai + 2 * ri) % 7]
            else:
                T = (PERSIST_T if o == 4 else PAIR_T)[n % 8]
                F, K = PERSIST_F[(ai + 3 * ri) % 8], PERSIST_K[n % 4]
                pitch = PITCHES[(ai + 2 * ri) % 6]
            cases.append(pitched(T, F, K, route, act, res, out, pitch, bias=(n % 6 != 5)))
    # the all-features mapper's row remap (visual tokens of every sequence into rows [rg_off, rg_off + rg_in) of rg_out)
    for ri, route in enumerate(PERSIST_ROUTES + PAIR_ROUTES):
        for gi, rg_in in enumerate((50, 197, 257)):
            P = (10, 30, 7)[(ri + gi) % 3]
            off = (0, P // 2, P)[(ri + 2 * gi) % 3]
            res, out = [("alias", "f32"), ("alias", "f32"), ("sep", "bf16"), ("none", "f32")][(ri + gi) % 4]
            F, K = (768, 100, 520)[(ri + gi) % 3], (256, 768, 64)[(2 * ri + gi) % 3]
            act = ACTS[(3 * ri + gi) % 8]
            cases.append(Case(3 * rg_in, F, K, route, act, res, out, remap=(rg_in, rg_in + P, off)))
    return cases


def _probes():
    cases = []
    for ri, route in enumerate(ROUTES):
        o, bn, s = route
        if o == 2:
            T, K = TILE_T[bn][1], max(SPLIT_K[s])
        else:
            T, K = (PERSIST_T if o == 4 else PAIR_T)[ri % 8], 640
        if route in ((2, 32, 8), (4, 96, 0)):
            K = 16384   # |sum| < 2^18: still exact in fp32
        cases.append(Case(T, 200, K, route, res=("sep", "alias")[ri % 2], data="int"))
        cases.append(Case(T, 130, K, route, data="onehot_x"))
        cases.append(Case(T, 300, K, route, data="onehot_w"))
    for route in [(2, 64, 2), (2, 32, 8), (4, 96, 0), (3, 128, 0)]:
        for ai, act in enumerate(ACTS):
            T = min(40, route[1]) if route[0] == 2 else 300
            K = 512 if route[1] != 32 else 3840
            cases.append(Case(T, 150, K, route, act, out=("f32", "bf16")[ai % 2], data="sat"))
    return cases


def _engine_shapes():
    """The engine's GEMMs with automatic routing, at the shapes and pitches engine.cu gives them.  `expect` holds the route
    the B200 (148 SMs) takes where the design documents it."""
    A = (0, 0, 0)
    d2, dx, dj = 768, 1600, 4096
    return [
        Case(200, 3 * d2, d2, A, out="bf16", tag="gpt2 prefill c_attn"),
        Case(200, d2, d2, A, res="alias", tag="gpt2 prefill c_proj"),
        Case(200, 4 * d2, d2, A, "gelu_new", out="bf16", tag="gpt2 prefill c_fc"),
        Case(200, d2, 4 * d2, A, res="alias", tag="gpt2 prefill mlp c_proj"),
        Case(2560, 3 * dx, dx, A, out="bf16", tag="gpt2-xl prefill c_attn"),
        Case(2560, dx, dx, A, res="alias", tag="gpt2-xl prefill c_proj"),
        Case(2560, 4 * dx, dx, A, "gelu_new", out="bf16", tag="gpt2-xl prefill c_fc"),
        Case(2560, dx, 4 * dx, A, res="alias", tag="gpt2-xl prefill mlp c_proj"),
        Case(64, 3 * dx, dx, A, out="bf16", tag="gpt2-xl 64-row decode c_attn",
             expect=("gemm_bf16_tn_kernel<64>", (38, 1, 3))),
        # GPT-J prefill: out_proj and fc_out are the two column ranges of one [d, 5d] matrix
        Case(400, dj, dj, A, res="alias", ldw=5 * dj, bias=False, tag="gptj prefill out_proj"),
        Case(400, dj, 4 * dj, A, res="alias", ldw=5 * dj, woff=dj, tag="gptj prefill fc_out"),
        # GPT-J 16-row decode: fc_in into the [att | mlp] operand, then out_proj + fc_out as one GEMM over K = 5d
        Case(16, 4 * dj, dj, A, "gelu_new", out="bf16", ldo=5 * dj, ocol=dj, tag="gptj decode fc_in",
             expect=("gemm_bf16_tn_kernel<32>", (128, 1, 2))),
        Case(16, dj, 5 * dj, A, res="alias", tag="gptj decode out_proj+fc_out",
             expect=("gemm_bf16_tn_kernel<32>", (32, 1, 8))),
        # lm_head at the GPT-2 vocabulary, logits pitch rounded up to 64
        Case(5, 50257, dx, A, ldo=50304, bias=False, tag="lm_head 5 rows", expect=("gemm_bf16_tn_kernel<32>", (393, 1, 1))),
        Case(64, 50257, d2, A, ldo=50304, bias=False, tag="lm_head 64 rows",
             expect=("gemm_bf16_tn_kernel<64>", (393, 1, 1))),
        Case(255, 50257, d2, A, ldo=50304, tag="lm_head 255 rows", expect=("gemm_bf16_tn_kernel<256>", (393, 1, 1))),
        # ViT-L/14: patch embedding (588 padded to K = 640) and c_fc with QuickGELU over 257 tokens per image
        Case(2 * 256, 1024, 640, A, bias=False, tag="vit-l/14 patch embed"),
        Case(2 * 257, 4096, 1024, A, "quick_gelu", out="bf16", tag="vit-l/14 c_fc"),
        # MLP mapper: Linear -> tanh -> Linear into rows of out_rows_per_image * d
        Case(5, 3840, 512, A, "tanh", out="bf16", tag="mlp mapper linear"),
        Case(5, 10 * d2, 3840, A, ldo=12 * d2, tag="mlp mapper linear 2"),
        # all-features mapper over ViT-B/16's 197 tokens: per-token linear added in place onto pre-filled rows
        Case(3 * 197, d2, d2, (1, 0, 0), res="alias", remap=(197, 207, 0), tag="all-features mapper"),
    ]


MATRIX = _matrix()
PROBES = _probes()
ENGINE = _engine_shapes()


def _case_id(c):
    s = "%s-%s-T%dF%dK%d-%s-%s-%s" % (c.tag.replace(" ", "_") or _route_label(c.route), c.act, c.T, c.F, c.K, c.res,
                                       c.out, c.data)
    if c.lda or c.ldw or c.ldo or c.ocol:
        s += "-lda%d-ldw%d@%d-ldo%d@%d" % (c.lda or c.K, c.ldw or c.K, c.woff, c.ldo or c.F, c.ocol)
    if c.remap:
        s += "-remap%d/%d/%d" % c.remap
    return s


def test_matrix_covers_every_route_activation_residual_and_pitch():
    """The covering design: each route x each activation, each route x each residual / output pair, every pitch variant
    on the one-tile and the persistent kernels; forced splits are never clamped by the launcher."""
    by_route = {}
    for c in MATRIX:
        by_route.setdefault(c.route, []).append(c)
    assert set(by_route) == set(ROUTES)
    for route, cs in by_route.items():
        assert {c.act for c in cs} == set(ACTS), route
        assert {(c.res, c.out) for c in cs} == set(RES_OUT), route
    for o in (2, 4, 3):
        cs = [c for c in MATRIX if c.route[0] == o]
        assert any(c.lda for c in cs) and any(c.woff for c in cs) and any(c.ocol for c in cs)
        assert any(c.ldo and c.ldo % 8 == 4 for c in cs) and any(c.ldo and c.ldo % 8 == 0 and not c.ocol for c in cs)
    assert any(c.ldo % 2 for c in MATRIX if c.ldo)
    for c in MATRIX + PROBES:
        o, bn, s = c.route
        if o == 2:
            kb = c.K // 64
            assert c.T <= bn and s <= kb and -(-kb // s) * (s - 1) < kb, c
    assert 150 <= len(MATRIX) <= 260


# ------------------------------------------------------------------------------------------------ running a case
def _bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def _fill(c, gen, dev):
    T, F, K = c.T, c.F, c.K
    R = int(remap_rows(T, c.remap)[-1]) + 1 if c.remap else T
    if c.data == "int":
        x = torch.randint(-4, 5, (T, K), generator=gen, device=dev).float()
        w = torch.randint(-4, 5, (F, K), generator=gen, device=dev).float()
        b = torch.randint(-64, 65, (F,), generator=gen, device=dev).float()
        r = torch.randint(-64, 65, (R, F), generator=gen, device=dev).float()
        return x, w, b, r
    x = torch.randn(T, K, generator=gen, device=dev)
    w = torch.randn(F, K, generator=gen, device=dev) / math.sqrt(K)
    b = torch.randn(F, generator=gen, device=dev) * 0.5
    r = torch.randn(R, F, generator=gen, device=dev)
    if c.data in ("onehot_x", "onehot_w"):
        # k at UMMA-slice (16), k-block (64) and split boundaries, and the last k
        kb = K // 64
        per = -(-kb // c.route[2]) * 64 if c.route[0] == 2 and c.route[2] > 1 else 128
        ks = sorted({k for k in (0, 15, 16, 31, 63, 64, 65, per - 1, per, per + 1, 2 * per - 1, 2 * per, K - 65, K - 64,
                                 K - 1) if 0 <= k < K})
        n = T if c.data == "onehot_x" else F
        hot = torch.zeros(n, K, device=dev)
        hot[torch.arange(n), torch.tensor([ks[i % len(ks)] for i in range(n)])] = 1.0
        if c.data == "onehot_x":
            x = hot
        else:
            w = hot
    elif c.data == "sat":
        w = w * 0.01
        b = torch.tensor([20.0, -20.0, 60.0, -60.0, 100.0, -100.0], device=dev).repeat(F // 6 + 1)[:F]
        b += 0.3 * torch.randn(F, generator=gen, device=dev)
    return x, w, b, r


def _setup(c, seed):
    """The case's operands inside NaN-filled buffers; returns a dict the launch and the checks share."""
    dev = DEV
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    T, F, K = c.T, c.F, c.K
    lda, ldw = c.lda or K, c.ldw or K
    ldo = c.ldo or F
    rows = remap_rows(T, c.remap).to(dev)
    R = int(rows[-1]) + 1
    xv, wv, bv, rv = _fill(c, gen, dev)
    xb = torch.full((T + 2 * G, lda), NAN, dtype=torch.bfloat16, device=dev)
    xb[G:G + T, :K] = xv.bfloat16()
    wb = torch.full((F + 2 * G, ldw), NAN, dtype=torch.bfloat16, device=dev)
    wb[G:G + F, c.woff:c.woff + K] = wv.bfloat16()
    bb = torch.full((F + 128,), NAN, dtype=torch.float32, device=dev)
    bb[64:64 + F] = bv
    odt = torch.float32 if c.out == "f32" else torch.bfloat16
    ob = torch.full((R + 2 * G, ldo), NAN, dtype=odt, device=dev)
    if c.remap:   # the rows the remap does not reach hold values that must survive (mapper: prefix / positions)
        ob[G:G + R, c.ocol:c.ocol + F] = rv.to(odt)
    if c.res == "alias":
        ob[G + rows, c.ocol:c.ocol + F] = rv[rows]
    rb = None
    if c.res == "sep":
        ldr = c.ldr or ldo + 4
        rb = torch.full((R + 2 * G, ldr), NAN, dtype=torch.float32, device=dev)
        rb[G + rows, :F] = rv[rows]   # rows no token reads stay NaN
    return dict(c=c, rows=rows, R=R, xb=xb, wb=wb, bb=bb, ob=ob, rb=rb, ob0=ob.clone(),
                r_used=rv[rows] if c.res != "none" else None)


def _launch(eng, s):
    c = s["c"]
    o, bn, sp = c.route
    T, F, K, R = c.T, c.F, c.K, s["R"]
    x = s["xb"][G:G + T, :K]
    w = s["wb"][G:G + F, c.woff:c.woff + K]
    out = s["ob"][G:G + R, c.ocol:c.ocol + F]
    residual = s["rb"][G:G + R, :F] if s["rb"] is not None else None
    bias = s["bb"][64:64 + F] if c.bias else None
    return eng.op_linear(x, w, bias, c.act, residual, orientation=o, bn=bn, split_k=sp, out=out,
                         residual_is_out=c.res == "alias", row_remap=c.remap)


WORST = {}   # "route out-dtype" -> (worst err / bound, case id)


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if WORST:
        print("\nworst err / bound per route:")
        for k in sorted(WORST):
            print("  %-19s %.4f  %s" % (k, WORST[k][0], WORST[k][1]))


def _check(eng, c, seed):
    s = _setup(c, seed)
    ins = [s["xb"].clone(), s["wb"].clone(), s["bb"].clone()] + ([s["rb"].clone()] if s["rb"] is not None else [])
    _launch(eng, s)
    torch.cuda.synchronize()
    first = s["ob"].clone()
    s["ob"].copy_(s["ob0"])
    _launch(eng, s)
    torch.cuda.synchronize()
    ob, ob0, rows = s["ob"], s["ob0"], s["rows"]
    assert torch.equal(_bits(ob), _bits(first)), "two calls differ"
    for before, after in zip(ins, [s["xb"], s["wb"], s["bb"]] + ([s["rb"]] if s["rb"] is not None else [])):
        assert torch.equal(_bits(before), _bits(after)), "an input buffer was written"
    written = torch.zeros(ob.shape, dtype=torch.bool, device=ob.device)
    written[(G + rows).unsqueeze(1), torch.arange(c.ocol, c.ocol + c.F, device=ob.device).unsqueeze(0)] = True
    assert torch.equal(_bits(ob)[~written], _bits(ob0)[~written]), "an element outside the output was written"
    got = ob[G + rows][:, c.ocol:c.ocol + c.F]
    assert torch.isfinite(got).all(), "non-finite output (a NaN sentinel was read?)"
    x = s["xb"][G:G + c.T, :c.K]
    w = s["wb"][G:G + c.F, c.woff:c.woff + c.K]
    b = s["bb"][64:64 + c.F] if c.bias else None
    y, bound = reference(x, w, b, c.act, s["r_used"], c.out == "bf16")
    q = ratio(got, y, bound)
    label = "%s %s" % (_route_label(c.route) if not c.tag else "auto", c.out)
    if q > WORST.get(label, (-1.0, ""))[0]:
        WORST[label] = (q, _case_id(c))
    assert q <= 1.0, "err / bound = %.3f" % q
    return got, x, w, b, s


@gpu
@pytest.mark.parametrize("c", MATRIX, ids=[_case_id(c) for c in MATRIX])
def test_matrix_case(tiny_engine, c):
    _check(tiny_engine, c, MATRIX.index(c))


@gpu
@pytest.mark.parametrize("c", ENGINE, ids=[_case_id(c) for c in ENGINE])
def test_engine_shape(tiny_engine, c):
    _check(tiny_engine, c, 1000 + ENGINE.index(c))


@gpu
@pytest.mark.parametrize("c", PROBES, ids=[_case_id(c) for c in PROBES])
def test_exact_probe(tiny_engine, c):
    got, x, w, b, s = _check(tiny_engine, c, 2000 + PROBES.index(c))
    if c.data == "int":
        y, _ = reference(x, w, b, "none", s["r_used"], False)
        assert torch.equal(got.double(), y), "integer sums are exact in fp32"
    elif c.data == "onehot_x":
        k = x.float().argmax(1)
        assert torch.equal(got, w.float()[:, k].t() + b), "out[t] must be w[:, k_t] + b"
    elif c.data == "onehot_w":
        k = w.float().argmax(1)
        assert torch.equal(got, x.float()[:, k] + b), "out[:, f] must be x[:, k_f] + b[f]"


# ------------------------------------------------------------------------------------------------ which kernel ran
def kernel_of(name):
    """A profiler kernel name (demangled or mangled) -> gemm_bf16_tn_kernel<BN> / gemm_persist_kernel / gemm_pair_kernel."""
    m = re.search(r"gemm_bf16_tn_kernel\s*<\s*(?:\(int\))?(\d+)\s*>|gemm_bf16_tn_kernelILi(\d+)E", name)
    if m:
        return "gemm_bf16_tn_kernel<%s>" % (m.group(1) or m.group(2))
    for k in ("gemm_persist_kernel", "gemm_pair_kernel"):
        if k in name:
            return k
    return None


def expected_route(c, sms):
    o, bn, s = c.route
    cdiv = lambda a, b: -(-a // b)
    if o == 2:
        return "gemm_bf16_tn_kernel<%d>" % bn, (cdiv(c.F, 128), cdiv(c.T, bn), s)
    if o == 4:
        return "gemm_persist_kernel", (min(cdiv(c.T, 128) * cdiv(c.F, bn), sms), 1, 1)
    if o == 3:
        return "gemm_pair_kernel", (2 * min(cdiv(c.T, 256) * cdiv(c.F, bn), sms // 2), 1, 1)
    return c.expect


@gpu
def test_profiler_names_the_kernel_and_grid_of_every_case(tiny_engine):
    """Every forced case runs the kernel it names with tiles x splits CTAs (one-tile kernel) or min(tiles, SMs) CTAs /
    pairs (persistent kernels); the engine shapes the design documents take their literal routes."""
    from torch.profiler import ProfilerActivity, profile
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    cases = [c for c in MATRIX + PROBES if c.route[0] in (2, 3, 4)] + [c for c in ENGINE if c.expect and sms == 148]
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        # (the first device activity of a profiling session can go unrecorded in a process that profiled before)
        torch.ones(8, device="cuda").add_(1)
        torch.cuda.synchronize()
        for i, c in enumerate(cases):
            _launch(tiny_engine, _setup(c, i))
            torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    ran = sorted((e["ts"], kernel_of(e["name"]), tuple(e.get("args", {}).get("grid", ()))) for e in events
                 if e.get("cat") == "kernel" and kernel_of(e.get("name", "")))
    assert len(ran) == len(cases), (len(ran), len(cases))
    bad = [(_case_id(c), expected_route(c, sms), (k, g)) for c, (_, k, g) in zip(cases, ran) if (k, g) != expected_route(c, sms)]
    assert not bad, bad[:10]


# ------------------------------------------------------------------------------------------------ rejections
@gpu
def test_out_of_range_arguments_are_refused_and_the_context_keeps_working(tiny_engine):
    """Each check of gemm_launch refuses with a message and writes nothing; a good call afterwards is right."""
    import ctypes as C
    eng = tiny_engine
    T, F, K = 40, 96, 128
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    x = torch.randn(T, K, generator=g, device="cuda").bfloat16()
    w = (torch.randn(F, K, generator=g, device="cuda") / math.sqrt(K)).bfloat16()
    b = torch.randn(F, generator=g, device="cuda")
    res = torch.randn(T, F, generator=g, device="cuda")
    out = torch.full((3 * T, F), NAN, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None

    def call(act=0, lda=K, ldw=0, ldo=F, residual=None, ldr=0, remap=(0, 0, 0), orientation=0, entry="ex"):
        if entry == "ex":
            return eng.lib.ccb_op_linear_ex(eng._h, p(x), lda, T, p(w), ldw, F, K, p(b), act, p(residual), ldr, p(out), ldo,
                                            0, remap[0], remap[1], remap[2], orientation, 0, 0, eng._stream())
        return eng.lib.ccb_op_linear(eng._h, p(x), lda, T, p(w), F, K, p(b), act, p(residual), ldr, p(out), ldo, 0,
                                     orientation, 0, 0, eng._stream())

    bad = [
        (dict(act=8), "activation 8"),                       # CCB_ACT_GEGLU is not an epilogue
        (dict(act=8, entry="old"), "activation 8"),
        (dict(act=-1), "activation -1"),
        (dict(act=9, orientation=1), "activation 9"),
        (dict(lda=K - 8), "lda=120"),
        (dict(ldw=K - 8), "ldw=120"),
        (dict(ldo=F - 1), "ldo=95"),
        (dict(residual=res, ldr=F - 4), "ldr=92"),
        (dict(remap=(0, 5, 0), orientation=1), "rg_in=0"),
        (dict(remap=(-4, 5, 0), orientation=1), "rg_in=-4"),
        (dict(remap=(20, 25, -1), orientation=1), "rg_off=-1"),
        (dict(remap=(20, 25, 6), orientation=1), "rg_off=6"),     # rows of two groups would collide
    ]
    for kw, msg in bad:
        assert call(**kw) != 0, kw
        err = eng.lib.ccb_last_error(eng._h).decode()
        assert msg in err, (kw, err)
        torch.cuda.synchronize()
        assert torch.isnan(out).all(), ("written although refused", kw)
        got = eng.op_linear(x, w, b, "gelu_new", res)
        y, bound = reference(x, w, b, "gelu_new", res, False)
        assert ratio(got, y, bound) <= 1.0
    with pytest.raises(RuntimeError, match="activation 8"):
        eng.op_linear(x, w, b, "geglu")
    # the limits themselves are accepted: lda = K, ldw = K, ldo = ldr = F, rg_off + rg_in = rg_out
    # (the residual is read at the remapped rows, so it spans as many rows as out)
    res_rows = torch.randn(out.shape[0], F, generator=g, device="cuda")
    assert call(ldw=K, residual=res_rows, ldr=F, remap=(20, 25, 5), orientation=1) == 0
    torch.cuda.synchronize()
    rows = remap_rows(T, (20, 25, 5)).cuda()
    y, bound = reference(x, w, b, "none", res_rows[rows], False)
    assert ratio(out[rows], y, bound) <= 1.0
