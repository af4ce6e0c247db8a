"""Every route of attention_prefill (csrc/attention.cu) against a float64 reference, and the shapes no kernel holds.

`attention_prefill` is the attention of the ViT, the CLIP text tower, the prefix mapper and the LM prefill /
teacher-forced pass.  It picks one of five kernels by (S, head_dim, causal, cache, rotary); `expected_route` below mirrors
that choice.  The tests here
  * run a matrix of shapes that visits every route and template bucket (ragged S, odd head_dim / 2, B and H > 1, causal,
    rotary, non-default scales) through `op_attention` against float64 attention over the same bf16 qkv;
  * feed inputs that random data does not probe: all scores very negative (a zero-padded key that is not masked takes the
    weight), scores of magnitude ~100 (a softmax without the max subtracted overflows), a constant V (the normaliser to one
    bf16 ulp) and identical keys (the mean of V);
  * check under torch.profiler that the kernel the mirror names is the one that ran;
  * repeat all of this in child processes with CCB_ATTN_UMMA=0 and CCB_ATTN_MMA=0 (the fallback kernels);
  * run the LM with an HF key mask and the KV-cache writes of each prefill route through lm_forward / generate / beam
    search against the fp32 oracle and the engine's own teacher-forced logits;
  * check that ccb_create, lm_forward and generate reject, with S and head_dim in the message and before any launch, the
    shapes the scalar kernel cannot hold, and accept and compute correctly the largest ones it can.
"""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import clipcap_oracle as orc  # noqa: E402

pytestmark = pytest.mark.gpu

TOL = 2e-2          # DESIGN §4: logits / mapper outputs against the fp32 oracle
ATT_REL, ATT_ABS = 1.5e-2, 1e-3   # operator tolerance: max|out - ref| <= ATT_REL * max|ref| + ATT_ABS
TIE = 2e-2          # DESIGN §4 tie rule


# ------------------------------------------------------------------------------------------------ the dispatcher, mirrored
def _env_on(name):
    """The library reads CCB_ATTN_MMA / CCB_ATTN_UMMA once: a value starting with '0' switches the kernel off."""
    return not os.environ.get(name, "").startswith("0")


MMA, UMMA = _env_on("CCB_ATTN_MMA"), _env_on("CCB_ATTN_UMMA")
SCALAR_SMEM_CAP = 200 * 1024


def scalar_smem(S, hd):
    """Dynamic shared memory of attention_prefill_kernel: K rows padded to hd/2 + 1 words, V rows, one word of alignment,
    and per warp (8) a q row of hd floats and a probability row of S floats = S * (4 hd + 36) + 32 hd + 4 bytes."""
    return (S * (hd // 2 + 1) + S * (hd // 2) + 1) * 4 + 8 * (hd + S) * 4


def expected_route(S, hd, causal, rotary_dim, mma=MMA, umma=UMMA, cache=False, key_mask=False):
    """The kernel attention_prefill launches for a shape, with the mma template arguments, or "reject" (csrc/attention.cu:
    attention_prefill_unsupported and the routing in attention_prefill below it; DESIGN.md §3.0)."""
    if hd <= 0 or hd % 2:
        return "reject"
    if S > 256:
        if causal or cache or rotary_dim or key_mask or hd % 8 or hd > 256:
            return "reject"
        return "attention_prefill_long_kernel"
    if mma and umma and hd == 64 and S <= 64 and rotary_dim == 0:
        return "attention_prefill_umma_kernel"
    if mma and S <= 80 and hd % 8 == 0 and 256 < hd <= 512 and rotary_dim == 0:
        return "attention_prefill_mma_kernel<10, 32, %s>" % ("false" if cache else "true")
    if mma and S <= 128 and hd % 8 == 0 and hd <= 256 and rotary_dim % 2 == 0:
        ks, nt = (hd + 15) // 16, 2 * ((S + 15) // 16)
        if 8 < nt <= 10 and 8 < ks <= 13 and not cache and rotary_dim == 0:
            return "attention_prefill_mma_kernel<10, 13, true>"
        NT = next(b for b in (4, 6, 8, 10, 16) if nt <= b)
        KS = next(b for b in (4, 8, 13, 16) if ks <= b)
        return "attention_prefill_mma_kernel<%d, %d, false>" % (NT, KS)
    if scalar_smem(S, hd) > SCALAR_SMEM_CAP:
        return "reject"
    return "attention_prefill_kernel"


def kernel_route(name):
    """A profiler kernel name -> the spelling expected_route uses (demangled with or without casts, or mangled)."""
    m = re.search(r"attention_prefill_mma_kernel<\s*(?:\(int\))?(\d+)\s*,\s*(?:\(int\))?(\d+)\s*,\s*(?:\(bool\))?(\w+)\s*>", name)
    if m:
        return "attention_prefill_mma_kernel<%s, %s, %s>" % (m.group(1), m.group(2), "true" if m.group(3) in ("true", "1") else "false")
    m = re.search(r"attention_prefill_mma_kernelILi(\d+)ELi(\d+)ELb([01])E", name)
    if m:
        return "attention_prefill_mma_kernel<%s, %s, %s>" % (m.group(1), m.group(2), "true" if m.group(3) == "1" else "false")
    for k in ("attention_prefill_umma_kernel", "attention_prefill_long_kernel", "attention_prefill_kernel"):
        if k in name:    # (attention_prefill_kernel is not a substring of the other names)
            return k
    return None


# ------------------------------------------------------------------------------------------------ float64 reference
def rotary64(x, rd):
    """GPT-J rotate_every_two on the first rd dims of x [B, S, H, hd] (float64), positions 0..S-1,
    inv_freq = 10000^(-2i / rd) (HF modeling_gptj.py)."""
    S = x.shape[1]
    inv = 10000.0 ** (-2.0 * torch.arange(rd // 2, dtype=torch.float64, device=x.device) / rd)
    ang = torch.arange(S, dtype=torch.float64, device=x.device)[:, None] * inv[None, :]
    c, s = torch.cos(ang)[None, :, None, :], torch.sin(ang)[None, :, None, :]
    a, b = x[..., 0:rd:2], x[..., 1:rd:2]
    out = x.clone()
    out[..., 0:rd:2] = a * c - b * s
    out[..., 1:rd:2] = b * c + a * s
    return out


def ref_attention(qkv, B, S, H, hd, causal, scale=None, rotary_dim=0):
    q, k, v = qkv.double().view(B, S, 3, H, hd).unbind(2)
    if rotary_dim:
        q, k = rotary64(q, rotary_dim), rotary64(k, rotary_dim)
    att = torch.einsum("bnhd,bmhd->bhnm", q, k) * (hd ** -0.5 if scale is None else scale)
    if causal:
        allowed = torch.ones(S, S, dtype=torch.bool, device=qkv.device).tril()
        att = att.masked_fill(~allowed, float("-inf"))
    att = att.softmax(-1)
    return torch.einsum("bhnm,bmhd->bnhd", att, v).reshape(B * S, H * hd)


def assert_close(out, ref, what=""):
    assert torch.isfinite(out.float()).all(), ("non-finite output", what)
    err = (out.double() - ref).abs().max().item()
    bound = ATT_REL * ref.abs().max().item() + ATT_ABS
    assert err <= bound, (what, err, bound)


def rand_qkv(B, S, H, hd, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B * S, 3 * H * hd, generator=g).bfloat16().cuda()


# ------------------------------------------------------------------------------------------------ the route matrix
# (S, hd, causal, rotary_dim, scale); B = 2, H = 3 everywhere (the (h, b) grid indexing)
def _matrix():
    cases = []

    def add(S, hd, causal, rotary=0, scale=None):
        cases.append((S, hd, causal, rotary, scale))

    for c in (False, True):
        for S in (1, 2, 31, 33, 63, 64):                      # umma: hd 64, S <= 64
            add(S, 64, c)
        for S in (65, 80, 81, 96, 127, 128):                  # mma past the umma limit (hd 64)
            add(S, 64, c)
    add(77, 64, True)                                         # the CLIP text tower
    for i, hd in enumerate((8, 24, 72, 128, 136, 208, 216, 248, 256)):   # mma KS buckets 4 / 8 / 13 / 16, NT 4 / 6 / 8
        for j, S in enumerate((16, 17, 48, 49)):
            add(S, hd, (i + j) % 2 == 1)
        add(128, hd, i % 2 == 0)                              # NT 16
    for S in (65, 72, 80):                                    # OVL (the GPT2-XL mapper: 80 x 200)
        for hd in (144, 200, 208):
            add(S, hd, False)
    add(80, 200, True)
    for hd in (264, 320, 512):                                # head_dim above 256: Q fragments streamed
        for S in (1, 7, 33, 80):
            for c in (False, True):
                add(S, hd, c)
    for S in (81, 90):                                        # ... and past 80 tokens the scalar kernel
        for c in (False, True):
            add(S, 512, c)
    for c in (False, True):                                   # scalar
        for hd in (64, 96):
            for S in (129, 197, 255, 256):
                add(S, hd, c)
        for S in (129, 197, 237):
            add(S, 200, c)
        for S in (129, 185):
            add(S, 256, c)
        for hd in (2, 6, 66, 130):
            for S in (5, 100, 200):
                add(S, hd, c)
    for S in (40, 100, 128):                                  # rotary on the mma route
        add(S, 256, True, 64)
        for rd in (64, 24, 2):
            add(S, 64, True, rd)
    add(129, 256, True, 64)                                   # rotary on the scalar route
    add(185, 256, True, 64)
    add(150, 66, True, 16)
    for scale in (0.05, 1.0):                                 # the scale argument, once per route
        add(50, 64, False, 0, scale)                          # umma
        add(100, 128, True, 0, scale)                         # mma
        add(75, 200, False, 0, scale)                         # OVL
        add(33, 512, False, 0, scale)                         # head_dim 512
        add(197, 64, False, 0, scale)                         # scalar
        add(300, 64, False, 0, scale)                         # long
    return cases


MATRIX = _matrix()
B_, H_ = 2, 3


def _case_id(c):
    S, hd, causal, rd, scale = c
    return "S%d-hd%d%s%s%s-%s" % (S, hd, "-causal" if causal else "", "-rot%d" % rd if rd else "",
                                   "-scale%g" % scale if scale is not None else "",
                                   expected_route(S, hd, causal, rd).replace("attention_prefill_", "").replace(", ", "."))


def _run_case(eng, c, seed):
    S, hd, causal, rd, scale = c
    qkv = rand_qkv(B_, S, H_, hd, seed)
    return qkv, eng.op_attention(qkv, B_, S, H_, hd, causal, rotary_dim=rd, scale=scale)


@pytest.mark.parametrize("case", MATRIX, ids=[_case_id(c) for c in MATRIX])
def test_route_matrix_matches_float64(tiny_engine, case):
    S, hd, causal, rd, scale = case
    assert expected_route(S, hd, causal, rd) != "reject"
    qkv, out = _run_case(tiny_engine, case, S * 1009 + hd * 7 + rd)
    assert_close(out, ref_attention(qkv, B_, S, H_, hd, causal, scale, rd), _case_id(case))


# shapes no kernel holds: ragged / odd head_dim, causal / rotary above 256 tokens, the scalar kernel's shared memory
REJECT = [(257, 64, True, 0), (300, 64, False, 64), (300, 264, False, 0), (100, 7, False, 0), (238, 200, False, 0),
          (186, 256, True, 0), (186, 256, True, 64), (256, 256, True, 0), (91, 512, False, 0), (129, 512, True, 0)]


@pytest.mark.parametrize("S,hd,causal,rd", REJECT)
def test_shapes_without_a_kernel_are_rejected(tiny_engine, S, hd, causal, rd):
    assert expected_route(S, hd, causal, rd) == "reject"
    qkv = rand_qkv(1, S, 2, hd, 5)
    with pytest.raises(RuntimeError, match="attention_prefill"):
        tiny_engine.op_attention(qkv, 1, S, 2, hd, causal, rotary_dim=rd)
    # the context stays usable
    small = rand_qkv(2, 40, 2, 64, 6)
    assert_close(tiny_engine.op_attention(small, 2, 40, 2, 64), ref_attention(small, 2, 40, 2, 64, False))


@pytest.mark.parametrize("S", [64, 128, 256])
def test_switch_over_pairs_on_identical_data(tiny_engine, S):
    """S and S + 1 at hd 64 cross a route boundary (umma | mma, mma | scalar, scalar | long) on the same tokens."""
    H, hd = 3, 64
    big = rand_qkv(2, S + 1, H, hd, 77 + S).view(2, S + 1, -1)
    small = big[:, :S].reshape(2 * S, -1).contiguous()
    big = big.reshape(2 * (S + 1), -1).contiguous()
    for causal in ((False, True) if S < 256 else (False,)):
        o_small = tiny_engine.op_attention(small, 2, S, H, hd, causal)
        o_big = tiny_engine.op_attention(big, 2, S + 1, H, hd, causal)
        assert_close(o_small, ref_attention(small, 2, S, H, hd, causal))
        assert_close(o_big, ref_attention(big, 2, S + 1, H, hd, causal))
        if causal:   # the first S rows see the same keys in both
            a = o_small.view(2, S, -1).double()
            b = o_big.view(2, S + 1, -1)[:, :S].double()
            assert (a - b).abs().max().item() <= ATT_REL * a.abs().max().item() + ATT_ABS


# ------------------------------------------------------------------------------------------------ inputs random data does not probe
# one ragged shape per route (S not a multiple of the route's key tile): umma (64), mma NT 16 (8), OVL (8), head_dim 512 (8),
# scalar (32), long (64)
PROBE_SHAPES = [(50, 64), (100, 128), (75, 200), (33, 512), (197, 64), (300, 64)]


def _probe_id(p):
    return "S%d-hd%d-%s" % (p[0], p[1], expected_route(p[0], p[1], False, 0).replace("attention_prefill_", "").replace(", ", "."))


def _signs(g, *shape):
    return torch.randint(0, 2, shape, generator=g).float() * 2 - 1


@pytest.mark.parametrize("S,hd", PROBE_SHAPES, ids=[_probe_id(p) for p in PROBE_SHAPES])
def test_negative_scores(tiny_engine, S, hd):
    """Every real score <= -30: keys are positive multiples of one direction u (|u|^2 = hd), queries -c u.  A zero-padded key
    that is not masked scores 0 and would take almost all the weight."""
    B, H = 2, 3
    g = torch.Generator().manual_seed(S + hd)
    x = torch.randn(B, S, 3, H, hd, generator=g)
    u = _signs(g, H, hd)
    x[:, :, 1] = u * (1 + 0.5 * torch.rand(B, S, H, 1, generator=g))
    x[:, :, 0] = -u * (40 / hd ** 0.5) * (1 + torch.rand(B, S, H, 1, generator=g))
    qkv = x.reshape(B * S, -1).bfloat16().cuda()
    q, k, _ = qkv.double().view(B, S, 3, H, hd).unbind(2)
    assert (torch.einsum("bnhd,bmhd->bhnm", q, k) * hd ** -0.5).max().item() <= -30
    assert_close(tiny_engine.op_attention(qkv, B, S, H, hd), ref_attention(qkv, B, S, H, hd, False))


@pytest.mark.parametrize("S,hd", PROBE_SHAPES, ids=[_probe_id(p) for p in PROBE_SHAPES])
def test_peaked_scores(tiny_engine, S, hd):
    """Scores of magnitude ~100: query i is a multiple of key t(i), t cycling over j = 0, S // 2 and S - 1.  exp(100)
    overflows fp32: without the row maximum subtracted the output is inf / NaN."""
    B, H = 2, 3
    g = torch.Generator().manual_seed(3 * S + hd)
    x = torch.randn(B, S, 3, H, hd, generator=g)
    x[:, :, 1] = _signs(g, B, S, H, hd)
    t = torch.tensor([(0, S // 2, S - 1)[i % 3] for i in range(S)])
    x[:, :, 0] = (100 / hd ** 0.5) * x[:, t, 1]
    qkv = x.reshape(B * S, -1).bfloat16().cuda()
    out = tiny_engine.op_attention(qkv, B, S, H, hd)
    ref = ref_attention(qkv, B, S, H, hd, False)
    assert_close(out, ref)
    # the dominant key carries the output
    v = qkv.double().view(B, S, 3, H, hd)[:, :, 2]
    assert (ref.view(B, S, H, hd) - v[:, t.cuda()]).abs().max().item() < 0.05


@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("S,hd", PROBE_SHAPES, ids=[_probe_id(p) for p in PROBE_SHAPES])
def test_constant_v_is_reproduced_to_one_ulp(tiny_engine, S, hd, causal):
    """V = 3.0 for every key: whatever the weights, every output is 3.0.  Within one bf16 ulp (2^-6 at 3.0); two on the
    long kernel, whose P is a single bf16 term.  This pins the normaliser, which the max-norm tolerance cannot."""
    if causal and S > 256:
        pytest.skip("the long kernel is non-causal")
    B, H = 2, 3
    g = torch.Generator().manual_seed(5 * S + hd)
    x = torch.randn(B, S, 3, H, hd, generator=g)
    x[:, :, 2] = 3.0
    qkv = x.reshape(B * S, -1).bfloat16().cuda()
    out = tiny_engine.op_attention(qkv, B, S, H, hd, causal).float()
    ulp = 2.0 ** -6
    assert torch.isfinite(out).all()
    assert (out - 3.0).abs().max().item() <= (2 if S > 256 else 1) * ulp


@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("S,hd", PROBE_SHAPES, ids=[_probe_id(p) for p in PROBE_SHAPES])
def test_identical_keys_give_the_mean_of_v(tiny_engine, S, hd, causal):
    if causal and S > 256:
        pytest.skip("the long kernel is non-causal")
    B, H = 2, 3
    g = torch.Generator().manual_seed(7 * S + hd)
    x = torch.randn(B, S, 3, H, hd, generator=g)
    x[:, :, 1] = torch.randn(B, 1, H, hd, generator=g)
    qkv = x.reshape(B * S, -1).bfloat16().cuda()
    v = qkv.double().view(B, S, 3, H, hd)[:, :, 2]
    if causal:
        mean = v.cumsum(1) / torch.arange(1, S + 1, device=v.device, dtype=torch.float64).view(1, S, 1, 1)
    else:
        mean = v.mean(1, keepdim=True).expand(B, S, H, hd)
    assert_close(tiny_engine.op_attention(qkv, B, S, H, hd, causal), mean.reshape(B * S, H * hd))


# ------------------------------------------------------------------------------------------------ which kernel ran
def _cuda_kernel_names(prof):
    """Names of the kernels the profile saw, in start order (one stream: launch order)."""
    cuda = torch.autograd.DeviceType.CUDA
    evs = [(e.time_range.start, e.name) for e in prof.events() if e.device_type == cuda]
    if not evs:   # device events straight from the kineto results (kernel_route also reads mangled names)
        evs = [(e.start_ns(), e.name()) for e in prof.profiler.kineto_results.events() if e.device_type() == cuda]
    return [n for _, n in sorted(evs)]


def test_profiler_names_the_expected_kernel_for_every_case(tiny_engine):
    from torch.profiler import ProfilerActivity, profile
    cases = MATRIX + [(50, 64, False, 0, None), (300, 64, False, 0, None), (577, 64, False, 0, None), (617, 200, False, 0, None)]
    inputs = [rand_qkv(B_, c[0], H_, c[1], i) for i, c in enumerate(cases)]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for c, qkv in zip(cases, inputs):
            S, hd, causal, rd, scale = c
            tiny_engine.op_attention(qkv, B_, S, H_, hd, causal, rotary_dim=rd, scale=scale)
        torch.cuda.synchronize()
    ran = [kernel_route(n) for n in _cuda_kernel_names(prof) if kernel_route(n)]
    want = [expected_route(c[0], c[1], c[2], c[3]) for c in cases]
    assert len(ran) == len(want), (len(ran), len(want))
    bad = [(_case_id(c), w, r) for c, w, r in zip(cases, want, ran) if w != r]
    assert not bad, bad[:10]
    # the matrix reaches every route the environment allows
    routes = set(want)
    if MMA and UMMA:
        assert "attention_prefill_umma_kernel" in routes
    if MMA:
        assert {"attention_prefill_mma_kernel<10, 13, true>", "attention_prefill_mma_kernel<10, 32, true>",
                "attention_prefill_mma_kernel<16, 16, false>", "attention_prefill_mma_kernel<4, 4, false>"} <= routes
    assert {"attention_prefill_kernel", "attention_prefill_long_kernel"} <= routes


# ------------------------------------------------------------------------------------------------ fallback kernels
@pytest.mark.parametrize("env", ["CCB_ATTN_UMMA=0", "CCB_ATTN_MMA=0"])
def test_fallback_kernels_in_a_child(env):
    """This file again in a child process with the tcgen05 kernel (UMMA=0: head_dim 64, S <= 64 goes to mma.sync) or both
    tensor-core kernels (MMA=0: everything up to 256 tokens goes to the scalar kernel or is rejected) switched off.  The
    mirror follows the environment, so the route and profiler checks hold there too."""
    k, v = env.split("=")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k", "not child",
                        "-p", "no:cacheprovider"], env=dict(os.environ, **{k: v}), cwd=ROOT, capture_output=True, text=True,
                       timeout=1800)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


# ------------------------------------------------------------------------------------------------ the LM: key mask + KV cache
def _lm_engine(arch):
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    if arch == "gpt2":
        cfg = cc.EngineConfig(lm_arch="gpt2", lm_d=128, lm_layers=2, lm_heads=2, lm_vocab=512, lm_n_pos=288, map_kind="none",
                              vit=False, max_images=6, max_beam=3, max_ctx=256, page_tokens=16)
    else:
        # max_ctx above 256 (GPT-J has no learned positions): a 256-token prefix plus new tokens passes the context check,
        # so generate reaches the attention limit it is tested against
        cfg = cc.EngineConfig(lm_arch="gptj", lm_d=512, lm_layers=2, lm_heads=2, lm_vocab=512, lm_rotary_dim=64,
                              map_kind="none", vit=False, max_images=3, max_beam=1, max_ctx=272, page_tokens=16)
    eng = cc.Engine(cfg)
    sd = synthetic.lm_state_dict(cfg, 4321 if arch == "gpt2" else 4322, "cuda")
    eng.load_state_dict(sd, prefix="language_model.")
    eng.check_weights()
    return eng, cfg, orc.OracleLM(sd, arch, cfg.lm_heads, cfg.lm_rotary_dim)


@pytest.fixture(scope="module")
def gpt2():
    eng, cfg, lm = _lm_engine("gpt2")
    yield eng, cfg, lm
    eng.close()


@pytest.fixture(scope="module")
def gptj():
    eng, cfg, lm = _lm_engine("gptj")
    yield eng, cfg, lm
    eng.close()


def _prefix(N, S, d, seed):
    return (0.5 * torch.randn(N, S, d, generator=torch.Generator().manual_seed(seed))).cuda()


def _check_masked_lm_forward(model, S, lens):
    eng, cfg, lm = model
    hd = cfg.lm_d // cfg.lm_heads
    B = len(lens)
    emb = _prefix(B, S, cfg.lm_d, S)
    mask = (torch.arange(S)[None, :] < torch.tensor(lens)[:, None]).cuda()
    logits = eng.lm_forward(emb, mask)
    assert torch.isfinite(logits).all()
    ref = lm.logits(emb, mask)
    for b, n in enumerate(lens):
        err = (logits[b, :n] - ref[b, :n]).abs().max().item()
        assert err <= TOL * ref[b, :n].abs().max().item(), (S, hd, b, err)
    return expected_route(S, hd, True, cfg.lm_rotary_dim, key_mask=True)


@pytest.mark.parametrize("S", [64, 65, 128, 129, 256])
def test_gpt2_lm_forward_with_right_padding(gpt2, S):
    """HF key mask + causal on the umma (64), mma (65, 128) and scalar (129, 256) routes."""
    assert _check_masked_lm_forward(gpt2, S, [S, S - 7, S // 2 + 1]) != "reject"


@pytest.mark.parametrize("S", [100, 128, 129, 185])
def test_gptj_lm_forward_with_right_padding(gptj, S):
    """Rotary + HF key mask + causal at head_dim 256 on the mma (100, 128) and scalar (129, 185) routes."""
    assert _check_masked_lm_forward(gptj, S, [S, S - 9]) != "reject"


def _teacher_forced_logits(model, prefix, tokens):
    """Logits of the positions that chose tokens[:, t]: the engine's own lm_forward over [prefix ; embed(tokens)] where
    a kernel holds that length, else the fp32 oracle."""
    eng, cfg, lm = model
    S0, T = prefix.shape[1], tokens.shape[1]
    emb = torch.cat([prefix, eng.embed_tokens(tokens[:, :T - 1])], dim=1)
    if expected_route(S0 + T - 1, cfg.lm_d // cfg.lm_heads, True, cfg.lm_rotary_dim) != "reject":
        logits = eng.lm_forward(emb)
    else:
        logits = lm.logits(emb)
    return logits[:, S0 - 1:S0 - 1 + T].float()


def _assert_greedy_under_tie_rule(logits, tokens):
    best = logits.max(-1).values
    chosen = logits.gather(-1, tokens[..., None].long())[..., 0]
    scale = best - logits.min(-1).values
    ok = (logits.argmax(-1) == tokens) | (best - chosen <= TIE * scale)
    assert ok.all(), (~ok).nonzero()[:5].tolist()


@pytest.mark.parametrize("S0", [64, 65, 128, 129, 200])
def test_gpt2_greedy_from_each_prefill_route(gpt2, S0):
    """Prefill writes the KV pages (page_tokens 16: S0 crosses page boundaries) from the umma / mma / scalar kernels; the
    decode steps read them.  Both decode paths (persistent kernel, operator chain) give the same tokens, and every token
    is the arg-max of the teacher-forced logits."""
    eng, cfg, lm = gpt2
    T = 12
    prefix = _prefix(3, S0, cfg.lm_d, 100 + S0)
    p = eng.gen_params("greedy", T, stop_token=-1, max_stops=0)
    toks = {}
    try:
        for mega in (1, 0):
            assert eng.lib.ccb_debug_set_mega(eng._h, mega) == 1
            toks[mega] = eng.generate(prefix, p)[0].long().clone()
    finally:
        eng.lib.ccb_debug_set_mega(eng._h, 1)
    assert torch.equal(toks[0], toks[1])
    _assert_greedy_under_tie_rule(_teacher_forced_logits(gpt2, prefix, toks[1]), toks[1])


@pytest.mark.parametrize("S0", [100, 129, 185])
def test_gptj_greedy_from_each_prefill_route(gptj, S0):
    """Rotary prefill with cache append on the mma (100) and scalar (129, 185) routes, then the head_dim-256 decode."""
    eng, cfg, lm = gptj
    T = 12
    prefix = _prefix(2, S0, cfg.lm_d, 200 + S0)
    tokens = eng.generate(prefix, eng.gen_params("greedy", T, stop_token=-1, max_stops=0))[0].long()
    _assert_greedy_under_tie_rule(_teacher_forced_logits(gptj, prefix, tokens), tokens)


@pytest.mark.parametrize("S0", [129, 200])
def test_gpt2_beam_scores_from_shared_prefix_pages(gpt2, S0):
    """Beam search stores the prefix once per image with page_tokens = 1 (scalar prefill route here).  Each beam's score
    (sum of log-probabilities / length, inference.py:138) equals the mean teacher-forced log-probability of its tokens."""
    eng, cfg, lm = gpt2
    N, beam, T = 2, 3, 12
    prefix = _prefix(N, S0, cfg.lm_d, 300 + S0)
    tokens, lengths, scores = eng.generate(prefix, eng.gen_params("beam", T, stop_token=-1, max_stops=0, beam_size=beam))
    tokens = tokens.long().view(N * beam, T)
    assert (lengths == T).all()
    logp = _teacher_forced_logits(gpt2, prefix.repeat_interleave(beam, 0), tokens).log_softmax(-1)
    mean = logp.gather(-1, tokens[..., None])[..., 0].mean(-1).view(N, beam)
    assert torch.isfinite(scores).all()
    assert ((scores - mean).abs() <= TOL * mean.abs()).all(), (scores.tolist(), mean.tolist())


# ------------------------------------------------------------------------------------------------ the contract
def _all_features_cfg(tower, lm_d, P, **kw):
    import clipcap_b200 as cc
    return cc.EngineConfig.for_clip(tower, vit=False, lm_d=lm_d, lm_layers=1, lm_heads=lm_d // 64, lm_vocab=512,
                                    lm_n_pos=128, map_kind="transformer_all", map_prefix_len=P, map_heads=8, map_layers=1,
                                    max_images=2, max_ctx=P + 8, **kw)


@pytest.mark.parametrize("tower,lm_d,P,S,hd", [("ViT-B/16", 4096, 40, 237, 512), ("ViT-B/32", 4096, 41, 91, 512),
                                               ("ViT-B/16", 1600, 41, 238, 200)])
def test_mapper_without_a_kernel_is_rejected_at_creation(tower, lm_d, P, S, hd):
    import clipcap_b200 as cc
    with pytest.raises(RuntimeError, match=r"ccb_create: mapper attention over %d tokens with head_dim %d:" % (S, hd)):
        cc.Engine(_all_features_cfg(tower, lm_d, P))


@pytest.mark.parametrize("tower,lm_d,P,S", [("ViT-B/16", 1600, 40, 237), ("ViT-B/32", 4096, 40, 90)])
def test_largest_mappers_the_scalar_kernel_holds(tower, lm_d, P, S):
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    cfg = _all_features_cfg(tower, lm_d, P)
    assert cfg.map_clip_len + P == S and expected_route(S, lm_d // 8, False, 0) == "attention_prefill_kernel"
    eng = cc.Engine(cfg)
    sd = synthetic.mapper_state_dict(cfg, 1235, "cuda")
    eng.load_state_dict(sd, prefix="clip_project.")
    feats = torch.randn(2, cfg.map_clip_len, cfg.map_dim_clip, generator=torch.Generator().manual_seed(S)).cuda()
    out = eng.map_prefix(feats)
    ref = orc.mapper_all_forward(sd, feats, cfg.map_heads, "relu")
    assert out.shape == ref.shape == (2, P, lm_d)
    assert torch.isfinite(out).all()
    assert (out - ref).abs().max().item() <= TOL * ref.abs().max().item()
    eng.close()


@pytest.mark.parametrize("S", [186, 256])
def test_gptj_sequences_past_the_scalar_kernel_fail_before_any_launch(gptj, S):
    eng, cfg, lm = gptj
    emb = _prefix(1, S, cfg.lm_d, S)
    torch.cuda.synchronize()
    n0 = eng.launch_count
    with pytest.raises(RuntimeError, match=r"ccb_lm_forward: S=%d with head_dim 256:" % S):
        eng.lm_forward(emb)
    with pytest.raises(RuntimeError, match=r"generate: prefix of S0=%d tokens with head_dim 256:" % S):
        eng.generate(emb, eng.gen_params("greedy", 4, stop_token=-1, max_stops=0))
    assert eng.launch_count == n0
    # the next call on the same engine succeeds
    ok = eng.lm_forward(emb[:, :185], last_only=True)
    assert torch.isfinite(ok).all()
