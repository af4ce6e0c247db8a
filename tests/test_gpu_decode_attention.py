"""Every decode-attention path over a paged KV cache against a float64 reference.

A decode step attends one new token per row over the row's cached K / V, read through a block table.  Three kernels do
that: `attention_decode_kernel<64 | 128>` (one warp per (row, head), lane = token) and `attention_decode_wide_kernel<256>`
(one CTA per (row, head), cp.async tiles of at most 96 tokens folded with an online softmax) on the operator chain, and
`attention_phase` of the persistent GPT-2 decode kernel (csrc/decode_mega.cu).  The tests here
  * check the reference itself on the CPU: the paged gather through a permuted table equals attention over the same tokens
    laid out contiguously;
  * run a matrix of head_dim, rotary_dim, page_tokens, output pitch and block-table shapes (identity, permuted, beam-like
    shared prefixes) through `op_attention_decode` with ragged contexts that cross the warp kernel's 32-token lane stride
    and the wide kernel's 96-token tile, with every pool slot and table entry a row must not read pointing at NaN;
  * check the cache append byte for byte, determinism, and under torch.profiler which kernel ran;
  * probe with structured inputs: one dominant key at the first / last cached token, at page and tile boundaries (the
    output is that token's V row), a dominant new token, constant V, identical keys, all scores <= -30, scores ~ +100;
  * run the persistent kernel and the operator chain through the engine (one GPT-2-shaped layer, peaked attention) and
    compare the prefix K / V the prefill wrote, the k / v the decode step appended and the attention output with float64.
"""
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

gpu = pytest.mark.gpu

ATT_REL, ATT_ABS = 1.5e-2, 1e-3   # as the prefill routes: max|out - ref| <= ATT_REL * max|ref| + ATT_ABS
CTXS = [0, 1, 31, 32, 33, 63, 64, 95, 96, 97, 191, 192, 193, 411]   # one call's ragged contexts
CTX_TAG = "ctx0-411"
MAXP = 416                        # block-table pitch: every context < MAXP (the kernels size scores / tiles from it)
WIDE_TILE = 96                    # attention_decode_wide_kernel: tokens per cp.async tile at this pitch


def expected_kernel(hd):
    return {64: "warp<64>", 128: "warp<128>", 256: "wide<256>"}[hd]


def kernel_of(name):
    """A profiler kernel name (demangled or mangled) -> warp<64> / warp<128> / wide<256>, else None."""
    m = re.search(r"attention_decode_wide_kernel\s*<\s*(?:\(int\))?(\d+)\s*>|attention_decode_wide_kernelILi(\d+)E", name)
    if m:
        return "wide<%s>" % (m.group(1) or m.group(2))
    m = re.search(r"attention_decode_kernel\s*<\s*(?:\(int\))?(\d+)\s*>|attention_decode_kernelILi(\d+)E", name)
    if m:
        return "warp<%s>" % (m.group(1) or m.group(2))
    return None


# ------------------------------------------------------------------------------------------------ float64 reference
def rotary_at(x, pos, rd):
    """GPT-J rotate_every_two on the first rd dims of x [..., hd] at position pos (float64, inv_freq = 10000^(-2i / rd),
    HF modeling_gptj.py), as rotary64 of the prefill tests does for positions 0..S-1."""
    if not rd:
        return x
    inv = 10000.0 ** (-2.0 * torch.arange(rd // 2, dtype=torch.float64, device=x.device) / rd)
    ang = float(pos) * inv
    c, s = torch.cos(ang), torch.sin(ang)
    a, b = x[..., 0:rd:2], x[..., 1:rd:2]
    out = x.clone()
    out[..., 0:rd:2] = a * c - b * s
    out[..., 1:rd:2] = b * c + a * s
    return out


def gather_kv(kv, layer, page_tokens, bt_row, n):
    """K, V [n, H, hd] of positions 0..n-1 of one row, through its block table (float64)."""
    t = torch.arange(n, device=kv.device)
    pages = bt_row.to(kv.device).long()[t // page_tokens]
    slots = t % page_tokens
    return kv[layer, 0][pages, :, slots].double(), kv[layer, 1][pages, :, slots].double()


def new_token(qkv_row, H, hd, ctx, rd):
    """q (rotated), k (rotated, rounded to bf16 as the kernels store it) and v of a row's new token, [H, hd] float64."""
    q, k, v = qkv_row[:3 * H * hd].double().view(3, H, hd).unbind(0)
    q, k = rotary_at(q, ctx, rd), rotary_at(k, ctx, rd)
    return q, k.bfloat16().double(), v


def ref_decode(qkv, kv, layer, page_tokens, bt, ctx_len, H, hd, rd=0, scale=None, return_probs=False):
    """out [rows, H*hd] float64: row r attends over its cached positions 0..ctx-1 plus the new token at position ctx."""
    scale = hd ** -0.5 if scale is None else scale
    outs, probs = [], []
    for r, c in enumerate(ctx_len.tolist()):
        q, kn, vn = new_token(qkv[r], H, hd, c, rd)
        K, V = gather_kv(kv, layer, page_tokens, bt[r], c)
        K = torch.cat([K, kn[None].to(K.device)], 0)
        V = torch.cat([V, vn[None].to(V.device)], 0)
        p = (torch.einsum("hd,thd->ht", q.to(K.device), K) * scale).softmax(-1)
        outs.append(torch.einsum("ht,thd->hd", p, V).reshape(-1))
        probs.append(p)
    out = torch.stack(outs)
    return (out, probs) if return_probs else out


def assert_close(out, ref, what=""):
    assert torch.isfinite(out.float()).all(), ("non-finite output", what)
    err = (out.double().to(ref.device) - ref).abs().max().item()
    bound = ATT_REL * ref.abs().max().item() + ATT_ABS
    assert err <= bound, (what, err, bound)


def bf16_ulp(x):
    """One bf16 ulp at |x| (float64; the ulp of the smallest normal below it)."""
    a = x.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


# ------------------------------------------------------------------------------------------------ paged pools
def build_table(kind, ctxs, page_tokens, seed):
    """Block table [rows, MAXP] int32 and the pool size for rows with contexts `ctxs`.

    Row r uses pages for positions 0..ctx_r (the new token included).  identity: consecutive pages, row after row;
    perm: the same pages under a random permutation of the pool, which also holds unreferenced pages; beam: rows in
    groups of three share their first full pages (as beams share the prefix) and own the rest, the page of the new token
    included.  Entries past a row's last page point at the pool's last page, which no row uses (build_pool fills it with NaN)."""
    g = torch.Generator().manual_seed(seed)
    need = [c // page_tokens + 1 for c in ctxs]
    rows = len(ctxs)
    lists = [None] * rows
    nxt = 0
    if kind == "beam":
        for g0 in range(0, rows, 3):
            grp = list(range(g0, min(rows, g0 + 3)))
            shared = min(ctxs[r] // page_tokens for r in grp) // 2
            common = list(range(nxt, nxt + shared))
            nxt += shared
            for r in grp:
                own = list(range(nxt, nxt + need[r] - shared))
                nxt += need[r] - shared
                lists[r] = common + own
    else:
        for r in range(rows):
            lists[r] = list(range(nxt, nxt + need[r]))
            nxt += need[r]
    num_pages = nxt + (nxt // 4 + 3 if kind == "perm" else 1)    # + unreferenced pages (the last one is the poison page)
    if kind == "perm":
        perm = torch.randperm(num_pages - 1, generator=g).tolist()
        lists = [[perm[p] for p in lst] for lst in lists]
    poison = num_pages - 1
    bt = torch.full((rows, MAXP), poison, dtype=torch.int32)
    for r, lst in enumerate(lists):
        bt[r, :len(lst)] = torch.tensor(lst, dtype=torch.int32)
    return bt, num_pages


def build_pool(bt, ctxs, layers, num_pages, H, page_tokens, hd, seed, fill=None):
    """Pool [layers, 2, num_pages, H, page_tokens, hd] bf16: NaN everywhere except the cached positions 0..ctx-1 of every
    row, which hold K / V of a contiguous [rows, max_ctx, H, hd] pair (random N(0, 1), or fill(kv_index, rows, T) when
    given).  Returns (pool, Kc, Vc) with Kc / Vc the contiguous float32 tensors."""
    rows = len(ctxs)
    T = max(max(ctxs), 1)
    g = torch.Generator().manual_seed(seed)
    if fill is None:
        Kc = torch.randn(rows, T, H, hd, generator=g).bfloat16().float()
        Vc = torch.randn(rows, T, H, hd, generator=g).bfloat16().float()
    else:
        Kc, Vc = fill(0, rows, T).bfloat16().float(), fill(1, rows, T).bfloat16().float()
    pool = torch.full((layers, 2, num_pages, H, page_tokens, hd), float("nan"), dtype=torch.bfloat16)
    for l in range(layers):
        for r, c in enumerate(ctxs):
            t = torch.arange(c)
            pages, slots = bt[r].long()[t // page_tokens], t % page_tokens
            pool[l, 0][pages, :, slots] = Kc[r, :c].bfloat16()
            pool[l, 1][pages, :, slots] = Vc[r, :c].bfloat16()
    return pool, Kc, Vc


def test_reference_paged_gather_equals_contiguous_attention():
    """CPU self-test of the reference: on a random permuted table (page_tokens 4, rotary 24 at head_dim 64, layer 1 of 2),
    ref_decode equals plain float64 attention over the same tokens laid out contiguously, rotary applied to the whole
    sequence at positions 0..ctx as rotary64 does."""
    H, hd, pt, rd = 3, 64, 4, 24
    ctxs = [0, 1, 5, 17, 40]
    bt, num_pages = build_table("perm", ctxs, pt, 11)
    pool, Kc, Vc = build_pool(bt, ctxs, 2, num_pages, H, pt, hd, 12)
    qkv = torch.randn(len(ctxs), 3 * H * hd, generator=torch.Generator().manual_seed(13)).bfloat16()
    ref = ref_decode(qkv, pool, 1, pt, bt, torch.tensor(ctxs), H, hd, rd)
    for r, c in enumerate(ctxs):
        q, k, v = qkv[r].double().view(3, H, hd).unbind(0)
        # the whole row's keys rotated at positions 0..c: the cached ones (already rotated when they were stored) are
        # un-rotated first, so rotating the sequence must reproduce them
        pos = torch.arange(c + 1, dtype=torch.float64)
        inv = 10000.0 ** (-2.0 * torch.arange(rd // 2, dtype=torch.float64) / rd)
        ang = pos[:, None] * inv[None, :]
        cs, sn = torch.cos(ang)[:, None, :], torch.sin(ang)[:, None, :]
        Kseq = torch.cat([Kc[r, :c].double(), k[None]], 0)
        raw = Kseq.clone()
        a, b = Kseq[:c, :, 0:rd:2], Kseq[:c, :, 1:rd:2]
        raw[:c, :, 0:rd:2] = a * cs[:c] + b * sn[:c]        # inverse rotation of the cached keys
        raw[:c, :, 1:rd:2] = b * cs[:c] - a * sn[:c]
        rot = raw.clone()
        a, b = raw[..., 0:rd:2], raw[..., 1:rd:2]
        rot[..., 0:rd:2] = a * cs - b * sn
        rot[..., 1:rd:2] = b * cs + a * sn
        rot[c] = rot[c].bfloat16().double()
        qr = q.clone()
        qr[:, 0:rd:2] = q[:, 0:rd:2] * cs[c] - q[:, 1:rd:2] * sn[c]
        qr[:, 1:rd:2] = q[:, 1:rd:2] * cs[c] + q[:, 0:rd:2] * sn[c]
        V = torch.cat([Vc[r, :c].double(), v[None]], 0)
        p = (torch.einsum("hd,thd->ht", qr, rot) / hd ** 0.5).softmax(-1)
        want = torch.einsum("ht,thd->hd", p, V).reshape(-1)
        assert (ref[r] - want).abs().max().item() < 1e-10, r
        assert torch.isfinite(ref[r]).all()
    # the gather really goes through the table: a different permutation of the same tokens gives the same result,
    # a table pointing one row at another row's pages does not
    bt2, _ = build_table("perm", ctxs, pt, 99)
    pool2, _, _ = build_pool(bt2, ctxs, 2, num_pages, H, pt, hd, 12)
    assert torch.allclose(ref, ref_decode(qkv, pool2, 1, pt, bt2, torch.tensor(ctxs), H, hd, rd), atol=1e-12)
    wrong = bt.clone()
    wrong[4, :5] = bt[3, :5]
    assert not torch.allclose(ref[4], ref_decode(qkv, pool, 1, pt, wrong, torch.tensor(ctxs), H, hd, rd)[4], atol=1e-3)


# ------------------------------------------------------------------------------------------------ the route matrix
def _matrix():
    cases = []
    for hd, rds in ((64, (0, 64, 24, 2)), (128, (0, 64)), (256, (0, 64))):
        for rd in rds:
            for pt in (1, 2, 16):
                for table in ("identity", "perm", "beam"):
                    for ldo in (1, 5):
                        cases.append((hd, rd, pt, table, ldo))
    return cases


MATRIX = _matrix()
H_ = 2


def _case_id(c):
    hd, rd, pt, table, ldo = c
    return "hd%d-rot%d-pt%d-%s-ldo%dx-%s-%s" % (hd, rd, pt, table, ldo, CTX_TAG, expected_kernel(hd))


def _setup(case, seed, ctxs=CTXS, layers=2, fill=None, qkv=None):
    hd, rd, pt, table, ldo = case
    bt, num_pages = build_table(table, ctxs, pt, seed)
    pool, _, _ = build_pool(bt, ctxs, layers, num_pages, H_, pt, hd, seed + 1, fill)
    if qkv is None:
        qkv = torch.randn(len(ctxs), 3 * H_ * hd, generator=torch.Generator().manual_seed(seed + 2)).bfloat16()
    return bt, pool.cuda(), qkv.cuda(), torch.tensor(ctxs, dtype=torch.int32)


def _run(eng, case, bt, pool, qkv, ctx, layer=1):
    hd, rd, pt, table, ldo = case
    out = eng.op_attention_decode(qkv, pool, layer, pt, bt, ctx, H_, hd, rotary_dim=rd, ldo=ldo * H_ * hd)
    return out[:, :H_ * hd]


@gpu
@pytest.mark.parametrize("case", MATRIX, ids=[_case_id(c) for c in MATRIX])
def test_route_matrix_matches_float64(tiny_engine, case):
    hd, rd, pt, table, ldo = case
    seed = hd * 31 + rd * 7 + pt
    bt, pool, qkv, ctx = _setup(case, seed)
    before = pool.clone()
    out_full = tiny_engine.op_attention_decode(qkv, pool, 1, pt, bt, ctx, H_, hd, rotary_dim=rd, ldo=ldo * H_ * hd)
    torch.cuda.synchronize()
    out = out_full[:, :H_ * hd]
    assert_close(out, ref_decode(qkv, before, 1, pt, bt, ctx, H_, hd, rd), _case_id(case))
    if ldo > 1:   # nothing written past a row's H*hd columns
        assert (out_full[:, H_ * hd:] == 0).all()
    # the cache append: the slot of position ctx of every row holds bf16(rotated k_new) and v_new; nothing else changed
    expect = before.clone()
    exact = torch.ones_like(before, dtype=torch.bool)
    for r, c in enumerate(ctx.tolist()):
        q, kn, vn = new_token(qkv[r], H_, hd, c, rd)
        page, slot = int(bt[r, c // pt]), c % pt
        expect[1, 0, page, :, slot] = kn.bfloat16()
        expect[1, 1, page, :, slot] = vn.bfloat16()
        if rd:   # fp32 rotation in the kernel, float64 here: a rotated element may round to the neighbouring bf16
            exact[1, 0, page, :, slot, :rd] = False
    got = pool.view(torch.int16)
    assert torch.equal(got[exact], expect.view(torch.int16)[exact]), _case_id(case)
    if rd:
        a, b = pool[~exact].double(), expect[~exact].double()
        assert ((a - b).abs() <= bf16_ulp(b)).all(), _case_id(case)
    # deterministic: the same call on the same pool, bit for bit
    pool2 = before.clone()
    again = _run(tiny_engine, case, bt, pool2, qkv, ctx)
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int16), again.view(torch.int16))
    assert torch.equal(pool.view(torch.int16), pool2.view(torch.int16))


def test_matrix_covers_what_it_claims():
    assert {c[0] for c in MATRIX} == {64, 128, 256}
    assert {c[1] for c in MATRIX if c[0] == 64} == {0, 2, 24, 64}
    assert {c[2] for c in MATRIX} == {1, 2, 16} and {c[3] for c in MATRIX} == {"identity", "perm", "beam"}
    assert max(CTXS) < MAXP and max(CTXS) > 3 * WIDE_TILE
    for b in (32, WIDE_TILE, 2 * WIDE_TILE):
        assert {b - 1, b, b + 1} <= set(CTXS)
    # the beam-like table shares pages between rows, and every page id a row uses is in range
    for pt in (1, 2, 16):
        bt, n = build_table("beam", CTXS, pt, 0)
        used = [set(bt[r, :c // pt + 1].tolist()) for r, c in enumerate(CTXS)]
        assert used[3] & used[4] and all(max(u) < n - 1 for u in used)
        assert len({int(bt[r, c // pt]) for r, c in enumerate(CTXS)}) == len(CTXS)   # the new token's page is private


@gpu
def test_op_attention_decode_rejects_bad_arguments(tiny_engine):
    import ctypes as C
    eng = tiny_engine
    case = (64, 0, 2, "identity", 1)
    bt, pool, qkv, ctx = _setup(case, 3, ctxs=[0, 5])
    with pytest.raises(RuntimeError, match="layer 2 outside"):
        eng.op_attention_decode(qkv, pool, 2, 2, bt, ctx, H_, 64)
    with pytest.raises(RuntimeError, match="head_dim 96"):
        p96 = torch.zeros(2, 2, 4, H_, 2, 96, dtype=torch.bfloat16, device="cuda")
        eng.op_attention_decode(torch.zeros(2, 3 * H_ * 96, dtype=torch.bfloat16), p96, 0, 2, bt, ctx, H_, 96)
    out = torch.empty(2, H_ * 64, dtype=torch.bfloat16, device="cuda")
    btd, cld = bt.cuda(), ctx.cuda()
    args = lambda **kw: [eng._h, C.c_void_p(qkv.data_ptr()), C.c_void_p(out.data_ptr()), H_ * 64, 2, H_, 64, 0.125,
                         C.c_void_p(pool.data_ptr()), 2, 0, pool.shape[2], kw.get("pt", 2), MAXP,
                         kw.get("bt", C.c_void_p(btd.data_ptr())), C.c_void_p(cld.data_ptr()), 0, None]
    for kw, msg in (({"pt": 0}, "page_tokens=0"), ({"bt": None}, "null argument")):
        assert eng.lib.ccb_op_attention_decode(*args(**kw)) != 0
        assert msg in eng.lib.ccb_last_error(eng._h).decode()
    # the context stays usable
    assert_close(_run(eng, case, bt, pool, qkv, ctx), ref_decode(qkv, pool, 1, 2, bt, ctx, H_, 64))


# ------------------------------------------------------------------------------------------------ which kernel ran
def _cuda_kernel_names(prof):
    cuda = torch.autograd.DeviceType.CUDA
    evs = [(e.time_range.start, e.name) for e in prof.events() if e.device_type == cuda]
    if not evs:
        evs = [(e.start_ns(), e.name()) for e in prof.profiler.kineto_results.events() if e.device_type() == cuda]
    return [n for _, n in sorted(evs)]


@gpu
def test_profiler_names_the_expected_kernel_for_every_case(tiny_engine):
    from torch.profiler import ProfilerActivity, profile
    inputs = [_setup(c, i, ctxs=[3, 40]) for i, c in enumerate(MATRIX)]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        # (the first device activity of a profiling session can go unrecorded in a process that profiled before)
        torch.ones(8, device="cuda").add_(1)
        torch.cuda.synchronize()
        for c, (bt, pool, qkv, ctx) in zip(MATRIX, inputs):
            _run(tiny_engine, c, bt, pool, qkv, ctx)
        torch.cuda.synchronize()
    ran = [kernel_of(n) for n in _cuda_kernel_names(prof) if kernel_of(n)]
    want = [expected_kernel(c[0]) for c in MATRIX]
    assert len(ran) == len(want), (len(ran), len(want))
    bad = [(_case_id(c), w, r) for c, w, r in zip(MATRIX, want, ran) if w != r]
    assert not bad, bad[:10]
    assert set(ran) == {"warp<64>", "warp<128>", "wide<256>"}


# ------------------------------------------------------------------------------------------------ structured probes
PROBES = [(hd, pt) for hd in (64, 128, 256) for pt in (1, 2, 16)]


def _probe_id(p):
    return "hd%d-pt%d-%s" % (p[0], p[1], expected_kernel(p[0]))


def _signs(g, *shape):
    return torch.randint(0, 2, shape, generator=g).float() * 2 - 1


def _dominant_rows(pt):
    """(ctx, dominant position) pairs: first and last cached token, both sides of a page boundary and of the wide
    kernel's 96-token tiles, and the tile boundary as the last cached token."""
    pb = 5 * pt if pt > 1 else 77
    return [(200, 0), (200, 199), (200, pb - 1), (200, pb), (200, WIDE_TILE - 1), (200, WIDE_TILE),
            (411, 2 * WIDE_TILE), (411, 410), (97, WIDE_TILE), (97, 0), (33, 32), (1, 0), (32, 31)]


def _probe_inputs(hd, pt, rows, q_fn, k_fn, v_fn, seed):
    """qkv and pool from per-row functions of (generator, row index, ctx) -> q [H, hd], keys / values [ctx + 1, H, hd] (the
    last one is the new token's)."""
    g = torch.Generator().manual_seed(seed)
    ctxs = [c for c, _ in rows]
    T = max(ctxs) + 1
    K = torch.zeros(len(rows), T, H_, hd)
    V = torch.zeros(len(rows), T, H_, hd)
    qkv = torch.zeros(len(rows), 3, H_, hd)
    for r, (c, extra) in enumerate(rows):
        K[r, :c + 1] = k_fn(g, r, c, extra)
        V[r, :c + 1] = v_fn(g, r, c, extra)
        qkv[r, 0] = q_fn(g, r, c, extra, K[r])
        qkv[r, 1], qkv[r, 2] = K[r, c], V[r, c]
    fill = lambda kv, n, t: (K if kv == 0 else V)[:, :t]
    case = (hd, 0, pt, "perm", 1)
    bt, pool, qkv_d, ctx = _setup(case, seed, ctxs=ctxs, fill=fill, qkv=qkv.reshape(len(rows), -1).bfloat16())
    return case, bt, pool, qkv_d, ctx, K.bfloat16().double(), V.bfloat16().double()


@gpu
@pytest.mark.parametrize("hd,pt", PROBES, ids=[_probe_id(p) for p in PROBES])
def test_dominant_key_gives_its_v_row(tiny_engine, hd, pt):
    """Key t scores >= 30 above every other key (the new token's included): the output is V row t within one bf16 ulp.
    This pins the page mapping: a key or value read from another slot, page or tile shows as a wrong row."""
    rows = _dominant_rows(pt)
    small = lambda g, r, c, t: 0.05 * torch.randn(c + 1, H_, hd, generator=g)

    def keys(g, r, c, t):
        k = small(g, r, c, t)
        k[t] = _signs(g, H_, hd)
        return k

    q = lambda g, r, c, t, K: K[t] * (48.0 / hd ** 0.5)          # score of key t: 48; of any other |.| <~ 10
    case, bt, pool, qkv, ctx, K, V = _probe_inputs(hd, pt, rows, q, keys, lambda g, r, c, t: torch.randn(c + 1, H_, hd, generator=g), hd + pt)
    ref, probs = ref_decode(qkv, pool.clone(), 1, pt, bt, ctx, H_, hd, return_probs=True)
    for r, (c, t) in enumerate(rows):
        assert probs[r][:, t].min().item() > 1 - 1e-9, (c, t)
    out = _run(tiny_engine, case, bt, pool, qkv, ctx).double().cpu()
    want = torch.stack([V[r, t].reshape(-1) for r, (c, t) in enumerate(rows)])
    err = (out - want).abs()
    bad = (err > bf16_ulp(want)).nonzero()
    assert not len(bad), [(rows[int(i)], int(j), float(err[i, j])) for i, j in bad[:5]]


@gpu
@pytest.mark.parametrize("hd,pt", PROBES, ids=[_probe_id(p) for p in PROBES])
def test_new_token_dominates(tiny_engine, hd, pt):
    rows = [(c, None) for c in (0, 1, 31, 33, 96, 97, 200, 411)]
    keys = lambda g, r, c, _: torch.cat([0.05 * torch.randn(c, H_, hd, generator=g), _signs(g, 1, H_, hd)], 0)
    q = lambda g, r, c, _, K: K[c] * (48.0 / hd ** 0.5)
    case, bt, pool, qkv, ctx, K, V = _probe_inputs(hd, pt, rows, q, keys, lambda g, r, c, _: torch.randn(c + 1, H_, hd, generator=g), 2 * hd + pt)
    out = _run(tiny_engine, case, bt, pool, qkv, ctx).double().cpu()
    want = torch.stack([V[r, c].reshape(-1) for r, (c, _) in enumerate(rows)])
    assert ((out - want).abs() <= bf16_ulp(want)).all()


@gpu
@pytest.mark.parametrize("hd,pt", PROBES, ids=[_probe_id(p) for p in PROBES])
def test_constant_v_is_reproduced_to_one_ulp(tiny_engine, hd, pt):
    rows = [(c, None) for c in CTXS]
    rnd = lambda g, r, c, _: torch.randn(c + 1, H_, hd, generator=g)
    case, bt, pool, qkv, ctx, K, V = _probe_inputs(hd, pt, rows, lambda g, r, c, _, K: torch.randn(H_, hd, generator=g) * 2,
                                                   rnd, lambda g, r, c, _: torch.full((c + 1, H_, hd), 3.0), 3 * hd + pt)
    out = _run(tiny_engine, case, bt, pool, qkv, ctx).float()
    assert torch.isfinite(out).all()
    assert (out - 3.0).abs().max().item() <= 2.0 ** -6


@gpu
@pytest.mark.parametrize("hd,pt", PROBES, ids=[_probe_id(p) for p in PROBES])
def test_identical_keys_give_the_mean_of_v(tiny_engine, hd, pt):
    rows = [(c, None) for c in CTXS]
    keys = lambda g, r, c, _: torch.randn(1, H_, hd, generator=g).expand(c + 1, H_, hd)
    case, bt, pool, qkv, ctx, K, V = _probe_inputs(hd, pt, rows, lambda g, r, c, _, K: torch.randn(H_, hd, generator=g),
                                                   keys, lambda g, r, c, _: torch.randn(c + 1, H_, hd, generator=g), 4 * hd + pt)
    mean = torch.stack([V[r, :c + 1].mean(0).reshape(-1) for r, (c, _) in enumerate(rows)])
    assert_close(_run(tiny_engine, case, bt, pool, qkv, ctx), mean, "mean of V")


@gpu
@pytest.mark.parametrize("hd,pt", PROBES, ids=[_probe_id(p) for p in PROBES])
def test_negative_scores(tiny_engine, hd, pt):
    """Every score <= -30 (keys positive multiples of u, queries negative ones): a zero-filled or skipped slot that took part
    would score 0 and take almost all the weight."""
    rows = [(c, None) for c in CTXS]
    u = _signs(torch.Generator().manual_seed(hd + pt), H_, hd)
    keys = lambda g, r, c, _: u * (1 + 0.5 * torch.rand(c + 1, H_, 1, generator=g))
    q = lambda g, r, c, _, K: -u * (40 / hd ** 0.5) * (1 + torch.rand(H_, 1, generator=g))
    case, bt, pool, qkv, ctx, K, V = _probe_inputs(hd, pt, rows, q, keys, lambda g, r, c, _: torch.randn(c + 1, H_, hd, generator=g), 5 * hd + pt)
    ref, probs = ref_decode(qkv, pool.clone(), 1, pt, bt, ctx, H_, hd, return_probs=True)
    Q = qkv.double().cpu().view(len(rows), 3, H_, hd)[:, 0]
    for r, (c, _) in enumerate(rows):
        assert (torch.einsum("hd,thd->ht", Q[r], K[r, :c + 1]) * hd ** -0.5).max().item() <= -30
    assert_close(_run(tiny_engine, case, bt, pool, qkv, ctx), ref, "negative scores")


@gpu
@pytest.mark.parametrize("hd,pt", PROBES, ids=[_probe_id(p) for p in PROBES])
def test_peaked_scores_across_tiles(tiny_engine, hd, pt):
    """One key scores ~100, the others ~N(0, 100 / sqrt(hd)) (exp(100) overflows fp32: the running maximum must be
    subtracted).  The peak sits in a later tile than the first (the online softmax must rescale what earlier tiles
    accumulated), in the first tile, and at the last cached token."""
    rows = [(200, 150), (200, 10), (411, 300), (411, 95), (97, 96), (193, 192), (64, 40)]
    keys = lambda g, r, c, t: _signs(g, c + 1, H_, hd)
    q = lambda g, r, c, t, K: K[t] * (100 / hd ** 0.5)
    case, bt, pool, qkv, ctx, K, V = _probe_inputs(hd, pt, rows, q, keys, lambda g, r, c, t: torch.randn(c + 1, H_, hd, generator=g), 6 * hd + pt)
    ref = ref_decode(qkv, pool.clone(), 1, pt, bt, ctx, H_, hd)
    assert_close(_run(tiny_engine, case, bt, pool, qkv, ctx), ref, "peaked")
    want = torch.stack([V[r, t].reshape(-1) for r, (c, t) in enumerate(rows)])
    assert (ref.cpu() - want).abs().max().item() < 0.05


# ------------------------------------------------------------------------------------------------ the persistent kernel
D_, HEADS_, VOCAB_ = 1600, 25, 2048
HD_ = D_ // HEADS_
MAX_ROWS, MAX_CTX = 256, 264
Q_WEIGHT_GAIN = 8.0           # q slice of c_attn x 8 (exact in bf16) ...
Q_BIAS, K_BIAS = 4.0, 2.0     # ... and per head a q bias +4 u, k bias -2 u (u = +-1): see _peaked_state_dict

# (page_tokens, S0): the step's context is S0.  A row holds its page ids one per lane while (ctx >> log2(page_tokens)) + 1
# <= 32, else reads each token's page id from the block table; each pair below has one S0 on each side.
MEGA_CASES = [(1, 31), (1, 32), (1, 33), (1, 200), (2, 63), (2, 64), (4, 127), (4, 128), (4, 256), (8, 255), (8, 256)]
MEGA_ROWS = [7, 64, 129, 256]


def in_warp(pt, ctx):
    return (ctx // pt) + 1 <= 32


def _peaked_state_dict(cfg, seed):
    """synthetic GPT-2 weights with peaked attention whose scores all sit far below zero.  The q slice of c_attn is
    scaled by 8 and gets a bias +4 u per head, the k slice a bias -2 u (u a +-1 vector per head): the top key of a query
    takes most of the weight (median 0.77 on float64 of these weights) and every score is shifted by about -32 (q.b_k,
    the largest score stays below -15), so that a zero-filled slot the kernel wrongly lets in (score 0) takes all of it.
    The bias on k cancels in k_t - sum_s p_s k_s and so leaves the q-ulp tolerance of _check_attention alone."""
    from clipcap_b200 import synthetic
    sd = synthetic.lm_state_dict(cfg, seed, "cpu")
    g = torch.Generator().manual_seed(seed + 1)
    u = _signs(g, HEADS_, HD_).reshape(-1)
    w = sd["transformer.h.0.attn.c_attn.weight"]
    w[:, :D_] *= Q_WEIGHT_GAIN
    b = sd["transformer.h.0.attn.c_attn.bias"]
    b[:D_] = Q_BIAS * u
    b[D_:2 * D_] = -K_BIAS * u
    b[2 * D_:] = 0.1 * torch.randn(D_, generator=g)
    return sd


_ENGINES = {}


@pytest.fixture(scope="module")
def mega_engines():
    yield _ENGINES
    for eng, _ in _ENGINES.values():
        eng.close()
    _ENGINES.clear()


def _mega_engine(engines, pt):
    if pt not in engines:
        import clipcap_b200 as cc
        cfg = cc.EngineConfig(lm_layers=1, lm_vocab=VOCAB_, map_kind="none", vit=False, max_images=MAX_ROWS,
                              max_beam=3 if pt == 1 else 1, max_ctx=MAX_CTX, page_tokens=pt)
        eng = cc.Engine(cfg)
        sd = _peaked_state_dict(cfg, 4242)
        eng.load_state_dict(sd, prefix="language_model.")
        eng.check_weights()
        engines[pt] = (eng, {k: v.double().cuda() for k, v in sd.items()})
    return engines[pt]


def _one_step(eng, prefix, p, mega):
    """prefill + one decode step on the persistent kernel (mega) or the operator chain: the pool, the block table, the
    attention output and (chain) the fused qkv of the step."""
    assert eng.lib.ccb_debug_set_mega(eng._h, 1 if mega else 0) == 1
    try:
        eng.generate(prefix, p)
        L, H, hd, pt, num_pages, maxp = eng.debug_kv_layout()
        rows = prefix.shape[0] * (p.beam_size if p.mode == 2 else 1)
        pool = eng.debug_copy_buffer(6, L * 2 * num_pages * H * pt * hd, torch.bfloat16).view(L, 2, num_pages, H, pt, hd)
        bt = eng.debug_copy_buffer(7, rows * maxp, torch.int32).view(rows, maxp)
        att = eng.debug_copy_buffer(2, rows * D_, torch.bfloat16).view(rows, D_)
        qkv = eng.debug_copy_buffer(5, rows * 3 * D_, torch.bfloat16).view(rows, 3 * D_)
        torch.cuda.synchronize()
    finally:
        eng.lib.ccb_debug_set_mega(eng._h, 1)
    return pool, bt, att, qkv, pt


def _prefix_kv_ref(sd, prefix):
    """bf16(bf16(LN_1(prefix + wpe[pos])) W_{k|v} + b_{k|v}) in float64 -> K, V [N, S0, H, hd], and the error one bf16
    ulp of every LayerNorm output would cause (root-sum-square over the d inputs, 4 sigma)."""
    N, S0, d = prefix.shape
    h = prefix.double() + sd["transformer.wpe.weight"][:S0][None]
    mu, var = h.mean(-1, keepdim=True), h.var(-1, unbiased=False, keepdim=True)
    x = ((h - mu) / torch.sqrt(var + 1e-5) * sd["transformer.h.0.ln_1.weight"] + sd["transformer.h.0.ln_1.bias"])
    x = x.bfloat16().double()
    w, b = sd["transformer.h.0.attn.c_attn.weight"], sd["transformer.h.0.attn.c_attn.bias"]
    out, slack = [], []
    for j in (1, 2):
        wj = w[:, j * d:(j + 1) * d]
        out.append((x @ wj + b[j * d:(j + 1) * d]).bfloat16().double().view(N, S0, HEADS_, HD_))
        slack.append(4 * torch.sqrt((bf16_ulp(x) ** 2) @ (wj ** 2)).view(N, S0, HEADS_, HD_))
    return out[0], out[1], slack[0], slack[1]


def _check_prefix_cache(pool, pt, table_of, K, V, sK, sV, what):
    """The pool's prefix K / V at the pages table_of(n) names for image n."""
    N, S0 = K.shape[:2]
    worst = 0.0
    for n in range(N):
        kk, vv = gather_kv(pool, 0, pt, table_of(n), S0)
        for got, ref, sl in ((kk, K[n], sK[n]), (vv, V[n], sV[n])):
            err = (got - ref).abs()
            tol = bf16_ulp(ref) + sl
            assert (err <= tol).all(), (what, n, (err - tol).max().item())
            worst = max(worst, (err / tol).max().item())
    return worst


def _check_appended(pool, pages, slot, qkv_c, sd, pos):
    """The k / v the persistent kernel appended for each row (page pages[r], slot `slot`) against the chain's qkv of the
    same step: within one bf16 ulp, plus what the two paths may legitimately differ by before that rounding.  The
    persistent kernel computes LN_1 itself, so its bf16 x may differ from the chain's by one ulp in some elements: 4 sigma
    of one ulp per element (as _prefix_kv_ref's slack), the largest over every token at position `pos`.  And it sums
    c_attn's products in another order (split-K partials against the GEMM's K loop: ~2 x 128 rounded additions of 2^-24
    over sum_i |x_i w_ik| <= sqrt(d) |w_k|_2).  Returns the worst err / tol."""
    rows = qkv_c.shape[0]
    w = sd["transformer.h.0.attn.c_attn.weight"]
    h = sd["transformer.wte.weight"] + sd["transformer.wpe.weight"][pos][None]
    x = ((h - h.mean(-1, keepdim=True)) / torch.sqrt(h.var(-1, unbiased=False, keepdim=True) + 1e-5)).bfloat16().double()
    worst = 0.0
    for j in (1, 2):
        wj = w[:, j * D_:(j + 1) * D_]
        got = pool[0, j - 1][pages.long().to(pool.device), :, slot].double().reshape(rows, D_)
        want = qkv_c[:, j * D_:(j + 1) * D_].double()
        slack = 4 * torch.sqrt((bf16_ulp(x) ** 2) @ (wj ** 2)).max(0).values + 2.0 ** -16 * D_ ** 0.5 * wj.norm(dim=0)
        tol = bf16_ulp(torch.maximum(want.abs(), got.abs())) + slack
        err = (got - want).abs()
        assert (err <= tol).all(), ("appended", "kv"[j - 1], (err - tol).max().item(), (err / tol).max().item())
        worst = max(worst, (err / tol).max().item())
    return worst


def _check_attention(att, qkv, pool, pt, bt, ctx, what):
    """att [rows, d] against float64 attention of the chain's q over the pool's K / V at positions 0..ctx.  Tolerance per
    element: one bf16 ulp of the reference plus the first-order effect of one bf16 ulp in every element of q (the
    persistent kernel sums c_attn's split-K partials in another order, so its q may differ from the chain's in the last
    bit): sum_i |d out_j / d q_i| ulp(q_i), d out / d q = scale * sum_t p_t (v_t - out)(k_t - sum_s p_s k_s)^T."""
    rows = att.shape[0]
    scale = HD_ ** -0.5
    q = qkv[:, :D_].double().view(rows, HEADS_, HD_)
    worst, tops = 0.0, []
    for r in range(rows):
        K, V = gather_kv(pool, 0, pt, bt[r], ctx + 1)
        p = (torch.einsum("hd,thd->ht", q[r], K) * scale).softmax(-1)
        o = torch.einsum("ht,thd->hd", p, V)
        kbar = torch.einsum("ht,thd->hd", p, K)
        A = p[:, :, None] * (V.transpose(0, 1) - o[:, None])          # [h, t, j]
        J = scale * (A.transpose(1, 2) @ (K.transpose(0, 1) - kbar[:, None]))   # [h, j, i]
        tol = bf16_ulp(o) + torch.einsum("hji,hi->hj", J.abs(), bf16_ulp(q[r])) + 1e-6
        err = (att[r].double().view(HEADS_, HD_) - o).abs()
        assert torch.isfinite(att[r].float()).all(), (what, r)
        assert (err <= tol).all(), (what, r, (err - tol).max().item(), (err / tol).max().item())
        worst = max(worst, (err / tol).max().item())
        tops.append(p.max(-1).values)
    return worst, torch.cat(tops)


def _greedy_cases():
    return [(pt, s0, rows) for pt, s0 in MEGA_CASES for rows in MEGA_ROWS]


def _mega_id(c):
    pt, s0, rows = c
    return "pt%d-S0_%d-rows%d-%s" % (pt, s0, rows, "in-warp" if in_warp(pt, s0) else "table")


@gpu
@pytest.mark.parametrize("case", _greedy_cases(), ids=[_mega_id(c) for c in _greedy_cases()])
def test_persistent_kernel_attention_matches_float64(mega_engines, case):
    """One GPT-2-shaped layer (d 1600, 25 heads: chain and persistent kernel see identical inputs), prefill + exactly one
    decode step.  Checks: the prefix K / V the prefill route wrote (S0 crosses umma / mma / scalar at 64 / 65, 128 / 129)
    at the pages the table names; the k / v the persistent kernel appended at position S0 within one bf16 ulp of the
    chain's qkv; the attention output of both decode paths against float64 attention over the pool.  page_tokens 16 is
    not here: a prefix of at most 256 tokens never leaves the in-warp page limit within one step ((256 >> 4) + 1 = 17)."""
    pt, S0, rows = case
    eng, sd = _mega_engine(mega_engines, pt)
    prefix = (0.5 * torch.randn(rows, S0, D_, generator=torch.Generator().manual_seed(S0 * 7 + rows))).cuda()
    p = eng.gen_params("greedy", 2, stop_token=-1, max_stops=0)
    pool_m, bt_m, att_m, _, ptm = _one_step(eng, prefix, p, True)
    pool_c, bt_c, att_c, qkv_c, _ = _one_step(eng, prefix, p, False)
    assert ptm == pt and torch.equal(bt_m, bt_c)
    K, V, sK, sV = _prefix_kv_ref(sd, prefix)
    w = _check_prefix_cache(pool_m, pt, lambda n: bt_m[n], K, V, sK, sV, "prefix")
    wa = _check_appended(pool_m, bt_m[:, S0 // pt], S0 % pt, qkv_c, sd, S0)
    wm, tops = _check_attention(att_m, qkv_c, pool_m, pt, bt_m, S0, "persistent")
    wc, _ = _check_attention(att_c, qkv_c, pool_c, pt, bt_c, S0, "chain")
    assert tops.median().item() > 0.5, tops.median().item()
    print("%s: max err / tol prefix %.3f appended %.3f persistent %.3f chain %.3f; median top weight %.3f" %
          (_mega_id(case), w, wa, wm, wc, tops.median().item()))


@gpu
@pytest.mark.parametrize("S0", [33, 100])
def test_persistent_kernel_beam_step_over_shared_prefix_pages(mega_engines, S0):
    """Beam 3 (page_tokens 1, prefix pages shared by an image's beams).  The block table read back afterwards has been
    permuted by the beam step; the decode step's own table follows the layout of init_state_kernel: image n owns pages
    [n * ppi, (n + 1) * ppi), ppi = S0 + beam * T, the S0 prefix pages are shared and beam k's token of this step goes to
    page n * ppi + S0 + k."""
    eng, sd = _mega_engine(mega_engines, 1)
    N, beam, T = 5, 3, 2
    prefix = (0.5 * torch.randn(N, S0, D_, generator=torch.Generator().manual_seed(S0))).cuda()
    p = eng.gen_params("beam", T, stop_token=-1, max_stops=0, beam_size=beam)
    pool_m, _, att_m, _, pt = _one_step(eng, prefix, p, True)
    pool_c, _, att_c, qkv_c, _ = _one_step(eng, prefix, p, False)
    assert pt == 1
    ppi = S0 + beam * T
    bt = torch.zeros(N * beam, S0 + 1, dtype=torch.int32)
    for n in range(N):
        for k in range(beam):
            bt[n * beam + k, :S0] = torch.arange(n * ppi, n * ppi + S0)
            bt[n * beam + k, S0] = n * ppi + S0 + k
    K, V, sK, sV = _prefix_kv_ref(sd, prefix)
    _check_prefix_cache(pool_m, 1, lambda n: bt[n * beam], K, V, sK, sV, "beam prefix")
    wa = _check_appended(pool_m, bt[:, S0], 0, qkv_c, sd, S0)
    wm, tops = _check_attention(att_m, qkv_c, pool_m, 1, bt, S0, "persistent beam")
    wc, _ = _check_attention(att_c, qkv_c, pool_c, 1, bt, S0, "chain beam")
    assert tops.median().item() > 0.5
    print("beam S0 %d: max err / tol appended %.3f persistent %.3f chain %.3f" % (S0, wa, wm, wc))
