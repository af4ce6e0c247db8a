"""Continuous batching for beam search (Engine.caption_dataset_continuous_beam / ccb_caption_dataset_beam) against
caption_dataset in beam mode and the reference's loop, on the golden tiny checkpoints.  The stop token is one of the
tokens the winning beams of caption_dataset emit most often: the one that ends groups earliest, so that groups finish at
different steps (a beam search on these weights rarely stops on the single most frequent one).

Where the work is identical (n == groups images, prefilled in one chunk as large as caption_dataset's single micro-batch,
and the same decode rows) the results are bit-identical, except that scores of groups whose beams have all stopped may
differ in the last bits: ccb_generate keeps stepping such a group and recomputes each score as (score / len) * len in
fp32, while the new path stops it there, as the reference does.

Elsewhere a refill prefills another number of images than a micro-batch and the decode step runs another number of
rows, so the last bits of the logits can differ and an image's winner may change where two captions are a near-tie:
both winners teacher-forced through lm_forward and scored by their mean log-probability lie within TIE of the reference
winner's score.  As in the beam rule of tests/test_gpu_config_parity.py, at least 99 % of the images must be identical
or tied, and at most one image per started hundred may be neither: a near-tie at the pruning to `beam` candidates can
keep a different caption alive, and the winners then differ by more than the tie (one image in 83 on this checkpoint
with 16 groups)."""
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
T = 24
TIE = 2e-2
ROUND_STEPS = 4        # decode steps per round (kRoundSteps in csrc/engine.cu)


def make_engine(name, max_images=64, mapper="sd_mapper"):
    import clipcap_b200 as cc
    fx = torch.load(os.path.join(GOLDEN, name + ".pt"), weights_only=False)
    all_feat = name == "tiny_allfeatures"
    cfg = cc.EngineConfig(
        lm_arch=fx.get("arch", "gpt2"), lm_d=fx["d"], lm_layers=2, lm_heads=fx["heads"], lm_vocab=fx["V"], lm_n_pos=64,
        lm_rotary_dim=fx.get("rotary_dim", 0), map_kind="transformer_all" if all_feat else "transformer",
        map_dim_clip=fx["dim_clip"], map_clip_len=fx["T"] if all_feat else fx["CL"], map_prefix_len=fx["P"],
        map_heads=fx["map_heads"], map_layers=2, vit_image=fx["vit_image"], vit_patch=fx["vit_patch"],
        vit_width=fx["vit_width"], vit_layers=fx["vit_layers"], vit_heads=fx["vit_heads"], vit_out=fx["dim_clip"],
        max_images=max_images, max_beam=5, max_ctx=32, page_tokens=4)
    eng = cc.Engine(cfg)
    eng.load_state_dict(fx["sd_lm"], prefix="language_model.")
    eng.load_state_dict(fx[mapper], prefix="clip_project.")
    eng.load_state_dict(fx["sd_vit"], prefix="visual.")
    eng.check_weights()
    return eng, fx


def images(fx, n, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 3, fx["vit_image"], fx["vit_image"], generator=g).cuda()


def set_mega(eng, on):
    return eng.lib.ccb_debug_set_mega(eng._h, 1 if on else 0)


def winners(res):
    """per image: the winning beam (argmax score, lowest index on ties) as a token list"""
    tok, ln, sc = res[0].cpu(), res[1].cpu(), res[2].cpu()
    out = []
    for i in range(tok.shape[0]):
        k = int(sc[i].argmax())
        out.append(tok[i, k, :int(ln[i, k])].tolist())
    return out


def frequent_winner_tokens(eng, fx, append_bos=-1):
    """The tokens the winning beams of caption_dataset emit most often on 64 images when nothing stops them"""
    p = eng.gen_params("beam", T, stop_token=-1, beam_size=5)
    counts = torch.zeros(fx["V"], dtype=torch.long)
    for w in winners(eng.caption_dataset(images(fx, 64, seed=99), p, append_bos=append_bos)):
        counts += torch.bincount(torch.tensor(w), minlength=fx["V"])
    return counts.argsort(descending=True).tolist()


def mean_logprob(eng, img, append_bos, caption):
    """the reference's decision quantity for one caption: its mean log-probability, teacher-forced"""
    prefix = eng.map_prefix(eng.vit_encode(img[None]))
    if append_bos >= 0:
        prefix = torch.cat([prefix, eng.embed_tokens(torch.tensor([[append_bos]], device=prefix.device))], 1)
    S0, L = prefix.shape[1], len(caption)
    if L > 1:
        prefix = torch.cat([prefix, eng.embed_tokens(torch.tensor([caption[:-1]], device=prefix.device))], 1)
    lp = F.log_softmax(eng.lm_forward(prefix)[0, S0 - 1:S0 - 1 + L].double(), -1)
    return float(lp.gather(-1, torch.tensor(caption, device=lp.device)[:, None]).mean())


def same_or_tied(eng, img, append_bos, ref, got):
    if ref == got:
        return True
    s_ref = mean_logprob(eng, img, append_bos, ref)
    return abs(s_ref - mean_logprob(eng, img, append_bos, got)) <= TIE * abs(s_ref)


def compare(eng, imgs, ref, got, append_bos=-1):
    """number of images whose winner is identical; asserts zeros past every length of `got` and that every differing
    winner is a near-tie"""
    gt, gl = got[0].cpu(), got[1].cpu()
    assert ((gl >= 1) & (gl <= T)).all()
    pos = torch.arange(gt.shape[-1])
    assert not gt.masked_fill(pos < gl[..., None], 0).any()
    same = tied = 0
    for i, (a, b) in enumerate(zip(winners(ref), winners(got))):
        if a == b:
            same += 1
        else:
            tied += same_or_tied(eng, imgs[i], append_bos, a, b)
    n = len(imgs)
    assert n - same - tied <= math.ceil(0.01 * n), (same, tied, n)
    if n >= 100:
        assert same >= 0.99 * n, (same, n)
    return same


def stop_token(eng, fx, cands, append_bos=-1):
    """among the candidates, the one with the shortest mean group length (longest beam) on 64 images"""
    imgs = images(fx, 64, seed=98)

    def mean_group_length(t):
        res = eng.caption_dataset(imgs, eng.gen_params("beam", T, stop_token=t, beam_size=5), append_bos=append_bos)
        return float(res[1].max(1).values.float().mean())

    return min(cands, key=mean_group_length)


@pytest.fixture(scope="module")
def gpt2():
    eng, fx = make_engine("tiny_gpt2")
    cands = frequent_winner_tokens(eng, fx)[:8]
    yield eng, fx, stop_token(eng, fx, cands), cands
    eng.close()


@pytest.mark.parametrize("mega", [True, False], ids=["persistent", "operator_chain"])
@pytest.mark.parametrize("beam", [2, 3, 5])
def test_bit_exact_where_the_work_is_identical(gpt2, beam, mega):
    eng, fx, stop, cands = gpt2
    set_mega(eng, mega)
    try:
        n = 12
        imgs = images(fx, n, seed=beam)
        p = eng.gen_params("beam", T, stop_token=-1, beam_size=beam)
        ref = eng.caption_dataset(imgs, p)
        got = eng.caption_dataset_continuous_beam(imgs, p, groups=n)
        for r, g in zip(ref, got[:3]):
            assert torch.equal(r, g)
        stopped = 0      # every frequent winner token that ends some beams early on these images
        for t in cands:
            p = eng.gen_params("beam", T, stop_token=t, beam_size=beam)
            ref = eng.caption_dataset(imgs, p)
            got = eng.caption_dataset_continuous_beam(imgs, p, groups=n)
            assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])
            torch.testing.assert_close(got[2], ref[2], rtol=1e-6, atol=0)
            stopped += bool((ref[1] < T).any())
        assert stopped > 0
    finally:
        set_mega(eng, True)


@pytest.mark.parametrize("groups", [1, 7, 16])
def test_many_images_few_groups(gpt2, groups):
    eng, fx, stop, cands = gpt2
    p = eng.gen_params("beam", T, stop_token=stop, beam_size=5)
    sizes = sorted({groups, 5 * groups + 3} | ({128} if groups == 16 else set()))
    for n in sizes:
        imgs = images(fx, n, seed=n)
        ref = eng.caption_dataset(imgs, p)
        got = eng.caption_dataset_continuous_beam(imgs, p, groups=groups)
        same = compare(eng, imgs, ref, got)
        if n == sizes[-1]:
            again = eng.caption_dataset_continuous_beam(imgs, p, groups=groups)
            for a, b in zip(again[:3], got[:3]):
                assert torch.equal(a, b)
            assert again[3] == got[3]
            print("groups %d, %d images: %d winners identical, %d decode steps" % (groups, n, same, got[3]))


def test_group_counts_agree(gpt2):
    eng, fx, stop, cands = gpt2
    p = eng.gen_params("beam", T, stop_token=stop, beam_size=5)
    imgs = images(fx, 5 * 16 + 3, seed=7)
    compare(eng, imgs, eng.caption_dataset_continuous_beam(imgs, p, groups=16),
            eng.caption_dataset_continuous_beam(imgs, p, groups=7))


def test_the_reference_loop_with_its_break(gpt2):
    """oracle.generate_beam (inference.py:70-148 with `if has_stopped.all(): break`) on the engine's own prefixes"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import clipcap_oracle as orc
    eng, fx, stop, cands = gpt2
    imgs = images(fx, 8, seed=31)
    got = winners(eng.caption_dataset_continuous_beam(imgs, eng.gen_params("beam", T, stop_token=stop, beam_size=5),
                                                      groups=3))
    prefix = eng.map_prefix(eng.vit_encode(imgs))
    lm = orc.OracleLM({k: v.float().cuda() for k, v in fx["sd_lm"].items()}, "gpt2", fx["heads"])
    same = 0
    for i in range(8):
        with torch.no_grad():
            rt, rl, _, order = orc.generate_beam(lm, prefix[i:i + 1].float(), beam_size=5, entry_length=T,
                                                 stop_token=stop, use_cache=True)
        k = int(order[0])
        ref = rt[k, :int(rl[k])].tolist()
        same += ref == got[i]
        assert same_or_tied(eng, imgs[i], -1, ref, got[i]), (i, ref, got[i])
    print("reference loop: %d of 8 winners identical" % same)


@pytest.mark.parametrize("name", ["tiny_gptj", "tiny_allfeatures"])
def test_gptj_and_all_features_mapper_with_bos(name):
    eng, fx = make_engine(name, max_images=16, mapper="sd_mapper_pos" if name == "tiny_allfeatures" else "sd_mapper")
    set_mega(eng, False)
    try:
        bos = 1
        stop = stop_token(eng, fx, frequent_winner_tokens(eng, fx, append_bos=bos)[:8], append_bos=bos)
        p = eng.gen_params("beam", T, stop_token=stop, beam_size=5)
        imgs = images(fx, 2 * 16 + 3, seed=3)
        compare(eng, imgs, eng.caption_dataset(imgs, p, append_bos=bos),
                eng.caption_dataset_continuous_beam(imgs, p, groups=16, append_bos=bos), append_bos=bos)
    finally:
        eng.close()


def test_decode_steps_follow_the_work(gpt2):
    """A group holds its unit for its length - 1 decode steps rounded up to a whole round, plus the round that runs
    while the host reads the state; its length is its longest beam's.  Stated as in tests/test_gpu_continuous.py."""
    eng, fx, stop, cands = gpt2
    groups, K = 16, ROUND_STEPS
    n = 5 * groups + 3
    imgs = images(fx, n, seed=23)

    p = eng.gen_params("beam", T, stop_token=stop, beam_size=5)
    total = int(eng.caption_dataset(imgs, p)[1].max(1).values.sum())
    l0 = eng.launch_count
    tok, lens, scores, steps = eng.caption_dataset_continuous_beam(imgs, p, groups=groups)
    assert eng.launch_count > l0
    print("%d images, mean group length %.1f, %d decode steps" % (n, total / n, steps))
    assert steps % K == 0
    assert steps <= math.ceil((total + 2 * K * n) / groups) + T + 2 * K, (steps, total)
    assert total / n < T - 1                  # groups stop early
    assert steps < math.ceil(n / groups) * (T - 1), (steps, total)


def still_works(eng, fx):
    p = eng.gen_params("greedy", 10, stop_token=fx["stop_id"], max_stops=1)
    tokens, lengths, _ = eng.generate(fx["prefix"], p)
    tokens, lengths = tokens.cpu(), lengths.cpu()
    for i, want in enumerate(fx["greedy"]):
        assert tokens[i, :int(lengths[i])].tolist() == want
    bt, bl, bs = eng.caption_images(fx["images"], eng.gen_params("beam", 10, stop_token=fx["stop_id"], beam_size=5))
    for i, (want, got) in enumerate(zip(fx["beam5"], winners((bt, bl, bs)))):
        assert got == want, (i, got, want)


def test_rejections_leave_the_context_usable(gpt2):
    eng, fx, stop, cands = gpt2
    imgs = images(fx, 6, seed=1)
    beam = lambda t=4, **kw: eng.gen_params("beam", t, **{"beam_size": 5, **kw})
    bad = [
        ("not beam search", eng.gen_params("greedy", 4), {}),
        ("not beam search", eng.gen_params("sample", 4, top_p=0.9), {}),
        ("beam_size", beam(beam_size=0), {}),
        ("beam_size", beam(beam_size=6), {}),         # above max_beam
        ("groups", beam(), {"groups": -1}),
        ("groups", beam(), {"groups": 65}),           # above max_images
        ("max_ctx", beam(29), {}),                    # 4 prefix tokens + 29 > 32
        ("BOS id outside the vocabulary", beam(), {"append_bos": fx["V"]}),
    ]
    for what, p, kw in bad:
        l0 = eng.launch_count
        with pytest.raises(RuntimeError, match=what):
            eng.caption_dataset_continuous_beam(imgs, p, **kw)
        assert eng.launch_count == l0, what
        still_works(eng, fx)
    l0 = eng.launch_count
    with pytest.raises(RuntimeError, match="beam"):
        eng.caption_dataset_continuous(imgs, beam())
    assert eng.launch_count == l0
    p = beam(T, stop_token=stop)
    compare(eng, imgs, eng.caption_dataset(imgs, p), eng.caption_dataset_continuous_beam(imgs, p, groups=4))


def test_rejects_a_beam_merge_above_its_shared_memory():
    """beam 8 over max_ctx = 2100 positions needs 8 * 2100 * 4 bytes > 64 KB in beam_merge_kernel"""
    import clipcap_b200 as cc
    fx = torch.load(os.path.join(GOLDEN, "tiny_gpt2.pt"), weights_only=False)
    cfg = cc.EngineConfig(
        lm_arch="gpt2", lm_d=fx["d"], lm_layers=2, lm_heads=fx["heads"], lm_vocab=fx["V"], lm_n_pos=2100,
        map_dim_clip=fx["dim_clip"], map_clip_len=fx["CL"], map_prefix_len=fx["P"], map_heads=fx["map_heads"],
        map_layers=2, vit_image=fx["vit_image"], vit_patch=fx["vit_patch"], vit_width=fx["vit_width"],
        vit_layers=fx["vit_layers"], vit_heads=fx["vit_heads"], vit_out=fx["dim_clip"], max_images=2, max_beam=8,
        max_ctx=2100, page_tokens=4)
    eng = cc.Engine(cfg)
    try:
        l0 = eng.launch_count
        with pytest.raises(RuntimeError, match="shared memory"):
            eng.caption_dataset_continuous_beam(images(fx, 2), eng.gen_params("beam", 8, beam_size=8), groups=2)
        assert eng.launch_count == l0
    finally:
        eng.close()
