"""Dataset captioning with and without continuous batching, timed in one process:

    python tools/bench_continuous.py [--mode sample|beam] [--beam 5] [--images 2048] [--new-tokens 67] [--repeats 3]
                                     [--out FILE]

Workload: BASELINE.json config 2's model (ViT-B/32, Transformer mapper with prefix 40, GPT2-XL, random init, 64 images
per micro-batch / 64 decode slots), sampling at temperature 1, T = 67 new tokens (the reference's entry_length).
Random-init weights never stop a caption, so the captions get a length distribution: a constant direction u is added
to ln_f's bias and a multiple of u to the EOS row of wte (tied to lm_head), which raises the EOS logit by about the same
amount at every position.  The multiple is calibrated on the first decision point (the logits after the prefix) so that
EOS is drawn with probability about 1/15 per step; the probability reached there and the mean caption length are
reported.

Engine.caption_dataset and Engine.caption_dataset_continuous run alternately on the same images after one warm-up
call each, every call ending in a device synchronisation.  Reported: captions/s of each (mean and spread over the
repeats), decode steps, the share of images whose captions are identical, and the card's name and power limit read in
the same run.

--mode beam: the same model with max_beam 5 (BASELINE.json config 4's beam), beam search against
Engine.caption_dataset_continuous_beam; caption_dataset runs micro-batches of 256 // beam images (51 for beam 5) and the
new path as many groups.  The stop token (13, the reference's) gets the same kind of bias as EOS above.  Beam search
magnifies it: on a flat random-init distribution a raised token becomes every beam's best extension, so the multiple is
calibrated by bisection on caption_dataset itself over 102 images, towards a mean winning-beam length of 18 (the
sampling run's mean caption length).  Reported besides the above: the mean winner length and the mean group length (an
image's longest beam, the decode steps its group needs)."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

EOS = 50256
TARGET_P = 1.0 / 15


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as e:   # the timing stands without it, but say so
        return torch.cuda.get_device_name(0), "unread (%s)" % type(e).__name__


def first_step_logits(eng, imgs, chunk=64):
    out = []
    for i in range(0, imgs.shape[0], chunk):
        out.append(eng.lm_forward(eng.map_prefix(eng.vit_encode(imgs[i:i + chunk])), last_only=True).double())
    return torch.cat(out)


def eos_p(logits):
    return float(torch.softmax(logits, -1)[:, EOS].mean())


def calibrate(eng, lm_sd, imgs):
    """ln_f.bias += alpha * u, wte[EOS] += beta * u, beta from the first-step logits; returns (beta, P(EOS) reached)"""
    d = eng.cfg.lm_d
    g = torch.Generator(device="cpu").manual_seed(77)
    u = torch.randn(d, generator=g)
    u = (u / u.norm()).to(eng.device)
    alpha = 10.0
    base = first_step_logits(eng, imgs)
    lo, hi = 0.0, 100.0         # the EOS logit shift that gives TARGET_P on the unmodified logits
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        shifted = base.clone()
        shifted[:, EOS] += mid
        lo, hi = (mid, hi) if eos_p(shifted) < TARGET_P else (lo, mid)
    beta = lo / alpha
    wte = lm_sd["transformer.wte.weight"].clone()
    wte[EOS] += beta * u
    eng.load_state_dict({"transformer.ln_f.bias": lm_sd["transformer.ln_f.bias"] + alpha * u, "transformer.wte.weight": wte},
                        prefix="language_model.")
    return beta, eos_p(first_step_logits(eng, imgs))


def sync_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def stats(n, ts):
    r = [n / t for t in ts]
    return {"captions_per_s_mean": sum(r) / len(r), "captions_per_s_min": min(r), "captions_per_s_max": max(r),
            "seconds": ts}


def emit(res, out):
    line = json.dumps(res)
    print(line)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(line + "\n")


STOP = 13
TARGET_WINNER_LEN = 18.0


def winners(res):
    tok, ln, sc = res[0].cpu(), res[1].cpu(), res[2].cpu()
    k = sc.argmax(1)
    idx = torch.arange(tok.shape[0])
    return tok[idx, k], ln[idx, k]


def main_beam(args):
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic

    T, beam = args.new_tokens, args.beam
    cfg = cc.EngineConfig(max_images=64, max_beam=beam, max_ctx=40 + T + 1)
    eng = cc.Engine(cfg)
    sds = synthetic.load_synthetic(eng, 1234)
    imgs = synthetic.synthetic_images(args.images, cfg, seed=0, device=eng.device)
    p = eng.gen_params("beam", T, stop_token=STOP, beam_size=beam)
    groups = eng.micro_batch_for(p)

    # ln_f.bias += alpha * u, wte[STOP] += beta * u: the stop logit rises by about alpha * beta at every position
    lm_sd = sds["lm"]
    g = torch.Generator(device="cpu").manual_seed(77)
    u = torch.randn(cfg.lm_d, generator=g)
    u = (u / u.norm()).to(eng.device)
    alpha = 10.0
    eng.load_state_dict({"transformer.ln_f.bias": lm_sd["transformer.ln_f.bias"] + alpha * u}, prefix="language_model.")
    wte = lm_sd["transformer.wte.weight"].clone()
    row = wte[STOP].clone()
    calib = imgs[:2 * groups]

    def winner_len(beta):
        wte[STOP] = row + beta * u
        eng.load_state_dict({"transformer.wte.weight": wte}, prefix="language_model.")
        return float(winners(eng.caption_dataset(calib, p))[1].float().mean())

    lo, hi = 0.0, 3.0            # winner length falls as beta grows
    for _ in range(12):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if winner_len(mid) > TARGET_WINNER_LEN else (lo, mid)
    beta = 0.5 * (lo + hi)
    calib_len = winner_len(beta)

    batched = lambda: eng.caption_dataset(imgs, p)
    continuous = lambda: eng.caption_dataset_continuous_beam(imgs, p, groups=groups)
    _, ref = sync_time(batched)
    _, got = sync_time(continuous)
    t_b, t_c = [], []
    for _ in range(args.repeats):
        t, ref = sync_time(batched)
        t_b.append(t)
        t, got = sync_time(continuous)
        t_c.append(t)
    n = args.images
    (rw, rwl), (gw, gwl) = winners(ref), winners(got)
    same_winner = sum(int(rwl[i]) == int(gwl[i]) and torch.equal(rw[i, :int(rwl[i])], gw[i, :int(gwl[i])]) for i in range(n))
    same_all = sum(torch.equal(ref[0][i], got[0][i]) and torch.equal(ref[1][i], got[1][i]) for i in range(n))

    def mean_logprob(i, cap):
        """teacher-forced mean log-probability of a caption: the quantity beam search ranks by"""
        emb = eng.map_prefix(eng.vit_encode(imgs[i:i + 1]))
        S0, L = emb.shape[1], len(cap)
        if L > 1:
            emb = torch.cat([emb, eng.embed_tokens(cap[None, :-1])], 1)
        lp = torch.log_softmax(eng.lm_forward(emb)[0, S0 - 1:S0 - 1 + L].double(), -1)
        return float(lp.gather(-1, cap[:, None].long().to(lp.device)).mean())

    gaps = []     # |score gap| / |score| of the two winners where they differ
    for i in range(n):
        a, b = rw[i, :int(rwl[i])], gw[i, :int(gwl[i])]
        if not torch.equal(a, b):
            s_a = mean_logprob(i, a)
            gaps.append(abs(s_a - mean_logprob(i, b)) / abs(s_a))
    name, power = card()
    res = {
        "card": name, "power_limit": power, "images": n, "new_tokens": T, "beam": beam, "groups": groups,
        "workload": "config 2/4 model (ViT-B/32, mapper prefix 40, GPT2-XL, random init), beam %d, stop token %d biased"
                    % (beam, STOP),
        "stop_shift_beta": beta, "calibration_images": calib.shape[0], "calibration_mean_winner_length": calib_len,
        "mean_winner_length_batched": float(rwl.float().mean()), "mean_winner_length_continuous": float(gwl.float().mean()),
        "mean_group_length_batched": float(ref[1].max(1).values.float().mean()),
        "mean_group_length_continuous": float(got[1].max(1).values.float().mean()),
        "identical_winners": same_winner / n, "identical_all_beams": same_all / n,
        "differing_winners_within_2e-2": sum(g <= 2e-2 for g in gaps) / max(len(gaps), 1),
        "differing_winners_max_relative_gap": max(gaps, default=0.0),
        "decode_steps_batched": (n + groups - 1) // groups * (T - 1), "decode_steps_continuous": got[3],
        "caption_dataset": stats(n, t_b), "caption_dataset_continuous_beam": stats(n, t_c),
        "library": os.environ.get("CCB_LIB", "default"),
    }
    res["speedup_mean"] = (res["caption_dataset_continuous_beam"]["captions_per_s_mean"]
                           / res["caption_dataset"]["captions_per_s_mean"])
    emit(res, args.out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["sample", "beam"], default="sample")
    ap.add_argument("--beam", type=int, default=5)
    ap.add_argument("--images", type=int, default=2048)
    ap.add_argument("--new-tokens", type=int, default=67)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_continuous.py needs a CUDA device (B200)")
    if args.mode == "beam":
        return main_beam(args)
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic

    T = args.new_tokens
    cfg = cc.EngineConfig(max_images=64, max_ctx=40 + T + 1)
    eng = cc.Engine(cfg)
    sds = synthetic.load_synthetic(eng, 1234)
    imgs = synthetic.synthetic_images(args.images, cfg, seed=0, device=eng.device)
    beta, p_first = calibrate(eng, sds["lm"], imgs[:256])
    p = eng.gen_params("sample", T, stop_token=-1, eos_token=EOS, temperature=1.0, seed=5)

    batched = lambda: eng.caption_dataset(imgs, p)
    continuous = lambda: eng.caption_dataset_continuous(imgs, p)
    _, ref = sync_time(batched)
    _, got = sync_time(continuous)
    t_b, t_c = [], []
    for _ in range(args.repeats):
        t, ref = sync_time(batched)
        t_b.append(t)
        t, got = sync_time(continuous)
        t_c.append(t)
    n = args.images
    rt, rl, gt, gl = ref[0].cpu(), ref[1].cpu(), got[0].cpu(), got[1].cpu()
    same = sum(int(rl[i]) == int(gl[i]) and torch.equal(rt[i, :int(rl[i])], gt[i, :int(gl[i])]) for i in range(n))
    name, power = card()
    res = {
        "card": name, "power_limit": power, "images": n, "new_tokens": T, "slots": 64,
        "workload": "config 2 model (ViT-B/32, mapper prefix 40, GPT2-XL, random init), sampling T=1, EOS-biased",
        "p_eos_first_step": p_first, "eos_shift_beta": beta,
        "mean_length_batched": float(rl.float().mean()), "mean_length_continuous": float(gl.float().mean()),
        "identical_captions": same / n,
        "decode_steps_batched": (n + 63) // 64 * (T - 1), "decode_steps_continuous": got[2],
        "caption_dataset": stats(n, t_b), "caption_dataset_continuous": stats(n, t_c),
        "library": os.environ.get("CCB_LIB", "default"),
    }
    res["speedup_mean"] = res["caption_dataset_continuous"]["captions_per_s_mean"] / res["caption_dataset"]["captions_per_s_mean"]
    emit(res, args.out)


if __name__ == "__main__":
    main()
