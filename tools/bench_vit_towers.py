"""The OpenAI CLIP image towers on one B200: vit_encode at batch 64 for ViT-B/32, ViT-B/16, ViT-L/14 and ViT-L/14@336px
(synthetic weights), the attention kernel alone at the long-sequence shapes (beside torch's scaled_dot_product_attention in
bf16, as a comparator only), and captions/s from pixels for ViT-L/14@336px + the all-features mapper + GPT2-XL.

    python tools/bench_vit_towers.py [out.json]          (default: profiles/r3_vit_towers.json)

Timings are CUDA events around a window of >= 1 s of back-to-back calls, after a warm-up, repeated; the median and the
spread of the repeats are reported.  FLOPs are computed from the shapes (2 per multiply-add): per ViT layer 24 S w^2 of
GEMMs (qkv, out_proj, fc1, fc2) and 4 S^2 w of attention (Q K^T and P V).  The card's name, power limit and maximum SM
clock are read with nvidia-smi (a query, nothing is set) in the same run.
"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import clipcap_b200 as cc  # noqa: E402
from clipcap_b200 import synthetic  # noqa: E402

B = 64
REPEATS = 5
WINDOW_S = 1.0


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn):
    """(median ms per call, [ms per call of each repeat]) over windows of >= WINDOW_S."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    n = max(3, int(WINDOW_S * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    reps = []
    for _ in range(REPEATS):
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        reps.append(e0.elapsed_time(e1) / n)
    return statistics.median(reps), reps


def vit_flops(cfg):
    g = cfg.vit_image // cfg.vit_patch
    S, w, L = g * g + 1, cfg.vit_width, cfg.vit_layers
    gemm = 2 * g * g * 3 * cfg.vit_patch ** 2 * w + L * 24 * S * w * w + 2 * w * cfg.vit_out
    attn = L * 4 * S * S * w
    return S, gemm, attn


def bench_towers():
    rows = []
    for name in ("ViT-B/32", "ViT-B/16", "ViT-L/14", "ViT-L/14@336px"):
        cfg = cc.EngineConfig.for_clip(name, lm_d=128, lm_layers=1, lm_heads=2, lm_vocab=503, lm_n_pos=64, map_kind="none",
                                       max_images=B, max_ctx=32)
        eng = cc.Engine(cfg)
        eng.load_state_dict(synthetic.lm_state_dict(cfg, 1234, "cuda"), prefix="language_model.")
        eng.load_state_dict(synthetic.vit_state_dict(cfg, 1236, "cuda"), prefix="visual.")
        eng.check_weights()
        images = synthetic.synthetic_images(B, cfg, device="cuda")
        ms, reps = timed(lambda: eng.vit_encode(images))
        S, gemm, attn = vit_flops(cfg)
        rows.append({"tower": name, "tokens": S, "batch": B, "ms_per_batch": ms, "ms_repeats": reps, "images_per_s": B / ms * 1e3,
                     "gemm_gflop_per_image": gemm / 1e9, "attention_gflop_per_image": attn / 1e9,
                     "achieved_tflops": B * (gemm + attn) / (ms * 1e-3) / 1e12})
        print(json.dumps(rows[-1]), flush=True)
        eng.close()
        del eng
        torch.cuda.empty_cache()
    return rows


def sdpa_backend(q, k, v):
    """Names of the CUDA kernels one default scaled_dot_product_attention call launches."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        torch.nn.functional.scaled_dot_product_attention(q, k, v)
        torch.cuda.synchronize()
    return sorted({e.key for e in prof.key_averages() if e.device_type.name == "CUDA"})


def bench_attention():
    eng_cfg = cc.EngineConfig(lm_d=128, lm_layers=1, lm_heads=2, lm_vocab=503, lm_n_pos=64, map_kind="none", vit=False,
                              max_images=8, max_ctx=32)
    eng = cc.Engine(eng_cfg)
    rows = []
    shapes = [("ViT-L/14@336px", 64, 577, 16, 64), ("ViT-L/14", 64, 257, 16, 64),
              ("GPT2-XL all-features mapper (ViT-L/14@336px)", 64, 617, 8, 200),
              ("GPT-2 small all-features mapper (ViT-L/14@336px)", 64, 587, 8, 96)]
    for what, b, S, H, hd in shapes:
        g = torch.Generator(device="cuda").manual_seed(S)
        qkv = torch.randn(b * S, 3 * H * hd, generator=g, device="cuda").bfloat16()
        flop = 4 * b * H * S * S * hd
        ms, reps = timed(lambda: eng.op_attention(qkv, b, S, H, hd))
        q, k, v = qkv.view(b, S, 3, H, hd).permute(2, 0, 3, 1, 4).unbind(0)   # [b, H, S, hd] views of the same buffer
        ms_t, reps_t = timed(lambda: torch.nn.functional.scaled_dot_product_attention(q, k, v))
        rows.append({"shape": what, "B": b, "S": S, "H": H, "hd": hd, "qkv_mbytes": qkv.numel() * 2 / 1e6,
                     "us": ms * 1e3, "us_repeats": [x * 1e3 for x in reps], "tflops": flop / (ms * 1e-3) / 1e12,
                     "torch_sdpa_us": ms_t * 1e3, "torch_sdpa_tflops": flop / (ms_t * 1e-3) / 1e12,
                     "torch_sdpa_kernels": sdpa_backend(q, k, v)})
        print(json.dumps(rows[-1]), flush=True)
    eng.close()
    return rows


def bench_end_to_end():
    cfg = cc.EngineConfig.for_clip("ViT-L/14@336px", map_kind="transformer_all", max_images=B, max_beam=1, max_ctx=80)
    eng = cc.Engine(cfg)
    synthetic.load_synthetic(eng)
    torch.cuda.empty_cache()
    images = synthetic.synthetic_images(B, cfg, device="cuda")
    p = eng.gen_params("greedy", 32, stop_token=-1, max_stops=0)
    ms, reps = timed(lambda: eng.caption_images(images, p))
    row = {"pipeline": "ViT-L/14@336px (577 tokens) + all-features mapper (8 layers, S = 617, head_dim 200) + GPT2-XL",
           "images": B, "mode": "greedy", "new_tokens": 32, "ms_per_call": ms, "ms_repeats": reps, "captions_per_s": B / ms * 1e3}
    print(json.dumps(row), flush=True)
    eng.close()
    return row


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_vit_towers.json")
    if not torch.cuda.is_available():
        raise SystemExit("bench_vit_towers.py measures on a CUDA device; none is visible")
    res = {"gpu": gpu_info(), "vit_encode": bench_towers(), "attention": bench_attention(), "end_to_end": bench_end_to_end()}
    l336 = next(r for r in res["vit_encode"] if r["tower"] == "ViT-L/14@336px")
    a336 = res["attention"][0]
    res["attention_share_of_l14_336_vit_encode"] = 24 * a336["us"] * 1e-3 / l336["ms_per_batch"]
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "attention_share_of_l14_336_vit_encode")}))


if __name__ == "__main__":
    main()
