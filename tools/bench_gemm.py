"""Micro-benchmark of the decode-shaped (weight-streaming) GEMM: rotates over enough weight matrices to stay HBM-cold.
usage: python tools/bench_gemm.py [tokens] [features] [K] [split_k] [bn] [orientation]
split_k 0 times the forced single split and the automatic choice; split-K needs the swapped orientation (tokens <= 256)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import clipcap_b200 as cc

tokens = int(sys.argv[1]) if len(sys.argv) > 1 else 64
cases = [(4800, 1600), (1600, 1600), (6400, 1600), (1600, 6400), (50257, 1600)]
if len(sys.argv) > 3:
    cases = [(int(sys.argv[2]), int(sys.argv[3]))]
split = int(sys.argv[4]) if len(sys.argv) > 4 else 0
bn = int(sys.argv[5]) if len(sys.argv) > 5 else 0
orient = int(sys.argv[6]) if len(sys.argv) > 6 else 0
cfg = cc.EngineConfig(lm_d=128, lm_layers=1, lm_heads=2, lm_vocab=503, lm_n_pos=64, map_kind="none", vit=False, max_images=8, max_ctx=32)
eng = cc.Engine(cfg)
for features, K in cases:
    n = max(2, int(600e6 // (features * K * 2)))
    W = (torch.randn(n, features, K, device="cuda") * 0.02).bfloat16()
    x = torch.randn(tokens, K, device="cuda").bfloat16()
    bias = torch.zeros(features, device="cuda")
    for s in ([split] if split else [1, 0]):
        for _ in range(2):
            for i in range(n):
                eng.op_linear(x, W[i], bias, "none", None, torch.bfloat16, orient, bn, s)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        e0.record()
        for _ in range(reps):
            for i in range(n):
                eng.op_linear(x, W[i], bias, "none", None, torch.bfloat16, orient, bn, s)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / (reps * n)
        print("tokens %d features %d K %d split %s: %.2f us  %.0f GB/s (weights only)  %.0f TFLOP/s" % (tokens, features, K, s or "auto", us, features * K * 2 / us / 1e3, 2.0 * tokens * features * K / us / 1e6))
    del W
