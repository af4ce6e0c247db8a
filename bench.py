"""Benchmark of the caption-generation hot path on BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4|5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1], the configuration the metric is quoted on): ViT-B/32 + 8-layer Transformer
mapper (prefix 40, clip_length 40) + GPT2-XL, greedy decoding of exactly 32 new tokens (stop token disabled so
every caption costs the same), batch 64 per GPU, seeded random-init bf16 weights, synthetic 224x224 images.
A "step" = one batch of 64 images -> 64 captions.  With N GPUs every rank captions its own 64 images with
replicated weights (weak scaling); the only collective is the final all-gather of the caption tokens.

  value     captions/s, images already resident in HBM, timed with CUDA events (max over ranks)
  e2e       the same through the public Python API with HOST buffers: pinned fp32 images -> H2D -> ViT -> mapper ->
            decode -> D2H of tokens + lengths, copies inside the timed region
  roofline  the decode step (one CUDA-graph replay = all kernels of one token for the whole batch): algorithmic
            HBM bytes (bf16 weights once + KV read/write, DESIGN.md) / its mean duration (events recorded by the
            library on its launching stream inside the timed region) against the measured HBM peak
  cpu_baseline / --impl reference: the reference's own algorithm (batch-1 loop, full re-forward every token, fp32;
            inference.py:70-148 with beam_size=1) on the host cores -- the reference's own modules (kind "reference": imported
            unmodified from /root/reference, or from oracle/_ref, the bytecode build() compiles from it, where that tree is
            absent), else the restatement in oracle/clipcap_oracle.py (kind "port").

The default line (N = 1, config 2) also carries `other_configs`: short child runs (3 timed steps each) of BASELINE.json's
configs 3 / 4 / 5 on the same GPU -- context, never part of `value` (--no-other-configs skips them).

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0's share) as DIR/<name>.npy in float32:
tokens, lengths and, for beam search, scores (token ids and lengths are exact in float32).  Weights, images and sampling
seeds are fixed, so two builds run with the same arguments can be compared output for output.

--config selects another BASELINE.json configuration (the default, 2, is the one the metric is quoted on and the only one
the CPU arm covers): 3 = nucleus sampling (top_p 0.9, temperature 1.0), batch 256; 4 = beam 5, 102 images per step (two
micro-batches of 51 = 255 rows, Engine.caption_dataset); 5 = GPT-J-6B + 4096-wide mapper, top_p 0.9, 16 images per GPU (128 on 8).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

_OUT = sys.stdout   # main() points it at the original stdout and redirects fd 1 to stderr

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree bench.py runs from may be read-only: nothing is written there
DUMP_LIMIT = 64 << 20            # bytes, all --dump-outputs arrays together

METRIC = "captions/sec (GPT2-XL, prefix 40, 32 tok)"
UNIT = "captions/s"
BATCH = 64
NEW_TOKENS = 32
WORKLOAD = "ViT-B/32 + 8-layer Transformer mapper (P=40, clip_len=40) + GPT2-XL, greedy, batch 64, 32 new tokens"
# BASELINE.json configs[1..4] (1-based ids 2..5); `batch` is per GPU
CONFIGS = {
    2: dict(metric=METRIC, workload=WORKLOAD, batch=64, mode="greedy", beam=1, kw={}, lm={}),
    3: dict(metric=METRIC, workload="config 2's model, nucleus sampling (top_p 0.9, temperature 1.0), batch 256, 32 new tokens",
            batch=256, mode="sample", beam=1, kw=dict(top_p=0.9, temperature=1.0, seed=1), lm={}),
    4: dict(metric=METRIC, workload="config 2's model, beam search (beam 5), 102 images per step in micro-batches of 51 (255 rows each: "
                                    "the persistent decode kernel's limit), 32 new tokens -- a GPU's share of the 16 k-image set is a stream of those",
            batch=102, mode="beam", beam=5, kw=dict(beam_size=5), lm={}),
    5: dict(metric="captions/sec (GPT-J-6B, prefix 40, 32 tok)",
            workload="ViT-B/32 + 8-layer Transformer mapper (d=4096) + GPT-J-6B, nucleus sampling (top_p 0.9), batch 16 per GPU "
                     "(128 on 8 GPUs), 32 new tokens",
            batch=16, mode="sample", beam=1, kw=dict(top_p=0.9, temperature=1.0, seed=1),
            lm=dict(lm_arch="gptj", lm_d=4096, lm_layers=28, lm_heads=16, lm_vocab=50400, lm_n_pos=2048, lm_rotary_dim=64)),
}


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """DRAM bytes of the dominant kernel of the decode step (the persistent layer-stack kernel), from the committed ncu
    --set full capture (profiles/r2_decode_mega_ncu.json: dram__bytes_read.sum + dram__bytes_write.sum of one launch)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_decode_mega_ncu.json")) as f:
            j = json.load(f)
        k = j["launches"][0] if "launches" in j else j
        return float(k["dram__bytes_read.sum"]) + float(k["dram__bytes_write.sum"])
    except Exception:
        return None


def decode_step_bytes(cfg, batch, prefix_len, step):
    """Algorithmic HBM bytes of decode step `step` (1-based; the token fed sits at position prefix_len + step - 1):
    every bf16 weight once + K/V of the cached context read + K/V of the new token written (SURVEY 8d)."""
    d, L, V = cfg.lm_d, cfg.lm_layers, cfg.lm_vocab
    weights = 2 * (L * (12 * d * d + 13 * d) + 2 * d + V * d)
    if cfg.lm_arch == "gptj":      # one LayerNorm per block, q/k/v/out without bias, untied biased head
        weights = 2 * (L * (12 * d * d + 7 * d) + 2 * d + V * d + V * d + V)
    kv_tok = 2 * L * d * 2
    ctx = prefix_len + step - 1
    return weights + batch * ctx * kv_tok + batch * kv_tok


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def build_oracle(threads):
    """Builds the fp32 GPT2-XL + mapper + ViT oracle once; returns run(tokens) -> seconds for one bounded sample."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import clipcap_oracle as orc
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic
    torch.set_num_threads(threads)
    cfg = cc.EngineConfig(max_images=1)
    lm_sd = synthetic.lm_state_dict(cfg, 1234, "cpu")
    map_sd = synthetic.mapper_state_dict(cfg, 1235, "cpu")
    vit_sd = synthetic.vit_state_dict(cfg, 1236, "cpu")
    lm = orc.OracleLM(lm_sd, "gpt2", cfg.lm_heads)
    image = synthetic.synthetic_images(1, cfg, 0, "cpu")

    def run(tokens_per_sample):
        with torch.no_grad():
            t0 = time.perf_counter()
            feat = orc.vit_forward(vit_sd, image, cfg.vit_heads, cfg.vit_patch)
            prefix = orc.mapper_forward(map_sd, feat, cfg.map_clip_len, cfg.map_heads)
            # the reference loop: full re-forward of prefix + generated tokens for every new token, batch 1
            orc.generate_beam(lm, prefix, beam_size=1, entry_length=tokens_per_sample, stop_token=-1, use_cache=False)
            return time.perf_counter() - t0
    return run


def build_reference_arm(threads):
    """The reference's OWN generation loop on the host cores: lms/GPT2.py's GPT2 (an HF GPT2LMHeadModel subclass) at GPT2-XL
    size, model.py's CLIPCaptionModel.clip_project (TransformerMapper) and inference.py:70-148 `generate_beam` with
    beam_size=1 -- the greedy, no-KV-cache, batch-1 loop config 2 is quoted on -- imported UNMODIFIED through
    oracle/ref_harness.py (from /root/reference in the build container, from the byte-compiled oracle/_ref on the GPU box), on the
    same synthetic weights as the GPU arm.  The image tower alone comes from the oracle (the reference takes it from the `clip`
    package, which is not installed; it is ~1 % of the sample's time).  Returns run(tokens) -> seconds, or None when the reference
    cannot be imported here (then the oracle's restatement is timed: kind "port")."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import ref_harness
        if not ref_harness.available():
            return None
        ref = ref_harness.load_reference()
        import clipcap_oracle as orc
        import clipcap_b200 as cc
        from clipcap_b200 import synthetic
        from transformers import GPT2Config
        torch.set_num_threads(threads)
        cfg = cc.EngineConfig(max_images=1)
        lm = ref.lms.GPT2(GPT2Config(vocab_size=cfg.lm_vocab, n_positions=cfg.lm_n_pos, n_embd=cfg.lm_d, n_layer=cfg.lm_layers,
                                     n_head=cfg.lm_heads, layer_norm_epsilon=cfg.lm_ln_eps))
        missing, unexpected = lm.load_state_dict(synthetic.lm_state_dict(cfg, 1234, "cpu"), strict=False)
        assert not unexpected and all(k == "lm_head.weight" or k.endswith(".attn.bias") or k.endswith(".masked_bias") for k in missing), (missing, unexpected)
        lm.tie_weights()
        lm.eval()

        class _Tok:                       # ids in, ids out; a stop id that never occurs: every caption runs its full length
            bos_token_id = None
            all_special_ids = []

            def encode_text(self, text, *a, **k):
                return [-1]

            def decode_tokens(self, tokens):
                return [int(t) for t in tokens]

        model = ref.model.CLIPCaptionModel(
            language_model=lm, tokenizer=_Tok(), visual_encoder=torch.nn.Identity(), validator=None, train_visual_encoder=False,
            use_all_vit_features=False, prefix_size=cfg.map_dim_clip, prefix_length=cfg.map_prefix_len,
            clip_prefix_length=cfg.map_clip_len, num_attention_heads=cfg.map_heads, num_layers=cfg.map_layers,
            mlp_ratio=cfg.map_mlp_ratio, prefix_init_std=1.0, act_fn_name=cfg.map_act, pos_embeddings=False)
        model.clip_project.load_state_dict(synthetic.mapper_state_dict(cfg, 1235, "cpu"))
        model.eval()
        vit_sd = synthetic.vit_state_dict(cfg, 1236, "cpu")
        image = synthetic.synthetic_images(1, cfg, 0, "cpu")
        tok = model.tokenizer

        def run(tokens_per_sample):
            with torch.no_grad():
                t0 = time.perf_counter()
                feat = orc.vit_forward(vit_sd, image, cfg.vit_heads, cfg.vit_patch)
                prefix = model.clip_project(feat.float())                                   # inference.py:312
                out = ref.inference.generate_beam(model, tok, prefix, beam_size=1, entry_length=tokens_per_sample)
                assert len(out[0]) == tokens_per_sample
                return time.perf_counter() - t0
        run.kind = "reference"
        run.what = ("the reference's own loop (inference.py generate_beam, beam_size=1: greedy, no KV cache, batch 1; lms/GPT2.py, "
                    "model.py mapper; imported unmodified from %s), fp32"
                    % ("/root/reference" if ref_harness.kind() == "source" else "oracle/_ref, its byte-compiled modules"))
        return run
    except Exception as e:   # noqa: BLE001 -- a baseline arm must not fail the bench: fall back to the restatement, and say so
        sys.stderr.write("bench.py: reference arm unavailable (%s: %s); timing the oracle port\n" % (type(e).__name__, str(e)[:300]))
        return None


def build_cpu_arm(threads):
    """The reference's own loop where it imports and runs (one warm token first), else the oracle's restatement of it."""
    run = build_reference_arm(threads)
    if run is not None:
        try:
            run(1)                            # warms the allocator / thread pool; a reference that cannot run here falls back
        except Exception as e:   # noqa: BLE001
            sys.stderr.write("bench.py: reference arm failed its warm run (%s: %s); timing the oracle port\n" % (type(e).__name__, str(e)[:300]))
            run = None
    if run is None:
        run = build_oracle(threads)
        run.kind = "port"
        run.what = "reference no-KV-cache batch-1 loop restated by the oracle (oracle/clipcap_oracle.py), fp32"
        run(1)
    return run


def sample_scale(tokens_per_sample, prefix_len=40, full=NEW_TOKENS):
    """The reference re-forwards prefix + t tokens for token t: cost ~ sum(prefix + t).  Scale of a sample of the
    first `tokens_per_sample` tokens up to a full caption of `full` tokens."""
    c = lambda n: sum(prefix_len + t for t in range(n))
    return c(full) / c(tokens_per_sample)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    # bounded sample: one image, the first `tok` tokens of its caption; sized so W + K steps end in a few minutes
    budget_s = 150.0
    run = build_cpu_arm(threads)          # (has run one warm token)
    per_full = run(2) * sample_scale(2)
    tok = NEW_TOKENS
    while tok > 2 and (args.steps + args.warmup) * per_full / sample_scale(tok) > budget_s:
        tok //= 2
    for _ in range(args.warmup):
        run(tok)
    times = [run(tok) for _ in range(args.steps)]
    ms = sum(times) / len(times) * 1e3
    scale = sample_scale(tok)
    value = 1.0 / (ms * 1e-3 * scale)
    sample = ("1 image per step, first %d of %d tokens with %s; "
              "captions/s = 1 / (step time x %.2f), the cost ratio sum(40+t) of a full caption to the sample" % (tok, NEW_TOKENS, run.what, scale))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD, "device": "host CPU"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": run.kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), file=_OUT, flush=True)


def cpu_baseline_leg():
    """Reported baseline at N=1: ~10-30 s of the oracle on the host cores."""
    threads = os.cpu_count() or 1
    run = build_cpu_arm(threads)
    t2 = run(2)
    tok = NEW_TOKENS
    while tok > 2 and t2 * sample_scale(2) / sample_scale(tok) > 25.0:
        tok //= 2
    t = run(tok)
    scale = sample_scale(tok)
    return {"value": 1.0 / (t * scale), "unit": UNIT, "cores": threads, "kind": run.kind,
            "sample": "1 image, first %d of %d tokens, %s, "
                      "scaled x%.2f by sum(40+t) to a full caption" % (tok, NEW_TOKENS, run.what, scale)}


def other_configs_leg():
    """BASELINE.json's configs 3 / 4 / 5 on this GPU, each a short child run of this script (3 timed steps), so that the
    driver's default invocation also carries their numbers.  Context for the headline line, never part of its `value`; a
    child that fails or overruns its time limit is reported as such and does not affect the line."""
    out = {}
    for cfg_id, limit in ((3, 150), (4, 150), (5, 240)):
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--config", str(cfg_id), "--steps", "3", "--warmup", "3",
                                "--no-cpu-baseline"], capture_output=True, text=True, timeout=limit,
                               env=dict({k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")},
                                        PYTHONDONTWRITEBYTECODE="1"))
            j = json.loads(r.stdout.strip().splitlines()[-1])
            out["config%d" % cfg_id] = {
                "metric": j["metric"], "workload": j["config"]["workload"], "value": j["value"], "unit": j["unit"],
                "e2e": j["e2e"]["value"], "ms_per_step": j["ms_per_step"], "steps": j["steps"],
                "decode_step_ms": j["roofline"]["ms_per_launch"], "decode_step_gbs": j["roofline"]["achieved"],
                "roofline_frac": j["roofline"]["frac"], "gpu_launches": j["gpu_launches"]}
        except Exception as e:   # noqa: BLE001 -- context only
            out["config%d" % cfg_id] = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}
    return out


def dump_outputs(out_dir, arrays):
    """Writes every tensor of `arrays` (name -> tensor, None skipped) as out_dir/<name>.npy in float32."""
    import numpy as np
    host = {k: v.detach().cpu().float().numpy() for k, v in arrays.items() if v is not None}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the short runs of BASELINE.json's configs 3 / 4 / 5 that the default N=1 line reports under `other_configs`")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0: tokens, lengths, beam scores) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    C_ = CONFIGS[args.config]
    BATCH = C_["batch"]
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    # stdout carries the JSON line and nothing else: whatever libraries print meanwhile (the "NCCL version ..." banner
    # of a box with NCCL_DEBUG set, ...) is sent to stderr
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
        return

    import torch.distributed as dist
    import clipcap_b200 as cc
    from clipcap_b200 import synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    cfg = cc.EngineConfig(max_images=BATCH, max_beam=C_["beam"], max_ctx=40 + NEW_TOKENS + 8, **C_["lm"])
    eng = cc.Engine(cfg, local)
    synthetic.load_synthetic(eng, 1234)          # same seed on every rank: replicated weights
    torch.cuda.empty_cache()
    # every rank captions its own contiguous range of image ids
    images = synthetic.synthetic_images(BATCH, cfg, seed=rank, device=dev)
    host_images = images.cpu().pin_memory()
    params = eng.gen_params(C_["mode"], NEW_TOKENS, stop_token=-1, max_stops=0, **C_["kw"])
    tok_shape = (BATCH, C_["beam"], NEW_TOKENS) if C_["mode"] == "beam" else (BATCH, NEW_TOKENS)
    gathered = [torch.empty(tok_shape, dtype=torch.int32, device=dev) for _ in range(world)] if world > 1 else None

    def caption(imgs):
        if args.config == 2:
            return eng.caption_images(imgs, params)
        # micro-batches where one call does not cover the step (beam 5 x 64 images), Philox streams keyed by global image id
        return eng.caption_dataset(imgs, params, first_row_id=rank * BATCH)

    def step_resident():
        tokens, lengths, scores = caption(images)
        if world > 1:
            dist.all_gather(gathered, tokens)      # the only collective: final captions
        return tokens, lengths, scores

    def step_e2e():
        dev_images = host_images.to(dev, non_blocking=True)
        tokens, lengths, _ = caption(dev_images)
        if world > 1:
            dist.all_gather(gathered, tokens)
        return tokens.cpu(), lengths.cpu()

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count
    profiled = os.environ.get("CCB_BENCH_PROFILE") == "1"   # `ncu --profile-from-start off`: the launch list of the timed region
    if profiled:
        torch.cuda.profiler.start()
    ms_total, (tokens, lengths, scores) = timed(step_resident, args.steps)
    if profiled:
        torch.cuda.profiler.stop()
    launches = eng.launch_count - l0
    calls_per_step = -(-BATCH // eng.micro_batch_for(params)) if args.config != 2 else 1
    n_sum = min(args.steps * calls_per_step, 64)
    prefill_ms, decode_ms, decode_steps = eng.timing_sum(n_sum)
    n_sum = n_sum / calls_per_step        # timed steps the sums cover
    for _ in range(2):
        step_e2e()
    e2e_ms_total, _ = timed(step_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"tokens": tokens, "lengths": lengths, "scores": scores})

    ms_per_step = ms_total / args.steps
    value = world * BATCH / (ms_per_step * 1e-3)
    e2e_value = world * BATCH / (e2e_ms_total / args.steps * 1e-3)
    peak, peak_src = measured_hbm_peak()
    rows_per_launch = min(BATCH, eng.micro_batch_for(params)) * C_["beam"] if args.config != 2 else BATCH
    step_bytes = sum(decode_step_bytes(cfg, rows_per_launch, cfg.map_prefix_len, t) for t in range(1, NEW_TOKENS)) / (NEW_TOKENS - 1)
    step_ms = decode_ms / max(decode_steps, 1)
    achieved = step_bytes / (step_ms * 1e-3) / 1e9

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline and args.config == 2:
            cpu = cpu_baseline_leg()
        other = None
        if world == 1 and args.config == 2 and not args.no_other_configs and not profiled:
            # free this process's engine first: the GPT-J-6B run needs its own 12 GB of weights
            eng.close()
            torch.cuda.empty_cache()
            other = other_configs_leg()
        line = {
            "metric": C_["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": C_["workload"], "baseline_config": args.config, "batch_per_gpu": BATCH, "global_batch": BATCH * world,
                       "new_tokens": NEW_TOKENS, "parallelism": "dp%d (replicated weights, sharded images)" % world,
                       "l2": "not flushed: every decode step streams %.1f GB of weights + KV >> 126 MB L2"
                             % (decode_step_bytes(cfg, 0, 0, 1) / 1e9),
                       "prefill_ms_per_step": prefill_ms / n_sum, "decode_ms_per_step": decode_ms / n_sum},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": host_images.numel() * host_images.element_size(),
                    "d2h_bytes_per_step": tokens.numel() * 4 + lengths.numel() * 4},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": measured_traffic() if args.config == 2 else None,
                         "kernel": ("decode step = 1 CUDA-graph replay for 64 rows: decode_mega_kernel (all 48 layers, ~97% of "
                                    "the step; `traffic` is its ncu DRAM bytes at step 2, context 41) + lm_head GEMM + argmax")
                         if args.config == 2 else "decode step = 1 CUDA-graph replay for %d rows (layer stack + lm_head + token selection)" % rows_per_launch,
                         "bytes_per_launch": step_bytes, "ms_per_launch": step_ms, "peak_source": peak_src},
            "cpu_baseline": cpu,
        }
        if other is not None:
            line["other_configs"] = other
        print(json.dumps(line), file=_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
