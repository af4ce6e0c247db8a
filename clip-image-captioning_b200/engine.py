"""Python host side of libclipcap_b200: one `Engine` per GPU wraps a ccb_ctx.

PyTorch is used for device memory and streams only; every computation is a call through the C ABI
(include/clipcap_b200.h).  All tensors handed to the library are CUDA tensors on the engine's device.
"""
import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, Optional

import torch

from . import _lib
from ._lib import GenParams, ModelDesc


# The OpenAI CLIP ViT towers by their `clip.load` name (the reference picks its tower that way, inference.py:419): the
# vision tower (image, patch, width, layers, heads, output) and the matching text tower, as published in
# openai/CLIP clip/model.py `build_model` (heads = width // 64) and the HF `openai/clip-vit-*` configs.
CLIP_TOWERS = {
    "ViT-B/32": dict(vit_image=224, vit_patch=32, vit_width=768, vit_layers=12, vit_heads=12, vit_out=512,
                     text_width=512, text_layers=12, text_heads=8, text_out=512),
    "ViT-B/16": dict(vit_image=224, vit_patch=16, vit_width=768, vit_layers=12, vit_heads=12, vit_out=512,
                     text_width=512, text_layers=12, text_heads=8, text_out=512),
    "ViT-L/14": dict(vit_image=224, vit_patch=14, vit_width=1024, vit_layers=24, vit_heads=16, vit_out=768,
                     text_width=768, text_layers=12, text_heads=12, text_out=768),
    "ViT-L/14@336px": dict(vit_image=336, vit_patch=14, vit_width=1024, vit_layers=24, vit_heads=16, vit_out=768,
                           text_width=768, text_layers=12, text_heads=12, text_out=768),
}


@dataclass
class EngineConfig:
    """Shapes of the three networks on the path and the capacities of one context.

    Defaults are BASELINE.json config 2: ViT-B/32 + 8-layer Transformer mapper (prefix 40, clip_length 40) +
    GPT2-XL.  `lm_*` follow HF GPT2Config / GPTJConfig; `map_*` follow CLIPCaptionModel hparams
    (reference model.py:53-78); `vit_*` follow OpenAI CLIP ViT-B/32.
    """
    lm_arch: str = "gpt2"            # "gpt2" | "gptj"
    lm_d: int = 1600
    lm_layers: int = 48
    lm_heads: int = 25
    lm_vocab: int = 50257
    lm_n_pos: int = 1024
    lm_rotary_dim: int = 0
    lm_ln_eps: float = 1e-5
    map_kind: str = "transformer"    # "transformer" | "transformer_all" (use_all_vit_features: one mapper token per ViT
                                     # token, map_clip_len = ViT tokens, layers/Transformer.py:164-203) | "mlp" | "none"
    map_dim_clip: int = 512          # hparams.prefix_size
    map_clip_len: int = 40           # hparams.clip_prefix_length
    map_prefix_len: int = 40         # hparams.prefix_length
    map_heads: int = 8
    map_layers: int = 8
    map_mlp_ratio: float = 4.0
    map_hidden: int = 0              # 0 -> int(lm_d * mlp_ratio) (transformer) / lm_d * prefix_len // 2 (mlp)
    map_act: str = "relu"
    vit: bool = True
    vit_image: int = 224
    vit_patch: int = 32
    vit_width: int = 768
    vit_layers: int = 12
    vit_heads: int = 12
    vit_out: int = 512
    text: bool = False               # CLIP text tower for re-ranking (clip_model.encode_text, sampling.py:31)
    text_vocab: int = 49408
    text_ctx: int = 77
    text_width: int = 512
    text_layers: int = 12
    text_heads: int = 8
    text_out: int = 512
    max_texts: int = 64
    max_images: int = 64
    max_beam: int = 1
    max_ctx: int = 80
    max_lm_tokens: int = 0           # 0 -> max_images * max_ctx
    page_tokens: int = 16

    @classmethod
    def for_clip(cls, name: str, **overrides) -> "EngineConfig":
        """EngineConfig with the image and text towers of `clip.load(name)` ("ViT-B/32", "ViT-B/16", "ViT-L/14",
        "ViT-L/14@336px"); the mapper takes the tower's output width (`map_dim_clip`) and, with the all-features mapper,
        one token per ViT token (`map_clip_len` = 1 + patches).  `overrides` win."""
        if name not in CLIP_TOWERS:
            raise ValueError("unknown CLIP tower %r (known: %s)" % (name, ", ".join(CLIP_TOWERS)))
        kw = dict(CLIP_TOWERS[name])
        kw["map_dim_clip"] = kw["vit_out"]
        if overrides.get("map_kind", cls.map_kind) == "transformer_all":
            kw["map_clip_len"] = (kw["vit_image"] // kw["vit_patch"]) ** 2 + 1
        kw.update(overrides)
        return cls(**kw)

    def desc(self) -> ModelDesc:
        d = ModelDesc()
        d.lm_arch = {"gpt2": _lib.LM_GPT2, "gptj": _lib.LM_GPTJ}[self.lm_arch]
        d.lm_d, d.lm_layers, d.lm_heads, d.lm_vocab = self.lm_d, self.lm_layers, self.lm_heads, self.lm_vocab
        d.lm_n_pos, d.lm_rotary_dim, d.lm_ln_eps = self.lm_n_pos, self.lm_rotary_dim, self.lm_ln_eps
        d.map_kind = {"none": _lib.MAP_NONE, "transformer": _lib.MAP_TRANSFORMER, "mlp": _lib.MAP_MLP,
                      "transformer_all": _lib.MAP_TRANSFORMER_ALL}[self.map_kind]
        d.map_dim_clip, d.map_clip_len, d.map_prefix_len = self.map_dim_clip, self.map_clip_len, self.map_prefix_len
        d.map_heads, d.map_layers = self.map_heads, self.map_layers
        hidden = self.map_hidden
        if hidden == 0:
            hidden = (self.lm_d * self.map_prefix_len) // 2 if self.map_kind == "mlp" else int(self.lm_d * self.map_mlp_ratio)
        d.map_hidden = hidden
        d.map_act = _lib.ACT[self.map_act]
        d.vit_present = 1 if self.vit else 0
        d.vit_image, d.vit_patch, d.vit_width = self.vit_image, self.vit_patch, self.vit_width
        d.vit_layers, d.vit_heads, d.vit_out = self.vit_layers, self.vit_heads, self.vit_out
        d.max_images, d.max_beam, d.max_ctx = self.max_images, self.max_beam, self.max_ctx
        d.max_lm_tokens = self.max_lm_tokens or self.max_images * self.max_ctx
        d.page_tokens = self.page_tokens
        d.text_present = 1 if self.text else 0
        d.text_vocab, d.text_ctx, d.text_width = self.text_vocab, self.text_ctx, self.text_width
        d.text_layers, d.text_heads, d.text_out, d.max_texts = self.text_layers, self.text_heads, self.text_out, self.max_texts
        return d


_TORCH_DTYPE = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16}


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class Engine:
    """A ccb_ctx bound to one CUDA device."""

    def __init__(self, cfg: EngineConfig, device: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("clipcap_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.cfg = cfg
        self.device = torch.device("cuda", device)
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.zeros(1, device=self.device)  # make sure the primary context exists
            h = C.c_void_p()
            desc = cfg.desc()
            if self.lib.ccb_create(C.byref(h), C.byref(desc), device) != 0:
                raise RuntimeError(self.lib.ccb_last_error(None).decode())
        self._h = h
        self._desc = desc
        self.ldv = (cfg.lm_vocab + 63) // 64 * 64
        self._keep = []  # tensors referenced by in-flight asynchronous calls

    # ------------------------------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None):
            self.lib.ccb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, status: int):
        if status != 0:
            raise RuntimeError(self.lib.ccb_last_error(self._h).decode())

    def _dev(self, t: torch.Tensor, dtype=None) -> torch.Tensor:
        t = t.to(self.device, dtype=dtype) if dtype is not None else t.to(self.device)
        return t.contiguous()

    @property
    def device_bytes(self) -> int:
        return int(self.lib.ccb_device_bytes(self._h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.ccb_launch_count(self._h))

    def last_timing(self):
        """(prefill_ms, decode_ms, decode_steps) of the last generate call; synchronises the device."""
        torch.cuda.synchronize(self.device)
        a, b, n = C.c_float(), C.c_float(), C.c_int()
        self._check(self.lib.ccb_last_timing(self._h, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def timing_sum(self, n_calls: int):
        """(prefill_ms, decode_ms, decode_steps) summed over the last n_calls generate calls; synchronises."""
        torch.cuda.synchronize(self.device)
        a, b, n = C.c_float(), C.c_float(), C.c_int()
        self._check(self.lib.ccb_timing_sum(self._h, n_calls, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    # ------------------------------------------------------------------------------------------ weights
    def load_state_dict(self, sd: Dict[str, torch.Tensor], prefix: str = "", strict: bool = True):
        """Ingest tensors named as in the reference checkpoint (`language_model.*`, `clip_project.*`,
        `visual_encoder.*` / `visual.*`); `prefix` is prepended to every key (e.g. "clip_project." for a bare
        TransformerMapper.state_dict()).  Returns the list of keys the context did not use."""
        unused = []
        with torch.cuda.device(self.device):
            for k, v in sd.items():
                if not torch.is_tensor(v) or v.dtype not in _TORCH_DTYPE:
                    unused.append(k)
                    continue
                t = self._dev(v.detach())
                shape = (C.c_int64 * max(t.dim(), 1))(*(t.shape if t.dim() else (1,)))
                r = self.lib.ccb_load_weight(self._h, (prefix + k).encode(), _ptr(t), _TORCH_DTYPE[t.dtype], shape,
                                             max(t.dim(), 1), self._stream())
                if r < 0:
                    self._check(r)
                if r == 1:
                    unused.append(k)
            torch.cuda.synchronize(self.device)
        return unused

    def weights_complete(self) -> bool:
        return self.lib.ccb_weights_complete(self._h) == 0

    def check_weights(self):
        self._check(self.lib.ccb_weights_complete(self._h))

    # ------------------------------------------------------------------------------------------ preprocessing
    CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)   # clip/clip.py _transform
    CLIP_STD = (0.26862954, 0.26130258, 0.27577711)

    @staticmethod
    def resize_geometry(h: int, w: int, n_px: int):
        """(new_h, new_w, crop_top, crop_left) of Resize(n_px) + CenterCrop(n_px) exactly as torchvision computes them."""
        short, long = (w, h) if w <= h else (h, w)
        new_short, new_long = n_px, int(n_px * long / short)
        new_w, new_h = (new_short, new_long) if w <= h else (new_long, new_short)
        return new_h, new_w, int(round((new_h - n_px) / 2.0)), int(round((new_w - n_px) / 2.0))

    def preprocess_images(self, images, n_px: Optional[int] = None, mean=None, std=None) -> torch.Tensor:
        """CLIP's `_transform` on the device: a list of decoded RGB images (uint8 tensors [H, W, 3], any sizes) ->
        [B, 3, n_px, n_px] f32, bit-identical to Resize(n_px, BICUBIC) -> CenterCrop -> ToTensor -> Normalize on PIL images."""
        n_px = n_px or self.cfg.vit_image
        mean = (C.c_float * 3)(*(mean or self.CLIP_MEAN))
        std = (C.c_float * 3)(*(std or self.CLIP_STD))
        out = torch.empty(len(images), 3, n_px, n_px, device=self.device, dtype=torch.float32)
        held = []
        for i, im in enumerate(images):
            im = self._dev(im, torch.uint8).contiguous()
            if im.dim() != 3 or im.shape[2] != 3:
                raise ValueError("images must be uint8 [H, W, 3]")
            h, w = int(im.shape[0]), int(im.shape[1])
            nh, nw, top, left = self.resize_geometry(h, w, n_px)
            nbytes = int(self.lib.ccb_preprocess_scratch_bytes(h, w, nh, nw, n_px))
            scratch = torch.empty(nbytes, device=self.device, dtype=torch.uint8)
            self._check(self.lib.ccb_preprocess_image(self._h, _ptr(im), h, w, nh, nw, top, left, n_px, mean, std, _ptr(out[i]),
                                                      _ptr(scratch), nbytes, self._stream()))
            held += [im, scratch]
        self._keep = held
        return out

    # ------------------------------------------------------------------------------------------ stages
    def vit_encode(self, images: torch.Tensor, all_tokens: Optional[bool] = None) -> torch.Tensor:
        """[B, vit_out] (CLS token through ln_post and proj), or with all_tokens (default for the "transformer_all"
        mapper: the fork's patched forward, inference.py:421-444) [B, 1 + patches, vit_out]."""
        images = self._dev(images)
        if images.dtype not in _TORCH_DTYPE:
            images = images.float()
        B = images.shape[0]
        if all_tokens is None:
            all_tokens = self.cfg.map_kind == "transformer_all"
        if all_tokens:
            n = (self.cfg.vit_image // self.cfg.vit_patch) ** 2 + 1
            out = torch.empty(B, n, self.cfg.vit_out, device=self.device, dtype=torch.float32)
            self._check(self.lib.ccb_vit_encode_tokens(self._h, _ptr(images), _TORCH_DTYPE[images.dtype], B, _ptr(out), self._stream()))
            return out
        out = torch.empty(B, self.cfg.vit_out, device=self.device, dtype=torch.float32)
        self._check(self.lib.ccb_vit_encode(self._h, _ptr(images), _TORCH_DTYPE[images.dtype], B, _ptr(out), self._stream()))
        return out

    def clip_encode_text(self, tokens: torch.Tensor) -> torch.Tensor:
        """clip_model.encode_text(tokens) (sampling.py:31): tokens [B, text_ctx] (clip.tokenize ids; the end-of-text token is
        the largest id) -> [B, text_out] f32, un-normalised."""
        tk = self._dev(tokens, torch.int32)
        if tk.dim() != 2 or tk.shape[1] != self.cfg.text_ctx:
            raise ValueError("tokens must be [B, %d]" % self.cfg.text_ctx)
        self._check_ids(tk, self.cfg.text_vocab, "clip_encode_text")
        out = torch.empty(tk.shape[0], self.cfg.text_out, device=self.device, dtype=torch.float32)
        self._check(self.lib.ccb_clip_encode_text(self._h, _ptr(tk), tk.shape[0], _ptr(out), self._stream()))
        return out

    def map_prefix(self, feat: torch.Tensor) -> torch.Tensor:
        feat = self._dev(feat, torch.float32)
        B = feat.shape[0]
        if self.cfg.map_kind == "transformer_all":
            if feat.dim() != 3 or feat.shape[1] != self.cfg.map_clip_len or feat.shape[2] != self.cfg.map_dim_clip:
                raise ValueError("transformer_all mapper expects features [B, %d, %d]" % (self.cfg.map_clip_len, self.cfg.map_dim_clip))
        elif feat.dim() != 2 or feat.shape[1] != self.cfg.map_dim_clip:
            raise ValueError("mapper expects features [B, %d]" % self.cfg.map_dim_clip)
        out = torch.empty(B, self.cfg.map_prefix_len, self.cfg.lm_d, device=self.device, dtype=torch.float32)
        self._check(self.lib.ccb_map_prefix(self._h, _ptr(feat), B, _ptr(out), self._stream()))
        return out

    @staticmethod
    def _check_ids(ids: torch.Tensor, n: int, what: str, also_ok: Optional[int] = None):
        """torch's embedding / cross_entropy raise on ids outside [0, n): same here (the reference dataset pads with -1,
        model.py:204 masks those before the lookup; the kernels clamp rather than fault)."""
        if ids.numel() == 0:
            return
        bad = (ids < 0) | (ids >= n)
        if also_ok is not None:
            bad &= ids != also_ok
        if bool(bad.any()):
            raise IndexError("%s: id out of range [0, %d): %d" % (what, n, int(ids[bad].flatten()[0])))

    def embed_tokens(self, tokens: torch.Tensor) -> torch.Tensor:
        self._check_ids(tokens, self.cfg.lm_vocab, "embed_tokens")
        tk = self._dev(tokens, torch.int32)
        out = torch.empty(*tk.shape, self.cfg.lm_d, device=self.device, dtype=torch.float32)
        if tk.numel():
            self._check(self.lib.ccb_embed_tokens(self._h, _ptr(tk), tk.numel(), _ptr(out), self._stream()))
        return out

    def lm_forward(self, embeds: torch.Tensor, attention_mask: Optional[torch.Tensor] = None,
                   last_only: bool = False) -> torch.Tensor:
        embeds = self._dev(embeds, torch.float32)
        B, S, _ = embeds.shape
        mask = None
        if attention_mask is not None:
            mask = self._dev(attention_mask.to(torch.bool)).to(torch.uint8).contiguous()
        rows = B if last_only else B * S
        buf = torch.empty(rows, self.ldv, device=self.device, dtype=torch.float32)
        self._check(self.lib.ccb_lm_forward(self._h, _ptr(embeds), B, S, _ptr(mask), _ptr(buf), self.ldv,
                                            1 if last_only else 0, self._stream()))
        V = self.cfg.lm_vocab
        return buf[:, :V] if last_only else buf.view(B, S, self.ldv)[:, :, :V]

    # ------------------------------------------------------------------------------------------ generation
    def gen_params(self, mode: str, max_new_tokens: int, stop_token: int = 13, max_stops: int = 1, eos_token: int = -1,
                   temperature: float = 1.0, top_p: float = 0.0, top_k: int = 0, repetition_penalty: float = 1.0,
                   beam_size: int = 1, seed: int = 0, q_noise: Optional[torch.Tensor] = None,
                   row_ids: Optional[torch.Tensor] = None, top_p_rows: Optional[torch.Tensor] = None,
                   top_k_rows: Optional[torch.Tensor] = None, typ_p: float = 0.0,
                   typ_p_rows: Optional[torch.Tensor] = None, normalized: bool = False):
        """`normalized=True`: the per-row budgets already follow the kernel's conventions (top_p_rows <= 0 / typ_p_rows < 0 =
        leave the row alone) -- no host-side inspection of device tensors, hence no synchronisation."""
        p = GenParams()
        p.mode = {"greedy": _lib.GEN_GREEDY, "sample": _lib.GEN_SAMPLE, "beam": _lib.GEN_BEAM}[mode]
        p.max_new_tokens, p.stop_token, p.max_stops, p.eos_token = max_new_tokens, stop_token, max_stops, eos_token
        p.temperature, p.top_p, p.top_k, p.repetition_penalty = temperature, top_p, top_k, repetition_penalty
        p.beam_size, p.seed = beam_size, seed
        p.typ_p = typ_p
        keep = []
        if q_noise is not None:
            q_noise = self._dev(q_noise, torch.float32)
            p.q_noise, p.q_ld = q_noise.data_ptr(), q_noise.shape[-1]
            keep.append(q_noise)
        if row_ids is not None:
            row_ids = self._dev(row_ids, torch.int64)
            p.row_ids = row_ids.data_ptr()
            keep.append(row_ids)
        if top_p_rows is not None:
            top_p_rows = self._dev(top_p_rows, torch.float32)
            # sampling.py:149-160: with a tensor of budgets the nucleus filter runs on EVERY row as soon as one budget is
            # positive, and a row whose budget is <= 0 then keeps its top-1 token only (cumsum > top_p holds everywhere);
            # the kernel skips rows with a budget <= 0, so those get the smallest positive budget instead
            if normalized:
                pass
            elif bool((top_p_rows > 0).any()):
                top_p_rows = torch.where(top_p_rows > 0, top_p_rows, torch.full_like(top_p_rows, 1e-30))
            else:
                top_p_rows = None
        if top_p_rows is not None:
            p.top_p_rows = top_p_rows.data_ptr()
            keep.append(top_p_rows)
        if top_k_rows is not None:
            top_k_rows = self._dev(top_k_rows, torch.int32)
            p.top_k_rows = top_k_rows.data_ptr()
            keep.append(top_k_rows)
        if typ_p_rows is not None:
            typ_p_rows = self._dev(typ_p_rows, torch.float32)
            p.typ_p_rows = typ_p_rows.data_ptr()
            keep.append(typ_p_rows)
        p._keep = keep
        return p

    def _gen_outputs(self, p: GenParams, N: int):
        T = p.max_new_tokens
        if p.mode == _lib.GEN_BEAM:
            tokens = torch.empty(N, p.beam_size, T, device=self.device, dtype=torch.int32)
            lengths = torch.empty(N, p.beam_size, device=self.device, dtype=torch.int32)
            scores = torch.empty(N, p.beam_size, device=self.device, dtype=torch.float32)
        else:
            tokens = torch.empty(N, T, device=self.device, dtype=torch.int32)
            lengths = torch.empty(N, device=self.device, dtype=torch.int32)
            scores = None
        return tokens, lengths, scores

    def generate(self, embeds: torch.Tensor, p: GenParams):
        """Prefix embeddings [N, S0, d] -> (tokens, lengths, scores) on the device, whole loop on the GPU."""
        embeds = self._dev(embeds, torch.float32)
        N, S0, _ = embeds.shape
        tokens, lengths, scores = self._gen_outputs(p, N)
        self._check(self.lib.ccb_generate(self._h, C.byref(p), _ptr(embeds), N, S0, _ptr(tokens), _ptr(lengths),
                                          _ptr(scores), self._stream()))
        self._keep = [embeds, p]
        return tokens, lengths, scores

    def caption_images(self, images: torch.Tensor, p: GenParams, append_bos: int = -1):
        """Images [N,3,H,W] -> (tokens, lengths, scores): ViT + mapper + generation in one library call."""
        images = self._dev(images)
        if images.dtype not in _TORCH_DTYPE:
            images = images.float()
        N = images.shape[0]
        tokens, lengths, scores = self._gen_outputs(p, N)
        self._check(self.lib.ccb_caption_images(self._h, C.byref(p), _ptr(images), _TORCH_DTYPE[images.dtype], N,
                                                append_bos, _ptr(tokens), _ptr(lengths), _ptr(scores), self._stream()))
        self._keep = [images, p]
        return tokens, lengths, scores

    def micro_batch_for(self, p: GenParams) -> int:
        """Images per call that keep the decode step on its fastest path: the persistent decode kernel takes at most
        256 rows, so beam search (beam rows per image) runs 256 // beam images at a time (51 for beam 5: 290 captions/s
        on GPT2-XL against 230 for 64 images = 320 rows on the operator chain); otherwise the engine's max_images."""
        n = self.cfg.max_images
        if p.mode == _lib.GEN_BEAM and p.beam_size > 0:
            n = min(n, max(1, 256 // p.beam_size))
        return n

    def caption_dataset(self, images: torch.Tensor, p: GenParams, micro_batch: Optional[int] = None,
                        first_row_id: int = 0, append_bos: int = -1):
        """Captions for any number of images (this rank's shard, SURVEY 8e): runs `caption_images` over micro-batches
        and concatenates.  In sampling mode the Philox streams are keyed by first_row_id + image index, so the result
        does not depend on the micro-batch size or on how the images were sharded over GPUs."""
        n = images.shape[0]
        mb = micro_batch or self.micro_batch_for(p)
        toks, lens, scs = [], [], []
        keep_ids = p.row_ids
        # ONE id buffer, rewritten in place per micro-batch (stream-ordered behind the previous call): the captured decode
        # step is keyed by the pointers it reads, so a fresh tensor per micro-batch would re-capture the graph every time
        ids = None
        if p.mode == _lib.GEN_SAMPLE and not p.q_noise:
            ids = torch.empty(mb, dtype=torch.int64, device=self.device)
            p.row_ids = ids.data_ptr()
        for lo in range(0, n, mb):
            hi = min(n, lo + mb)
            if ids is not None:
                ids[:hi - lo].copy_(torch.arange(first_row_id + lo, first_row_id + hi, dtype=torch.int64, device=self.device))
            t, l, sc = self.caption_images(images[lo:hi], p, append_bos)
            toks.append(t)
            lens.append(l)
            scs.append(sc)
        p.row_ids = keep_ids
        self._keep.append(ids)       # read by the kernels of the last call
        tokens, lengths = torch.cat(toks, 0), torch.cat(lens, 0)
        scores = torch.cat(scs, 0) if scs and scs[0] is not None else None
        return tokens, lengths, scores

    def caption_dataset_continuous(self, images: torch.Tensor, p: GenParams, rows: Optional[int] = None,
                                   first_row_id: int = 0, append_bos: int = -1):
        """`caption_dataset` with continuous batching (ccb_caption_dataset), greedy or sampling: `rows` decode slots
        (default `micro_batch_for(p)`) stay busy, and a slot whose caption has finished takes the next image instead of
        decoding to max_new_tokens.  Returns (tokens [n, T], lengths [n], decode steps run).  Per image the caption equals
        `caption_dataset`'s; positions at or past a caption's length are 0.  Sampling keys the Philox streams by
        first_row_id + image index, as `caption_dataset` does.  Synchronises the host once per round of decode steps."""
        images = self._dev(images)
        if images.dtype not in _TORCH_DTYPE:
            images = images.float()
        n = images.shape[0]
        rows = rows or self.micro_batch_for(p)
        tokens = torch.empty(n, p.max_new_tokens, device=self.device, dtype=torch.int32)
        lengths = torch.empty(n, device=self.device, dtype=torch.int32)
        steps = C.c_int64()
        self._check(self.lib.ccb_caption_dataset(self._h, C.byref(p), _ptr(images), _TORCH_DTYPE[images.dtype], n, rows,
                                                 append_bos, first_row_id, _ptr(tokens), _ptr(lengths), C.byref(steps),
                                                 self._stream()))
        self._keep = [images, p]
        return tokens, lengths, int(steps.value)

    def caption_dataset_continuous_beam(self, images: torch.Tensor, p: GenParams, groups: Optional[int] = None,
                                        append_bos: int = -1):
        """`caption_dataset` in beam mode with continuous batching (ccb_caption_dataset_beam): `groups` images (default
        `micro_batch_for(p)`) are in flight with beam_size decode rows each, and an image whose beams have all stopped,
        or that has max_new_tokens tokens, gives its group to the next image (generate_beam, inference.py:70-148, stops
        there too).  Returns (tokens [n, beam, T], lengths [n, beam], scores [n, beam], decode steps run), the layout of
        `caption_dataset` in beam mode; positions past a beam's length are 0.  Synchronises the host once per round of
        decode steps."""
        images = self._dev(images)
        if images.dtype not in _TORCH_DTYPE:
            images = images.float()
        n = images.shape[0]
        groups = groups or self.micro_batch_for(p)
        # (non-empty even for the arguments the library rejects, so that it names the reason)
        beam, T = max(p.beam_size, 1), max(p.max_new_tokens, 1)
        tokens = torch.empty(n, beam, T, device=self.device, dtype=torch.int32)
        lengths = torch.empty(n, beam, device=self.device, dtype=torch.int32)
        scores = torch.empty(n, beam, device=self.device, dtype=torch.float32)
        steps = C.c_int64()
        self._check(self.lib.ccb_caption_dataset_beam(self._h, C.byref(p), _ptr(images), _TORCH_DTYPE[images.dtype], n,
                                                      groups, append_bos, _ptr(tokens), _ptr(lengths), _ptr(scores),
                                                      C.byref(steps), self._stream()))
        self._keep = [images, p]
        return tokens, lengths, scores, int(steps.value)

    # ------------------------------------------------------------------------------------------ samplers
    def sample(self, logits: torch.Tensor, p: GenParams, history: Optional[torch.Tensor] = None, step: int = 0,
               return_filtered: bool = False, return_alt: bool = False):
        logits = self._dev(logits, torch.float32)
        B, V = logits.shape
        hist = self._dev(history, torch.int32) if history is not None and history.numel() else None
        filt = torch.empty_like(logits) if return_filtered else None
        nxt = torch.empty(B, device=self.device, dtype=torch.int32)
        alt = torch.empty(B, device=self.device, dtype=torch.int32) if return_alt else None
        self._check(self.lib.ccb_sample(self._h, _ptr(logits), logits.stride(0), B, V, C.byref(p), _ptr(hist),
                                        hist.stride(0) if hist is not None else 0,
                                        hist.shape[1] if hist is not None else 0, step, _ptr(filt), _ptr(nxt), _ptr(alt),
                                        self._stream()))
        return nxt, filt, alt

    def argmax(self, logits: torch.Tensor) -> torch.Tensor:
        logits = self._dev(logits, torch.float32)
        B, V = logits.shape
        nxt = torch.empty(B, device=self.device, dtype=torch.int32)
        self._check(self.lib.ccb_argmax(self._h, _ptr(logits), logits.stride(0), B, V, _ptr(nxt), self._stream()))
        return nxt

    def cross_entropy(self, logits: torch.Tensor, targets: torch.Tensor, ignore_index: int = -100,
                      row_map: Optional[torch.Tensor] = None):
        """`F.cross_entropy(logits, targets, ignore_index=...)` (mean reduction) on the device: logits [n, V] f32 (rows may be
        strided), targets [rows]; `row_map` [rows] picks the logits row of each target (default: row r).  Returns
        (loss 0-d tensor, per-row loss [rows], number of counted rows 0-d tensor)."""
        if logits.dim() != 2 or logits.stride(1) != 1:
            raise ValueError("cross_entropy: logits must be [n, V] with unit stride along V")
        logits = logits.to(self.device, dtype=torch.float32)      # (rows may be strided: the pitch goes to the kernel, no copy)
        tg = self._dev(targets).to(torch.int32).contiguous().view(-1)
        rows, V = tg.numel(), logits.shape[1]
        self._check_ids(tg, V, "cross_entropy targets", also_ok=ignore_index)
        rm = None
        if row_map is not None:
            rm = self._dev(row_map).to(torch.int32).contiguous().view(-1)
            if rm.numel() != rows:
                raise ValueError("cross_entropy: row_map and targets differ in length")
        elif logits.shape[0] != rows:
            raise ValueError("cross_entropy: %d logits rows for %d targets" % (logits.shape[0], rows))
        row_loss = torch.empty(rows, device=self.device, dtype=torch.float32)
        out = torch.empty(2, device=self.device, dtype=torch.float32)
        self._check(self.lib.ccb_cross_entropy(self._h, _ptr(logits), logits.stride(0), rows, V, _ptr(tg), _ptr(rm), ignore_index,
                                               _ptr(row_loss), _ptr(out), self._stream()))
        return out[0], row_loss, out[1]

    def beam_step(self, logits, scores, seq_lengths, has_stopped, tokens, step: int, beam: int, temperature=1.0,
                  stop_token=13):
        """One step of inference.py:98-131 for N images; state tensors are updated in place."""
        logits = self._dev(logits, torch.float32)
        N = scores.shape[0]
        V = logits.shape[1]
        nxt = torch.empty(N * beam, device=self.device, dtype=torch.int32)
        src = torch.empty(N * beam, device=self.device, dtype=torch.int32)
        self._check(self.lib.ccb_beam_step(self._h, _ptr(logits), logits.stride(0), N, beam, V, temperature, stop_token,
                                           step, _ptr(scores), _ptr(seq_lengths), _ptr(has_stopped), _ptr(tokens),
                                           tokens.shape[-1], _ptr(nxt), _ptr(src), self._stream()))
        return nxt, src

    # ------------------------------------------------------------------------------------------ single ops
    def _rows(self, t, dtype, tma):
        """t as a [rows, cols] GEMM operand on this device.  A view with unit column stride is passed as it is, its
        stride(0) becoming the row pitch, when the kernels can address it (16-byte aligned base; for operands read through
        a tensor map (`tma`) also a pitch of whole 16 bytes); anything else is copied contiguous."""
        if (t.device == self.device and t.dtype == dtype and t.dim() == 2 and t.stride(1) == 1 and
                t.stride(0) >= t.shape[1] and t.data_ptr() % 16 == 0 and
                (not tma or t.stride(0) * t.element_size() % 16 == 0)):
            return t
        return self._dev(t, dtype)

    def op_linear(self, x, w, bias=None, act="none", residual=None, out_dtype=torch.float32, orientation=0, bn=0,
                  split_k=0, *, out=None, residual_is_out=False, row_remap=None):
        """act(x @ w.T + bias) + residual with x [tokens, K] bf16, w [features, K] bf16 (tcgen05 GEMM,
        ccb_op_linear_ex).  x, w and residual may be row-strided views: their row pitches go to the kernel.

        out: a caller-owned [rows, features] f32 or bf16 view (row pitch stride(0), any offset) written in place and
        returned; by default a new [tokens, features] tensor of out_dtype.  residual_is_out: the residual is read from
        `out` itself (f32), as the engine's residual stream does.  row_remap (rg_in, rg_out, rg_off): token row t lands in
        out row (t // rg_in) * rg_out + rg_off + t % rg_in (normal orientation only)."""
        x = self._rows(x, torch.bfloat16, True)
        w = self._rows(w, torch.bfloat16, True)
        tokens, K = x.shape
        features = w.shape[0]
        rg_in, rg_out, rg_off = row_remap or (0, 0, 0)
        bias = self._dev(bias, torch.float32) if bias is not None else None
        if residual_is_out and (out is None or residual is not None or out.dtype != torch.float32):
            raise ValueError("residual_is_out needs an f32 `out` and no separate residual")
        if out is None:
            out = torch.empty(tokens, features, device=self.device, dtype=out_dtype)
        elif (out.device != self.device or out.dtype not in (torch.float32, torch.bfloat16) or out.dim() != 2 or
              out.stride(1) != 1 or out.shape[1] != features):
            raise ValueError("out must be a [rows, %d] f32 or bf16 view on %s with unit column stride" % (features, self.device))
        last = tokens - 1 if not rg_in else (tokens - 1) // rg_in * rg_out + rg_off + (tokens - 1) % rg_in
        if out.shape[0] <= last:
            raise ValueError("out has %d rows; token row %d lands in row %d" % (out.shape[0], tokens - 1, last))
        if residual_is_out:
            residual = out
        elif residual is not None:
            residual = self._rows(residual, torch.float32, False)
        self._check(self.lib.ccb_op_linear_ex(self._h, _ptr(x), x.stride(0), tokens, _ptr(w), w.stride(0), features, K,
                                              _ptr(bias), _lib.ACT[act], _ptr(residual),
                                              residual.stride(0) if residual is not None else 0, _ptr(out), out.stride(0),
                                              1 if out.dtype == torch.bfloat16 else 0, rg_in, rg_out, rg_off, orientation,
                                              bn, split_k, self._stream()))
        return out

    def op_layernorm(self, x, gamma, beta, eps=1e-5):
        x = self._dev(x, torch.float32)
        rows, d = x.shape
        y = torch.empty(rows, d, device=self.device, dtype=torch.bfloat16)
        g, b = self._dev(gamma, torch.float32), self._dev(beta, torch.float32)  # keep both alive across the call
        self._check(self.lib.ccb_op_layernorm(self._h, _ptr(x), _ptr(g), _ptr(b), eps, _ptr(y), rows, d, self._stream()))
        return y

    def op_attention(self, qkv, B, S, H, hd, causal=False, rotary_dim=0, scale=None):
        qkv = self._dev(qkv, torch.bfloat16)
        out = torch.empty(B * S, H * hd, device=self.device, dtype=torch.bfloat16)
        self._check(self.lib.ccb_op_attention(self._h, _ptr(qkv), _ptr(out), B, S, H, hd,
                                              scale if scale is not None else hd ** -0.5, 1 if causal else 0, rotary_dim,
                                              self._stream()))
        return out

    def op_attention_decode(self, qkv, kv, layer, page_tokens, block_table, ctx_len, H, hd, rotary_dim=0, scale=None,
                            ldo=None):
        """One decode step over a paged KV cache (ccb_op_attention_decode): qkv [rows, 3*H*hd] bf16 (the new tokens),
        kv [layers, 2, num_pages, H, page_tokens, hd] bf16 (the new k / v are written into it), block_table
        [rows, max_pages_per_row] int32, ctx_len [rows] int32.  Returns out [rows, ldo] bf16 (ldo defaults to H*hd); the
        columns past H*hd are left as allocated."""
        if kv.dtype != torch.bfloat16 or not kv.is_contiguous() or kv.dim() != 6 or tuple(kv.shape[3:]) != (H, page_tokens, hd):
            raise ValueError("kv must be a contiguous bf16 [layers, 2, num_pages, %d, %d, %d] tensor" % (H, page_tokens, hd))
        qkv = self._dev(qkv, torch.bfloat16)
        bt = self._dev(block_table, torch.int32)
        cl = self._dev(ctx_len, torch.int32)
        rows = qkv.shape[0]
        ldo = ldo or H * hd
        out = torch.zeros(rows, ldo, device=self.device, dtype=torch.bfloat16)
        self._check(self.lib.ccb_op_attention_decode(self._h, _ptr(qkv), _ptr(out), ldo, rows, H, hd,
                                                     scale if scale is not None else hd ** -0.5, _ptr(kv), kv.shape[0], layer,
                                                     kv.shape[2], page_tokens, bt.shape[1], _ptr(bt), _ptr(cl), rotary_dim,
                                                     self._stream()))
        self._keep = [qkv, bt, cl]
        return out

    def debug_kv_layout(self):
        """(layers, heads, head_dim, page_tokens, num_pages, max_pages_per_row) of the last generate call's KV pool."""
        out = (C.c_int64 * 6)()
        self._check(self.lib.ccb_debug_kv_layout(self._h, out))
        return tuple(int(v) for v in out)

    def debug_copy_buffer(self, which: int, numel: int, dtype) -> torch.Tensor:
        """The first `numel` elements of internal buffer `which` (ccb_debug_copy_buffer), copied on the current stream."""
        out = torch.empty(numel, dtype=dtype, device=self.device)
        self._check(self.lib.ccb_debug_copy_buffer(self._h, which, _ptr(out), out.numel() * out.element_size(), self._stream()))
        return out
