"""ctypes binding of include/clipcap_b200.h (libclipcap_b200.so).

There is no CPU fallback: if the shared library is missing the import fails with instructions, and every entry
point raises RuntimeError(ccb_last_error) on a non-zero status.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CCB_LIB: another build of the same library (tools/build_variant.py: A/B measurements of kernel variants)
LIB_PATH = os.environ.get("CCB_LIB") or os.path.join(_HERE, "libclipcap_b200.so")

DTYPE_F32, DTYPE_F16, DTYPE_BF16 = 0, 1, 2
LM_GPT2, LM_GPTJ = 0, 1
MAP_NONE, MAP_TRANSFORMER, MAP_MLP, MAP_TRANSFORMER_ALL = 0, 1, 2, 3
ACT = {"none": 0, "relu": 1, "quick_gelu": 2, "gelu_new": 3, "gelu": 4, "elu": 5, "selu": 6, "tanh": 7, "geglu": 8}
GEN_GREEDY, GEN_SAMPLE, GEN_BEAM = 0, 1, 2


class ModelDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "lm_arch", "lm_d", "lm_layers", "lm_heads", "lm_vocab", "lm_n_pos", "lm_rotary_dim")] + [
        ("lm_ln_eps", C.c_float)] + [(n, C.c_int32) for n in (
            "map_kind", "map_dim_clip", "map_clip_len", "map_prefix_len", "map_heads", "map_layers", "map_hidden",
            "map_act",
            "vit_present", "vit_image", "vit_patch", "vit_width", "vit_layers", "vit_heads", "vit_out",
            "max_images", "max_beam", "max_ctx", "max_lm_tokens", "page_tokens",
            "text_present", "text_vocab", "text_ctx", "text_width", "text_layers", "text_heads", "text_out", "max_texts")]


class GenParams(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("max_new_tokens", C.c_int32), ("stop_token", C.c_int32), ("max_stops", C.c_int32),
        ("eos_token", C.c_int32), ("temperature", C.c_float), ("top_p", C.c_float), ("top_k", C.c_int32),
        ("repetition_penalty", C.c_float), ("beam_size", C.c_int32), ("seed", C.c_uint64),
        ("q_noise", C.c_void_p), ("q_ld", C.c_int64), ("row_ids", C.c_void_p), ("top_p_rows", C.c_void_p),
        ("top_k_rows", C.c_void_p), ("typ_p", C.c_float), ("typ_p_rows", C.c_void_p)]


_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> (restype, argtypes); mirrors include/clipcap_b200.h one to one
PROTOTYPES = {
    "ccb_create": (_I, [C.POINTER(_P), C.POINTER(ModelDesc), _I]),
    "ccb_destroy": (None, [_P]),
    "ccb_last_error": (C.c_char_p, [_P]),
    "ccb_device_bytes": (_L, [_P]),
    "ccb_load_weight": (_I, [_P, C.c_char_p, _P, _I, C.POINTER(_L), _I, _P]),
    "ccb_weights_complete": (_I, [_P]),
    "ccb_preprocess_scratch_bytes": (_L, [_I, _I, _I, _I, _I]),
    "ccb_preprocess_image": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, C.POINTER(_F), C.POINTER(_F), _P, _P, _L, _P]),
    "ccb_vit_encode": (_I, [_P, _P, _I, _I, _P, _P]),
    "ccb_vit_encode_tokens": (_I, [_P, _P, _I, _I, _P, _P]),
    "ccb_clip_encode_text": (_I, [_P, _P, _I, _P, _P]),
    "ccb_map_prefix": (_I, [_P, _P, _I, _P, _P]),
    "ccb_embed_tokens": (_I, [_P, _P, _I, _P, _P]),
    "ccb_lm_forward": (_I, [_P, _P, _I, _I, _P, _P, _L, _I, _P]),
    "ccb_generate": (_I, [_P, C.POINTER(GenParams), _P, _I, _I, _P, _P, _P, _P]),
    "ccb_caption_images": (_I, [_P, C.POINTER(GenParams), _P, _I, _I, _I, _P, _P, _P, _P]),
    "ccb_launch_count": (_L, [_P]),
    "ccb_last_timing": (_I, [_P, C.POINTER(_F), C.POINTER(_F), C.POINTER(_I)]),
    "ccb_timing_sum": (_I, [_P, _I, C.POINTER(_F), C.POINTER(_F), C.POINTER(_I)]),
    "ccb_sample": (_I, [_P, _P, _L, _I, _I, C.POINTER(GenParams), _P, _L, _I, _I, _P, _P, _P, _P]),
    "ccb_argmax": (_I, [_P, _P, _L, _I, _I, _P, _P]),
    "ccb_cross_entropy": (_I, [_P, _P, _L, _I, _I, _P, _P, _I, _P, _P, _P]),
    "ccb_beam_step": (_I, [_P, _P, _L, _I, _I, _I, _F, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P]),
    "ccb_op_linear": (_I, [_P, _P, _L, _I, _P, _I, _I, _P, _I, _P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "ccb_op_linear_ex": (_I, [_P, _P, _L, _I, _P, _L, _I, _I, _P, _I, _P, _L, _P, _L, _I, _I, _I, _I, _I, _I, _I, _P]),
    "ccb_debug_gemm_trace": (_I, [_P, _P, _L, _I]),
    "ccb_debug_mega_trace": (_I, [_P, _P]),
    "ccb_debug_set_mega": (_I, [_P, _I]),
    "ccb_debug_copy_buffer": (_I, [_P, _I, _P, _L, _P]),
    "ccb_debug_kv_layout": (_I, [_P, C.POINTER(_L)]),
    "ccb_op_layernorm": (_I, [_P, _P, _P, _P, _F, _P, _I, _I, _P]),
    "ccb_op_attention": (_I, [_P, _P, _P, _I, _I, _I, _I, _F, _I, _I, _P]),
    "ccb_op_attention_decode": (_I, [_P, _P, _P, _L, _I, _I, _I, _F, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P]),
}

_lib = None


def load():
    """dlopen libclipcap_b200.so and attach the prototypes (cached)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libclipcap_b200.so is not built (%s). Run `python tools/build.py` (nvcc, sm_100a). "
            "There is no CPU / PyTorch fallback for this path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
