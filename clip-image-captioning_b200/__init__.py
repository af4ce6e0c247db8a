"""clipcap_b200 -- B200-native caption-generation hot path (CLIP ViT-B/32 -> prefix mapper -> GPT-2 / GPT-J decode).

The compute lives in libclipcap_b200.so (hand-written sm_100a CUDA behind the C ABI of include/clipcap_b200.h);
this package is the Python host code that mirrors the reference's call surface.  Importing it needs no GPU;
creating an `Engine` does, and there is no CPU fallback.
"""
from . import _lib
from ._lib import GenParams, ModelDesc
from .engine import CLIP_TOWERS, Engine, EngineConfig
from . import evaluate_model, inference, lms, model, sampling, sharding, synthetic
from .lms import GPT2, GPTJ, IdTokenizer
from .model import CLIPCaptionModel, CLIPCaptionPrefixOnly

__all__ = ["CLIP_TOWERS", "Engine", "EngineConfig", "GenParams", "ModelDesc", "CLIPCaptionModel", "CLIPCaptionPrefixOnly", "GPT2", "GPTJ",
           "IdTokenizer", "inference", "evaluate_model", "sampling", "sharding", "synthetic", "lms", "model", "_lib"]
