"""The C-ABI library loads on a machine without a GPU and exports every entry point include/clipcap_b200.h declares
(no compute call is made here); creating a context without a device fails loudly instead of falling back."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "clipcap_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"CCB_API\s+[\w\s\*]+?\b(ccb_\w+)\s*\(", text)))


def test_header_declares_the_path():
    names = declared_symbols()
    for must in ("ccb_create", "ccb_destroy", "ccb_load_weight", "ccb_vit_encode", "ccb_map_prefix", "ccb_embed_tokens",
                 "ccb_lm_forward", "ccb_generate", "ccb_caption_images", "ccb_sample", "ccb_argmax", "ccb_beam_step"):
        assert must in names


def test_library_exports_every_declared_symbol():
    import clipcap_b200 as cc
    lib = cc._lib.load()
    missing = [n for n in declared_symbols() if not hasattr(lib, n)]
    assert not missing, missing


def test_bindings_cover_every_declared_symbol():
    import clipcap_b200 as cc
    bound = set(cc._lib.PROTOTYPES) if hasattr(cc._lib, "PROTOTYPES") else None
    if bound is None:
        pytest.skip("prototype table not exposed")
    assert set(declared_symbols()) <= bound | {"ccb_last_error", "ccb_create", "ccb_destroy"}


NO_DEVICE_CHILD = r"""
import sys
sys.path.insert(0, %(root)r)
import clipcap_b200 as cc
try:
    cc.Engine(cc.EngineConfig(lm_layers=1, map_layers=1, vit_layers=1, max_images=1))
except Exception as e:
    print("raised: %%s" %% e)
else:
    print("no error")
"""


def test_no_cpu_fallback():
    """In a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so that a GPU machine checks it too."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, "-c", NO_DEVICE_CHILD % {"root": ROOT}], env=env, capture_output=True, text=True,
                       timeout=300)
    out = r.stdout.strip().splitlines()
    assert r.returncode == 0 and out and out[-1].startswith("raised: "), r.stdout[-2000:] + r.stderr[-2000:]
    assert "CUDA" in out[-1] or "device" in out[-1]


def test_product_path_never_touches_the_oracle():
    """oracle/ is test / baseline infrastructure: only tests/, __graft_entry__.smoke() / build() and bench.py's CPU arms may
    import, link or execute anything under it.  No file of the package (host Python, CUDA sources, headers) names it."""
    import re
    pkg = os.path.join(ROOT, "clip-image-captioning_b200")
    offenders = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith((".py", ".cu", ".cuh", ".h")):
                continue
            text = open(os.path.join(dirpath, f), errors="ignore").read()
            if re.search(r"clipcap_oracle|ref_harness|build_ref|[\"'/]oracle[\"'/]|import oracle|from oracle", text):
                offenders.append(os.path.relpath(os.path.join(dirpath, f), ROOT))
    assert not offenders, offenders
    shim = open(os.path.join(ROOT, "clipcap_b200.py")).read()
    assert "oracle" not in shim
