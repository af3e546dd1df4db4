"""Executes the REFERENCE's own source for the hot path — TEST INFRASTRUCTURE.

The reference (the original comfyui-vrgamedevgirl node pack) is not part of this repository.  It is looked for where
VRGDG_REFERENCE_ROOT points, else in the git-ignored oracle/_ref/, else at /root/reference, where the golden vectors were
frozen from.  Nothing under `-m gpu`, smoke() or bench.py may import this module.  It is used by tests/golden/make_golden.py
to freeze golden vectors and by tests/test_oracle_golden.py (skipped without a reference checkout) to pin oracle/vrgdg_oracle.py.

Technique = the reference's own tests (tests/test_standalone_video_enhancer.py:19-36): ast.parse the file,
keep the wanted top-level definitions, exec them in a namespace of stand-ins for what ComfyUI provides.
No reference source is copied into this repository; it is compiled from where it lies.
"""
import ast
import importlib.util
import os
import sys
import types
from typing import Tuple, Union

import numpy as np
import torch
import torch.nn.functional as F

def _reference_root():
    if os.environ.get("VRGDG_REFERENCE_ROOT"):
        return os.environ["VRGDG_REFERENCE_ROOT"]
    for root in (os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"), "/root/reference"):
        if os.path.isfile(os.path.join(root, "nodes.py")):
            return root
    return "/root/reference"


REFERENCE_ROOT = _reference_root()


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "nodes.py"))


def _extract(path, names, namespace):
    with open(path, "r", encoding="utf-8") as fh:
        tree = ast.parse(fh.read(), filename=path)
    body = [n for n in tree.body if isinstance(n, (ast.ClassDef, ast.FunctionDef)) and n.name in names]
    missing = set(names) - {n.name for n in body}
    if missing:
        raise RuntimeError("reference no longer defines %s in %s" % (sorted(missing), path))
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), namespace)
    return namespace


def _comfy_stub():
    mm = types.SimpleNamespace(get_torch_device=lambda: torch.device("cpu"), intermediate_device=lambda: torch.device("cpu"))
    return types.SimpleNamespace(model_management=mm)


def _kornia_stub():
    # kornia is not vendored by the reference and not installed here: inject the restatement (parity unpinned)
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import vrgdg_oracle as oracle
    color = types.SimpleNamespace(rgb_to_lab=oracle.rgb_to_lab, lab_to_rgb=oracle.lab_to_rgb)
    return types.SimpleNamespace(color=color)


def load_filter_nodes():
    """The five filter classes of nodes.py:18-384, executed from the reference file."""
    ns = {"torch": torch, "F": F, "np": np, "Tuple": Tuple, "Union": Union, "comfy": _comfy_stub(), "kornia": _kornia_stub()}
    names = {"FastFilmGrain", "ColorMatchToReference", "FastUnsharpSharpen", "FastLaplacianSharpen", "FastSobelSharpen"}
    return _extract(os.path.join(REFERENCE_ROOT, "nodes.py"), names, ns)


def load_iv_adjustments():
    """VRGDG_IV_Adjustments.py imports as-is (os, numpy, torch only)."""
    path = os.path.join(REFERENCE_ROOT, "VRGDG_IV_Adjustments.py")
    spec = importlib.util.spec_from_file_location("_ref_iv_adjustments", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_enhancer_helpers():
    ns = {"torch": torch, "F": F}
    names = {"_auto_batch_size", "_resize_frames", "_apply_unsharp", "_apply_seeded_grain", "_apply_effects_batch"}
    return _extract(os.path.join(REFERENCE_ROOT, "VRGDG_StandaloneVideoEnhancerNodes.py"), names, ns)


def load_lut_video_helpers(iv=None):
    iv = iv if iv is not None else load_iv_adjustments()
    ns = {"torch": torch, "VRGDG_LUTS": iv.VRGDG_LUTS}
    names = {"_apply_lut_tensor", "_apply_film_grain_tensor", "_normalize_adjust_settings", "_apply_adjust_tensor"}
    return _extract(os.path.join(REFERENCE_ROOT, "VRGDG_LUTVideoTools.py"), names, ns)


def load_video_enhance_helpers():
    """_interpolation / _resize_batch / _restore_batch of VRGDG_VideoEnhanceNodes.py:45-106."""
    ns = {"torch": torch, "F": F}
    names = {"_interpolation", "_resize_batch", "_restore_batch"}
    return _extract(os.path.join(REFERENCE_ROOT, "VRGDG_VideoEnhanceNodes.py"), names, ns)
