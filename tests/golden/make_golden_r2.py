"""Round-2 additions to the golden vectors, produced by EXECUTING THE REFERENCE'S OWN SOURCE (oracle/ref_harness.py).

Needs a checkout of the reference:   VRGDG_REFERENCE_ROOT=<checkout> python tests/golden/make_golden_r2.py
  lut_big.npz : VRGDG_LUTS._parse_cube_file + _apply_cube_lut + the strength blend of apply_lut on generated 64^3 / 65^3 tables
                (tests/helpers.py::write_big_cube; the 65^3 file carries integer DOMAIN_MIN/MAX lines)
"""
import hashlib
import os
import sys
import tempfile
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ref_harness as RH  # noqa: E402
from helpers import natural_frames, white_frames, write_big_cube  # noqa: E402

warnings.filterwarnings("ignore")
torch.set_num_threads(4)


def main():
    assert RH.available(), "reference tree not found"
    iv = RH.load_iv_adjustments()
    out = {}
    xw = white_frames(1, 48, 64, seed=31)
    xw[0, 0, 0] = torch.tensor([1.0, 0.0, 1.0])
    xw[0, 0, 1] = torch.tensor([0.0, 0.0, 0.0])
    xw[0, 0, 2] = torch.tensor([1.0, 1.0, 1.0])
    xw[0, 0, 3] = torch.tensor([0.5, 0.25, 0.75])                     # exact grid nodes of the 65^3 table
    xw[0, 0, 4] = torch.tensor([1.0 / 63.0, 62.0 / 63.0, 0.5])        # grid nodes / mid-cell of the 64^3 table
    xn = natural_frames(1, 48, 64, seed=32)
    out["x"], out["xn"] = xw, xn
    with tempfile.TemporaryDirectory() as tmp:
        iv.LUTS_DIR = tmp
        node = iv.VRGDG_LUTS()
        for size in (64, 65):
            name = "big_%d.cube" % size
            write_big_cube(os.path.join(tmp, name), size)
            data = iv.VRGDG_LUTS._parse_cube_file(os.path.join(tmp, name))
            assert data["size"] == size
            out["sha_%d" % size] = np.frombuffer(hashlib.sha256(data["lut"].contiguous().numpy().tobytes()).digest(), dtype=np.uint8)
            out["s%d__s10" % size] = node.apply_lut(xw, name, "cpu", 10.0)[0]
            out["s%d__s3p5" % size] = node.apply_lut(xw, name, "cpu", 3.5)[0]
            out["s%d__nat" % size] = node.apply_lut(xn, name, "cpu", 10.0)[0]
            out["s%d__fp16" % size] = node.apply_lut(xw.half(), name, "cpu", 10.0)[0]
    arrays = {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in out.items()}
    np.savez_compressed(os.path.join(HERE, "lut_big.npz"), **arrays)
    print("lut_big", {k: tuple(v.shape) for k, v in arrays.items()})
    restore_node_and_api()


def restore_node_and_api():
    """the two reference node classes of the "next" rows (SURVEY 8b): API dump + outputs of VRGDGVideoEnhanceRestoreOriginal.restore"""
    import json
    import torch.nn.functional as F
    ns = {"torch": torch, "F": F, "VIDEO_ENHANCE_CONTEXT": "VRGDG_VIDEO_ENHANCE_CONTEXT", "_log": lambda *a, **k: None}
    RH._extract(os.path.join(RH.REFERENCE_ROOT, "VRGDG_VideoEnhanceNodes.py"),
                {"_interpolation", "_resize_batch", "_restore_batch", "VRGDGVideoEnhanceRestoreOriginal"}, ns)
    ns2 = {}
    RH._extract(os.path.join(RH.REFERENCE_ROOT, "VRGDG_StandaloneVideoEnhancerNodes.py"), {"VRGDGStandaloneVideoEnhancer"}, ns2)
    api = {}
    for key, cls in (("VRGDGVideoEnhanceRestoreOriginal", ns["VRGDGVideoEnhanceRestoreOriginal"]), ("VRGDGStandaloneVideoEnhancer", ns2["VRGDGStandaloneVideoEnhancer"])):
        api[key] = {"INPUT_TYPES": json.loads(json.dumps(cls.INPUT_TYPES())), "RETURN_TYPES": list(cls.RETURN_TYPES), "FUNCTION": cls.FUNCTION,
                    "CATEGORY": cls.CATEGORY, "RETURN_NAMES": list(getattr(cls, "RETURN_NAMES", ())), "DESCRIPTION": getattr(cls, "DESCRIPTION", None),
                    "OUTPUT_NODE": bool(getattr(cls, "OUTPUT_NODE", False))}
    display = {"VRGDGVideoEnhanceRestoreOriginal": "Video Enhance - Restore Original Resolution", "VRGDGStandaloneVideoEnhancer": "VRGDG Standalone Video Enhancer"}
    for key, name in display.items():      # check against the reference's own mapping text
        src = open(os.path.join(RH.REFERENCE_ROOT, "VRGDG_VideoEnhanceNodes.py" if "Restore" in key else "VRGDG_StandaloneVideoEnhancerNodes.py"), encoding="utf-8").read()
        assert '"%s": "%s"' % (key, name) in src, key
    with open(os.path.join(HERE, "reference_meta_r2.json"), "w", encoding="utf-8") as fh:
        json.dump({"api": api, "display_names": display}, fh, indent=1, ensure_ascii=True)
    node = ns["VRGDGVideoEnhanceRestoreOriginal"]()
    originals = natural_frames(5, 30, 40, seed=41)
    ltx = natural_frames(4, 24, 32, seed=42)
    out = {"originals": originals, "ltx": ltx}
    cases = []
    for ci, (fit, method, strength) in enumerate((("Stretch to dimensions", "Bicubic (recommended)", 1.0), ("Stretch to dimensions", "Bilinear", 0.4),
                                                  ("Fit with letterbox (preserve all)", "Area", 0.75), ("Crop to fill", "Nearest", 1.0))):
        ctx = {"original_frames": originals, "source_height": 30, "source_width": 40, "frame_count": 5, "fit_mode": fit, "fps": 24.0}
        res = node.restore(ltx, ctx, method, strength)
        out["case%d" % ci] = res[0]
        assert res[1:] == (5, 40, 30, 24.0)
        cases.append([fit, method, strength])
    arrays = {k: v.detach().cpu().numpy() for k, v in out.items()}
    np.savez_compressed(os.path.join(HERE, "restore_node.npz"), **arrays)
    with open(os.path.join(HERE, "restore_node_cases.json"), "w", encoding="utf-8") as fh:
        json.dump(cases, fh)
    print("restore_node", {k: tuple(v.shape) for k, v in arrays.items()})


if __name__ == "__main__":
    main()
