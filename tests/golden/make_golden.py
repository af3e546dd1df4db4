"""Freezes golden input/output vectors by EXECUTING THE REFERENCE'S OWN SOURCE (oracle/ref_harness.py).

Needs a checkout of the reference:   VRGDG_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py
The .npz / .json files it writes are committed; the tests read them and never need the reference.
"""
import hashlib
import json
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ref_harness as RH  # noqa: E402
from helpers import LUTS, natural_frames, save_golden, white_frames  # noqa: E402

warnings.filterwarnings("ignore")
torch.set_num_threads(4)


def save(name, **arrays):
    out = {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in arrays.items()}
    save_golden(name, out, HERE)
    print(name, {k: tuple(v.shape) for k, v in out.items()})


def sha(t):
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()


def main():
    assert RH.available(), "reference tree not found"
    nodes = RH.load_filter_nodes()
    iv = RH.load_iv_adjustments()
    enh = RH.load_enhancer_helpers()
    lvt = RH.load_lut_video_helpers(iv)
    iv.LUTS_DIR = LUTS          # the reference node lists/loads from this module-level folder
    meta = {}

    # ---- grain: FastFilmGrain.apply_grain with the noise it drew -------------------------------------
    x = white_frames(1, 72, 96, seed=11)
    x_odd = white_frames(1, 37, 53, seed=12)
    g = {}
    for tag, img in (("a", x), ("odd", x_odd)):
        torch.manual_seed(123)
        z = torch.randn_like(img)
        torch.manual_seed(123)
        o1 = nodes["FastFilmGrain"]().apply_grain(img, 0.5, 0.5, 0)[0]
        torch.manual_seed(123)
        o2 = nodes["FastFilmGrain"]().apply_grain(img, 0.04, 0.37, 0)[0]
        g.update({f"x_{tag}": img, f"z_{tag}": z, f"out_{tag}_i50_s50": o1, f"out_{tag}_i04_s37": o2})
    save("grain", **g)

    # config 1: 1x512x512, intensity 0.5 — hashes + crop (inputs are regenerated from seeds on the test side)
    x1 = torch.rand(1, 512, 512, 3, generator=torch.Generator().manual_seed(0))
    torch.manual_seed(123)
    z1 = torch.randn_like(x1)
    torch.manual_seed(123)
    o1 = nodes["FastFilmGrain"]().apply_grain(x1, 0.5, 0.5, 4)[0]
    meta["config1"] = {"x_sha256": sha(x1), "z_sha256": sha(z1), "out_sha256": sha(o1)}
    save("config1_crop", out_crop=o1[0, 100:132, 200:232])

    # ---- seeded per-frame grain + the reference's only chain (_apply_effects_batch) --------------------
    frames = torch.full((4, 12, 16, 3), 0.5)
    st = {"sharpen_enabled": False, "grain_enabled": True, "grain_intensity": 0.04, "saturation_mix": 0.5, "seed": 42, "use_gpu": False}
    whole = enh["_apply_effects_batch"](frames, st, 100)
    zs = []
    for off in range(4):
        gen = torch.Generator(device="cpu")
        gen.manual_seed((42 + 100 + off) & 0x7FFFFFFF)
        zs.append(torch.randn((12, 16, 3), generator=gen))
    xe = natural_frames(2, 40, 88, seed=5)
    st2 = dict(st, sharpen_enabled=True, sharpen_strength=0.8)
    eff = enh["_apply_effects_batch"](xe, st2, 7)
    ze = []
    for off in range(2):
        gen = torch.Generator(device="cpu")
        gen.manual_seed((42 + 7 + off) & 0x7FFFFFFF)
        ze.append(torch.randn((40, 88, 3), generator=gen))
    sharp_only = enh["_apply_effects_batch"](xe, dict(st2, grain_enabled=False), 7)
    save("effects", frames=frames, whole=whole, z=torch.stack(zs), xe=xe, eff=eff, ze=torch.stack(ze), sharp_only=sharp_only)

    # ---- 3x3 stencils, both reference paths ----------------------------------------------------------------
    xs = natural_frames(1, 72, 96, seed=3)
    xs[0, :4, :4] = white_frames(1, 4, 4, seed=4)[0]
    s = {"x": xs, "x_odd": x_odd, "x_tiny": white_frames(1, 2, 3, seed=6), "x_one": white_frames(1, 1, 1, seed=7)}
    for key, cls, fn in (("unsharp", "FastUnsharpSharpen", "apply_unsharp"), ("laplacian", "FastLaplacianSharpen", "apply_laplacian"),
                         ("sobel", "FastSobelSharpen", "apply_sobel")):
        node = nodes[cls]()
        s[f"{key}_np"] = getattr(node, fn)(xs, 0.5, False)[0]
        s[f"{key}_torch"] = getattr(node, fn)(xs, 0.5, True)[0]
        s[f"{key}_np_odd"] = getattr(node, fn)(x_odd, 1.3, False)[0]
        s[f"{key}_np_tiny"] = getattr(node, fn)(s["x_tiny"], 0.7, False)[0]
        s[f"{key}_np_one"] = getattr(node, fn)(s["x_one"], 0.7, False)[0]
    s["unsharp_np_s10"] = nodes["FastUnsharpSharpen"]().apply_unsharp(xs, 10.0, False)[0]
    save("stencil", **s)

    # ---- 3D LUT --------------------------------------------------------------------------------------------
    xl = white_frames(1, 72, 96, seed=21)
    xl[0, 0, 0] = torch.tensor([1.0, 0.0, 1.0])
    xl[0, 0, 1] = torch.tensor([0.0, 0.0, 0.0])
    xl[0, 0, 2] = torch.tensor([1.0, 1.0, 1.0])
    xl[0, 0, 3] = torch.tensor([0.5, 0.25, 0.75])           # exact grid nodes for S=33 / 17 / 25
    xl[0, 0, 4] = torch.tensor([1.0 / 32.0, 31.0 / 32.0, 0.5])
    xn = natural_frames(1, 72, 96, seed=22)
    lut_out = {"x": xl, "xn": xn}
    node = iv.VRGDG_LUTS()
    for fname in sorted(os.listdir(LUTS)):
        if not fname.endswith(".cube"):
            continue
        key = fname.split(".")[0].replace(" ", "_")
        lut_out[f"{key}__s10"] = node.apply_lut(xl, fname, "cpu", 10.0)[0]
        lut_out[f"{key}__s3p5"] = node.apply_lut(xl, fname, "cpu", 3.5)[0]
        lut_out[f"{key}__nat"] = node.apply_lut(xn, fname, "cpu", 10.0)[0]
    v33 = "B200 Vintage 33.cube"
    lut_out["v33_fp16"] = node.apply_lut(xl.half(), v33, "cpu", 10.0)[0]
    lut_out["v33_fp16_s3p5"] = node.apply_lut(xl.half(), v33, "cpu", 3.5)[0]
    x4 = torch.cat([xl, white_frames(1, 72, 96, seed=23)[..., :1]], dim=-1)
    lut_out["x4"] = x4
    lut_out["v33_rgba"] = node.apply_lut(x4, v33, "cpu", 10.0)[0]
    lut_out["v33_rgba_s3p5"] = node.apply_lut(x4, v33, "cpu", 3.5)[0]
    # non-unit domain, tiny table written by the reference's own writer then edited
    dom_path = os.path.join(HERE, "domain_5.cube")
    tbl = torch.rand(5, 5, 5, 3, generator=torch.Generator().manual_seed(31))
    with open(dom_path, "w", encoding="utf-8") as fh:
        fh.write("# non-unit domain fixture\nLUT_3D_SIZE 5\nDOMAIN_MIN -0.1 0.0 0.05\nDOMAIN_MAX 1.2 1.1 0.9\n")
        for row in tbl.reshape(-1, 3).tolist():
            fh.write("%.6f %.6f %.6f\n" % tuple(row))
    dom = iv.VRGDG_LUTS._parse_cube_file(dom_path)
    lut_out["domain5_s10"] = iv.VRGDG_LUTS._apply_cube_lut(xl, dom["lut"], dom["domain_min"], dom["domain_max"])
    lut_out["tensor_fn_s7"] = lvt["_apply_lut_tensor"](xl, v33, 7.0, "cpu")
    save("lut", **lut_out)

    # ---- palette LUT builder ----------------------------------------------------------------------------------
    save("palette", three=iv._build_palette_lut("#0b1d51, #1f6aa5, #f3d27a", 9), one=iv._build_palette_lut("teal", 8),
         names=iv._build_palette_lut("black, #f80, white, pink", 11))

    # ---- colour match (kornia restatement injected: parity unpinned for the Lab conversion) ---------------------
    xc = natural_frames(2, 72, 96, seed=41)
    xc[1] = (xc[1] * 0.7 + 0.1).clamp(0, 1)
    ref = natural_frames(1, 40, 56, seed=42) * torch.tensor([0.9, 0.8, 1.0])
    cm = nodes["ColorMatchToReference"]()
    save("colormatch", x=xc, ref=ref, out_t100=cm.match_color(xc, ref, 1.0, 1)[0], out_t60=cm.match_color(xc, ref, 0.6, 2)[0])

    # ---- chains: reference nodes applied one after another -----------------------------------------------------
    xch = natural_frames(2, 72, 96, seed=51)
    torch.manual_seed(7)
    zch = torch.randn_like(xch)
    torch.manual_seed(7)
    a = nodes["FastFilmGrain"]().apply_grain(xch, 0.04, 0.5, 0)[0]
    b = node.apply_lut(a, v33, "cpu", 10.0)[0]
    c = nodes["FastUnsharpSharpen"]().apply_unsharp(b, 0.5, False)[0]
    refc = natural_frames(1, 48, 64, seed=52)
    a2 = cm.match_color(a, refc, 1.0, 1)[0]
    b2 = node.apply_lut(a2, v33, "cpu", 10.0)[0]
    c2 = nodes["FastUnsharpSharpen"]().apply_unsharp(b2, 0.5, False)[0]
    b3 = node.apply_lut(a, v33, "cpu", 6.0)[0]
    c3 = nodes["FastSobelSharpen"]().apply_sobel(b3, 0.3, False)[0]
    save("chain", x=xch, z=zch, ref=refc, grain_lut_unsharp=c, grain_cm_lut_unsharp=c2, grain_lut60_sobel=c3)

    # ---- uint8 BGR wire format (cv2 present in the container) ------------------------------------------------------
    import ast
    ns = {}
    with open(os.path.join(RH.REFERENCE_ROOT, "VRGDG_LUTVideoTools.py"), encoding="utf-8") as fh:
        tree = ast.parse(fh.read())
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in {"_frames_to_tensor", "_tensor_to_frames"}]
    exec(compile(ast.Module(body=body, type_ignores=[]), "VRGDG_LUTVideoTools.py", "exec"), ns)
    u8 = torch.randint(0, 256, (3, 9, 14, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(61)).numpy()
    as_t = ns["_frames_to_tensor"](list(u8))
    back_in = white_frames(3, 9, 14, seed=62) * 1.2 - 0.1
    back = np.stack(ns["_tensor_to_frames"](back_in), axis=0)
    save("u8", bgr=u8, rgb_float=as_t, float_in=back_in, bgr_out=back)

    # ---- uint8 wire format through the whole chain: decode -> grain -> LUT -> unsharp -> encode (bytes in, bytes out) ----
    xu = (natural_frames(2, 72, 96, seed=71) * 255.0).round().clamp(0, 255).to(torch.uint8).numpy()[..., ::-1].copy()   # BGR bytes
    ft = ns["_frames_to_tensor"](list(xu))
    torch.manual_seed(9)
    zu = torch.randn_like(ft)
    torch.manual_seed(9)
    ga = nodes["FastFilmGrain"]().apply_grain(ft, 0.04, 0.5, 0)[0]
    gb = node.apply_lut(ga, v33, "cpu", 10.0)[0]
    gc = nodes["FastUnsharpSharpen"]().apply_unsharp(gb, 0.5, False)[0]
    save("u8chain", bgr_in=xu, z=zu, grain_only=np.stack(ns["_tensor_to_frames"](ga)), lut_only=np.stack(ns["_tensor_to_frames"](node.apply_lut(ft, v33, "cpu", 10.0)[0])),
         unsharp_only=np.stack(ns["_tensor_to_frames"](nodes["FastUnsharpSharpen"]().apply_unsharp(ft, 0.5, False)[0])),
         grain_lut_unsharp=np.stack(ns["_tensor_to_frames"](gc)))

    # ---- adjust (_apply_adjust_tensor) --------------------------------------------------------------------------------
    xa = natural_frames(2, 72, 96, seed=81) * 1.1 - 0.05                      # some values outside [0,1]: the function clamps first
    adj = {"x": xa}
    ADJ_CASES = {
        "pointwise": {"temperature": 30, "tint": -20, "exposure": 25, "contrast": 40, "saturation": -35, "highlights": 50, "shadows": -40, "whites": 20, "blacks": -60},
        "fade_vignette": {"fade": 40, "vignette": 70, "exposure": -10},
        "sharpen": {"sharpen": 60, "contrast": 10},
        "clarity": {"clarity": 80, "saturation": 20},
        "everything": {"temperature": -45, "tint": 15, "exposure": 12, "contrast": -20, "saturation": 30, "highlights": -30, "shadows": 35, "whites": -15,
                       "blacks": 25, "sharpen": 35, "clarity": -60, "vignette": 50, "fade": 20},
        "disabled": {"enabled": False, "exposure": 50},
    }
    for name, st in ADJ_CASES.items():
        adj[name] = lvt["_apply_adjust_tensor"](xa, st, "cpu")
    adj["tiny_5x7"] = lvt["_apply_adjust_tensor"](xa[:, :5, :7].contiguous(), ADJ_CASES["everything"], "cpu")    # blur kernel shrinks to 5
    save("adjust", **adj)
    meta["adjust_cases"] = ADJ_CASES

    # ---- resize / restore (VRGDG_VideoEnhanceNodes.py) -------------------------------------------------------------------------
    ve = RH.load_video_enhance_helpers()
    xr = natural_frames(2, 54, 96, seed=85)
    rz = {"x": xr}
    RESIZE_CASES = []
    for method in ("Nearest", "Bilinear", "Bicubic (recommended)", "Area"):
        for fit, (tw, th) in (("Stretch to dimensions", (160, 72)), ("Crop to fill", (64, 64)), ("Fit with letterbox (preserve all)", (80, 80)),
                              ("Stretch to dimensions", (40, 30))):
            key = "%s|%s|%dx%d" % (method.split()[0], fit.split()[0], tw, th)
            RESIZE_CASES.append([key, method, fit, tw, th])
            rz[key] = ve["_resize_batch"](xr, tw, th, fit, method)
    up = ve["_resize_batch"](xr, 80, 80, "Fit with letterbox (preserve all)", "Bicubic (recommended)")
    rz["restore_letterbox"] = ve["_restore_batch"](up, 96, 54, "Fit with letterbox (preserve all)", "Bicubic (recommended)")
    rz["restore_stretch"] = ve["_restore_batch"](up, 96, 54, "Stretch to dimensions", "Bilinear")
    save("resize", **rz)
    meta["resize_cases"] = RESIZE_CASES

    # ---- the enhancer's Lanczos4 resize: cv2 itself is the reference (EnhancerNodes.py:213-230) ---------------------------------------
    import cv2
    se = RH.load_enhancer_helpers()
    rngl = np.random.default_rng(77)
    lz = {"cv2_version": np.array(cv2.__version__)}
    LANCZOS_CASES = []
    nat = (natural_frames(1, 90, 160, seed=86)[0].numpy()[..., ::-1] * 255).astype(np.uint8)
    for name, img, (ow, oh) in (("noise_up", rngl.integers(0, 256, (37, 53, 3), dtype=np.uint8), (106, 74)),
                                ("noise_down", rngl.integers(0, 256, (37, 53, 3), dtype=np.uint8), (31, 20)),
                                ("noise_odd", rngl.integers(0, 256, (48, 64, 3), dtype=np.uint8), (100, 61)),
                                ("tiny", rngl.integers(0, 256, (9, 7, 3), dtype=np.uint8), (3, 30)),
                                ("float_sum_317", rngl.integers(0, 256, (64, 317, 3), dtype=np.uint8), (2252, 64)),   # x+3 rounded in fp32 matters here
                                ("float_sum_500", rngl.integers(0, 256, (64, 500, 3), dtype=np.uint8), (378, 64)),
                                ("extremes", (rngl.integers(0, 2, (40, 40, 3)) * 255).astype(np.uint8), (90, 70)),
                                ("natural_up", nat, (320, 180)), ("natural_down", nat, (96, 54)), ("same", nat, (160, 90))):
        lz[name + "_in"] = img
        lz[name] = se["_resize_frames"]([img], ow, oh)[0]
        LANCZOS_CASES.append([name, ow, oh])
    save("lanczos", **lz)
    meta["lanczos_cases"] = LANCZOS_CASES

    # ---- node API surface ---------------------------------------------------------------------------------------------
    api = {}
    classes = dict(nodes)
    classes.update({"VRGDG_LUTS": iv.VRGDG_LUTS, "VRGDG_MakeLUT": iv.VRGDG_MakeLUT})
    for key in ("FastFilmGrain", "ColorMatchToReference", "FastUnsharpSharpen", "FastLaplacianSharpen", "FastSobelSharpen", "VRGDG_LUTS", "VRGDG_MakeLUT"):
        cls = classes[key]
        it = cls.INPUT_TYPES()
        if key == "VRGDG_LUTS":
            it["required"]["lut_name"] = ["<lut files>"]
        api[key] = {"INPUT_TYPES": json.loads(json.dumps(it)), "RETURN_TYPES": list(cls.RETURN_TYPES), "FUNCTION": cls.FUNCTION,
                    "CATEGORY": cls.CATEGORY, "RETURN_NAMES": list(getattr(cls, "RETURN_NAMES", ())), "DESCRIPTION": getattr(cls, "DESCRIPTION", None)}
    import re
    src = open(os.path.join(RH.REFERENCE_ROOT, "nodes.py"), encoding="utf-8").read()
    names = {k: re.search(r'"%s":\s*"(.*?)"' % k, src).group(1) for k in list(api)[:5]}
    names.update(iv.NODE_DISPLAY_NAME_MAPPINGS)
    meta["display_names"] = names
    meta["api"] = api
    meta["auto_batch"] = {"1280x720": enh["_auto_batch_size"](1280, 720), "1920x1080": enh["_auto_batch_size"](1920, 1080),
                          "2560x1440": enh["_auto_batch_size"](2560, 1440), "3072x1728": enh["_auto_batch_size"](3072, 1728),
                          "3840x2160": enh["_auto_batch_size"](3840, 2160)}
    meta["torch"] = torch.__version__
    meta["numpy"] = np.__version__
    with open(os.path.join(HERE, "reference_meta.json"), "w", encoding="utf-8") as fh:
        json.dump(meta, fh, indent=1, ensure_ascii=True)
    print("reference_meta.json written")


if __name__ == "__main__":
    main()
