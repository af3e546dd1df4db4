"""Pins oracle/vrgdg_oracle.py: (1) against the golden vectors frozen from the reference's own source
(tests/golden/make_golden.py), bit for bit; (2) where a checkout of the reference is found (oracle/ref_harness.py), against
the live reference code on fresh inputs.  CPU only."""
import json
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, LUTS, load_golden, natural_frames, t, white_frames


def test_grain_restatement_bit_exact(oracle):
    g = load_golden("grain")
    for tag in ("a", "odd"):
        x, z = t(g[f"x_{tag}"]), t(g[f"z_{tag}"])
        assert torch.equal(oracle.film_grain(x, 0.5, 0.5, 0, noise=z), t(g[f"out_{tag}_i50_s50"]))
        assert torch.equal(oracle.film_grain(x, 0.04, 0.37, 0, noise=z), t(g[f"out_{tag}_i04_s37"]))
    # and with its own RNG draw (same torch CPU generator as the reference used)
    torch.manual_seed(123)
    z = torch.randn_like(t(g["x_a"]))
    if torch.equal(z, t(g["z_a"])):
        torch.manual_seed(123)
        assert torch.equal(oracle.film_grain(t(g["x_a"]), 0.5, 0.5, 0), t(g["out_a_i50_s50"]))


def test_effects_and_seeded_grain_restatement(oracle):
    g = load_golden("effects")
    st = {"sharpen_enabled": False, "grain_enabled": True, "grain_intensity": 0.04, "saturation_mix": 0.5, "seed": 42}
    z = oracle.seeded_grain_noise((12, 16, 3), 42, 100, 4)
    if torch.equal(z, t(g["z"])):
        assert torch.equal(oracle.effects_batch(t(g["frames"]), st, 100), t(g["whole"]))
        # the reference's own invariant: batch boundaries do not matter
        split = torch.cat([oracle.effects_batch(t(g["frames"])[:2], st, 100), oracle.effects_batch(t(g["frames"])[2:], st, 102)])
        assert torch.equal(split, t(g["whole"]))
        st2 = dict(st, sharpen_enabled=True, sharpen_strength=0.8)
        assert torch.equal(oracle.effects_batch(t(g["xe"]), st2, 7), t(g["eff"]))
    assert torch.equal(oracle.effects_batch(t(g["xe"]), {"sharpen_enabled": True, "sharpen_strength": 0.8}, 7), t(g["sharp_only"]))


def test_stencil_restatement_bit_exact(oracle):
    g = load_golden("stencil")
    fns = {"unsharp": (oracle.unsharp_numpy, oracle.unsharp_torch), "laplacian": (oracle.laplacian_numpy, oracle.laplacian_torch),
           "sobel": (oracle.sobel_numpy, oracle.sobel_torch)}
    for key, (f_np, f_t) in fns.items():
        assert torch.equal(f_np(t(g["x"]), 0.5), t(g[f"{key}_np"]))
        assert torch.equal(f_t(t(g["x"]), 0.5), t(g[f"{key}_torch"]))
        assert torch.equal(f_np(t(g["x_odd"]), 1.3), t(g[f"{key}_np_odd"]))
        assert torch.equal(f_np(t(g["x_tiny"]), 0.7), t(g[f"{key}_np_tiny"]))
        assert torch.equal(f_np(t(g["x_one"]), 0.7), t(g[f"{key}_np_one"]))
    assert torch.equal(oracle.unsharp_numpy(t(g["x"]), 10.0), t(g["unsharp_np_s10"]))
    # SURVEY D5 facts: interior of both unsharp paths identical, laplacian paths differ in sign
    a, b = t(g["unsharp_np"]), t(g["unsharp_torch"])
    assert torch.equal(a[:, 1:-1, 1:-1], b[:, 1:-1, 1:-1]) and not torch.equal(a, b)
    assert float((t(g["laplacian_np"]) - t(g["laplacian_torch"])).abs().max()) > 0.01


def test_lut_restatement_bit_exact(oracle):
    g = load_golden("lut")
    x, xn = t(g["x"]), t(g["xn"])
    for fname in sorted(os.listdir(LUTS)):
        if not fname.endswith(".cube"):
            continue
        key = fname.split(".")[0].replace(" ", "_")
        data = oracle.parse_cube(os.path.join(LUTS, fname))
        assert torch.equal(oracle.apply_lut(x, data, 10.0), t(g[f"{key}__s10"]))
        assert torch.equal(oracle.apply_lut(x, data, 3.5), t(g[f"{key}__s3p5"]))
        assert torch.equal(oracle.apply_lut(xn, data, 10.0), t(g[f"{key}__nat"]))
    v33 = oracle.parse_cube(os.path.join(LUTS, "B200 Vintage 33.cube"))
    assert torch.equal(oracle.apply_lut(x.half(), v33, 10.0), t(g["v33_fp16"]))
    assert torch.equal(oracle.apply_lut(x.half(), v33, 3.5), t(g["v33_fp16_s3p5"]))
    assert torch.equal(oracle.apply_lut(t(g["x4"]), v33, 10.0), t(g["v33_rgba"]))
    assert torch.equal(oracle.apply_lut(t(g["x4"]), v33, 3.5), t(g["v33_rgba_s3p5"]))
    assert torch.equal(oracle.apply_lut(x, v33, 7.0), t(g["tensor_fn_s7"]))
    dom = oracle.parse_cube(os.path.join(GOLDEN, "domain_5.cube"))
    assert dom["domain_min"].tolist() == pytest.approx([-0.1, 0.0, 0.05]) and dom["size"] == 5
    assert torch.equal(oracle.apply_cube_lut(x, dom["lut"], dom["domain_min"], dom["domain_max"]), t(g["domain5_s10"]))
    assert oracle.apply_lut(x, v33, 0.0) is x


def test_palette_restatement_bit_exact(oracle):
    g = load_golden("palette")
    hexes = lambda *cs: np.array([[int(c[i:i + 2], 16) / 255.0 for i in (0, 2, 4)] for c in cs], dtype=np.float32)
    assert torch.equal(oracle.palette_lut(hexes("0b1d51", "1f6aa5", "f3d27a"), 9), t(g["three"]))
    assert torch.equal(oracle.palette_lut(hexes("008080"), 8), t(g["one"]))


def test_colormatch_and_chain_restatement(oracle):
    g = load_golden("colormatch")
    assert torch.equal(oracle.color_match(t(g["x"]), t(g["ref"]), 1.0, 1), t(g["out_t100"]))
    assert torch.equal(oracle.color_match(t(g["x"]), t(g["ref"]), 0.6, 2), t(g["out_t60"]))
    c = load_golden("chain")
    v33 = oracle.parse_cube(os.path.join(LUTS, "B200 Vintage 33.cube"))
    assert torch.equal(oracle.chain_grain_lut_unsharp(t(c["x"]), t(c["z"]), 0.04, 0.5, v33, 10.0, 0.5), t(c["grain_lut_unsharp"]))
    assert torch.equal(oracle.chain_full(t(c["x"]), t(c["z"]), 0.04, 0.5, t(c["ref"]), 1.0, v33, 10.0, 0.5), t(c["grain_cm_lut_unsharp"]))


def test_adjust_restatement_bit_exact(oracle):
    g = load_golden("adjust")
    with open(os.path.join(GOLDEN, "reference_meta.json"), encoding="utf-8") as fh:
        cases = json.load(fh)["adjust_cases"]
    assert set(cases) >= {"pointwise", "fade_vignette", "sharpen", "clarity", "everything", "disabled"}
    for name, st in cases.items():
        assert torch.equal(oracle.adjust(t(g["x"]), st), t(g[name])), name
    assert torch.equal(oracle.adjust(t(g["x"])[:, :5, :7].contiguous(), cases["everything"]), t(g["tiny_5x7"]))
    assert oracle.normalize_adjust_settings({"sharpen": -3, "fade": 1e9, "tint": "x", "enabled": False}) == dict(
        oracle.normalize_adjust_settings({}), enabled=False, fade=100.0)


def test_resize_restatement_bit_exact(oracle):
    """_resize_batch / _restore_batch (VRGDG_VideoEnhanceNodes.py:54-106): every interpolation x fit mode, torch on both sides."""
    g = load_golden("resize")
    with open(os.path.join(GOLDEN, "reference_meta.json"), encoding="utf-8") as fh:
        cases = json.load(fh)["resize_cases"]
    assert len(cases) == 16 and {c[1] for c in cases} == set(oracle.INTERPOLATIONS)
    for key, method, fit, tw, th in cases:
        assert torch.equal(oracle.resize_batch(t(g["x"]), tw, th, fit, method), t(g[key])), key
    up = t(g["Bicubic|Fit|80x80"])
    assert torch.equal(oracle.restore_batch(up, 96, 54, "Fit with letterbox (preserve all)", "Bicubic (recommended)"), t(g["restore_letterbox"]))
    assert torch.equal(oracle.restore_batch(up, 96, 54, "Stretch to dimensions", "Bilinear"), t(g["restore_stretch"]))
    with pytest.raises(ValueError):
        oracle.resize_batch(t(g["x"])[0], 8, 8, "Stretch to dimensions", "Nearest")


def test_lanczos4_restatement_bit_exact_vs_cv2_fixtures(oracle):
    """_resize_frames (EnhancerNodes.py:213-230): the fixtures are outputs of cv2.resize itself (opencv version in the file)."""
    g = load_golden("lanczos")
    with open(os.path.join(GOLDEN, "reference_meta.json"), encoding="utf-8") as fh:
        cases = json.load(fh)["lanczos_cases"]
    assert {c[0] for c in cases} >= {"noise_up", "noise_down", "tiny", "float_sum_317", "float_sum_500", "extremes", "natural_up", "same"}
    for name, ow, oh in cases:
        src = g[name + "_in"]
        out = oracle.resize_frames([src], ow, oh)[0]
        assert np.array_equal(out, g[name]), name
    assert oracle.resize_frames([g["same_in"]], 160, 90)[0] is g["same_in"]
    try:
        import cv2
    except ImportError:
        return
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (45, 80, 3), dtype=np.uint8)
    for ow, oh in ((120, 68), (33, 19), (80, 90)):
        assert np.array_equal(oracle.resize_lanczos4_u8(img, ow, oh), cv2.resize(img, (ow, oh), interpolation=cv2.INTER_LANCZOS4))


def test_u8_restatement(oracle):
    g = load_golden("u8")
    assert torch.equal(oracle.frames_to_tensor(g["bgr"]), t(g["rgb_float"]))
    assert np.array_equal(oracle.tensor_to_frames(t(g["float_in"])), g["bgr_out"])


def test_lab_restatement_against_independent_float64(oracle):
    """kornia is absent (parity unpinned): at least the restated formulas agree with a float64 textbook evaluation and
    round-trip."""
    x = white_frames(1, 64, 64, seed=5)
    lab = oracle.rgb_to_lab(x.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
    ref = oracle.lab_reference_f64(x.numpy())
    assert np.abs(lab.numpy() - ref).max() < 2e-4          # fp32 vs fp64 on a 0..100 scale
    back = oracle.lab_to_rgb(lab.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
    assert float((back - x).abs().max()) < 2e-5
    white = oracle.rgb_to_lab(torch.ones(1, 3, 1, 1))
    assert abs(float(white[0, 0]) - 100.0) < 1e-3 and float(white[0, 1:].abs().max()) < 2e-2


def test_golden_files_stay_small_and_reassemble(tmp_path):
    from helpers import GOLDEN_FILE_BYTES, save_golden
    for f in os.listdir(GOLDEN):
        assert os.path.getsize(os.path.join(GOLDEN, f)) <= GOLDEN_FILE_BYTES, f
    arrays = {"a%d" % i: np.random.default_rng(i).random((100, 100)) for i in range(5)}     # 5 x 80 kB that does not compress
    assert len(save_golden("split", arrays, str(tmp_path))) == 1 and os.listdir(tmp_path) == ["split.npz"]
    paths = save_golden("split", arrays, str(tmp_path), limit=200000)
    assert sorted(os.listdir(tmp_path)) == ["split.npz", "split_part2.npz", "split_part3.npz"] and all(os.path.getsize(p) <= 200000 for p in paths)
    back = load_golden("split", str(tmp_path))
    assert set(back) == set(arrays) and all(np.array_equal(back[k], arrays[k]) for k in arrays)
    save_golden("split", arrays, str(tmp_path))                                          # a later, smaller save leaves no stale parts
    assert os.listdir(tmp_path) == ["split.npz"]


def test_golden_meta_consistent():
    with open(os.path.join(GOLDEN, "reference_meta.json"), encoding="utf-8") as fh:
        meta = json.load(fh)
    assert set(meta["api"]) == {"FastFilmGrain", "ColorMatchToReference", "FastUnsharpSharpen", "FastLaplacianSharpen", "FastSobelSharpen",
                                "VRGDG_LUTS", "VRGDG_MakeLUT"}
    assert len(meta["config1"]["out_sha256"]) == 64


# ---- live reference (needs a checkout of the reference, which this repository does not contain) -------------------------
def _harness():
    import ref_harness
    if not ref_harness.available():
        pytest.skip("no checkout of the original comfyui-vrgamedevgirl node pack found (set VRGDG_REFERENCE_ROOT)")
    return ref_harness


def test_live_reference_filters_match_oracle(oracle):
    rh = _harness()
    import warnings
    warnings.filterwarnings("ignore")
    nodes = rh.load_filter_nodes()
    x = natural_frames(3, 45, 67, seed=99)
    torch.manual_seed(5)
    a = nodes["FastFilmGrain"]().apply_grain(x, 0.1, 0.3, 2)[0]
    torch.manual_seed(5)
    assert torch.equal(a, oracle.film_grain(x, 0.1, 0.3, 2))
    for s in (0.0, 0.5, 2.0):
        assert torch.equal(nodes["FastUnsharpSharpen"]().apply_unsharp(x, s, False)[0], oracle.unsharp_numpy(x, s))
        assert torch.equal(nodes["FastUnsharpSharpen"]().apply_unsharp(x, s, True)[0], oracle.unsharp_torch(x, s))
        assert torch.equal(nodes["FastLaplacianSharpen"]().apply_laplacian(x, s, False)[0], oracle.laplacian_numpy(x, s))
        assert torch.equal(nodes["FastLaplacianSharpen"]().apply_laplacian(x, s, True)[0], oracle.laplacian_torch(x, s))
        assert torch.equal(nodes["FastSobelSharpen"]().apply_sobel(x, s, False)[0], oracle.sobel_numpy(x, s))
        assert torch.equal(nodes["FastSobelSharpen"]().apply_sobel(x, s, True)[0], oracle.sobel_torch(x, s))
    ref = natural_frames(1, 30, 41, seed=98)
    assert torch.equal(nodes["ColorMatchToReference"]().match_color(x, ref, 0.7, 2)[0], oracle.color_match(x, ref, 0.7, 2))
    enh = rh.load_enhancer_helpers()
    st = {"sharpen_enabled": True, "sharpen_strength": 0.4, "grain_enabled": True, "grain_intensity": 0.05, "saturation_mix": 0.2, "seed": 9, "use_gpu": False}
    assert torch.equal(enh["_apply_effects_batch"](x, st, 3), oracle.effects_batch(x, st, 3))
    lvt = rh.load_lut_video_helpers()
    assert torch.equal(lvt["_apply_film_grain_tensor"](x, 0.07, 0.4, "cpu", 11), oracle.film_grain_tensor(x, 0.07, 0.4, 11))
    st = {"temperature": 12, "tint": 7, "exposure": -8, "contrast": 22, "saturation": -11, "shadows": 14, "blacks": -9, "sharpen": 25, "clarity": 33, "fade": 5, "vignette": 44}
    assert torch.equal(lvt["_apply_adjust_tensor"](x * 1.1 - 0.05, st, "cpu"), oracle.adjust(x * 1.1 - 0.05, st))
    assert lvt["_normalize_adjust_settings"]({"fade": 500, "clarity": "no"}) == oracle.normalize_adjust_settings({"fade": 500, "clarity": "no"})


def test_live_reference_parses_all_its_own_luts_like_the_oracle(oracle, pkg):
    rh = _harness()
    iv = rh.load_iv_adjustments()
    lut_dir = os.path.join(rh.REFERENCE_ROOT, "LUTS")
    names = sorted(n for n in os.listdir(lut_dir) if n.endswith(".cube"))
    assert len(names) >= 40
    x = white_frames(1, 16, 16, seed=1)
    for n in names[::4] + ["Vintage Color.cube"]:          # every 4th (sizes 25/32/33/64/65) keeps this under a minute
        a = iv.VRGDG_LUTS._parse_cube_file(os.path.join(lut_dir, n))
        b = oracle.parse_cube(os.path.join(lut_dir, n))
        c = pkg.VRGDG_LUTS._parse_cube_file(os.path.join(lut_dir, n))
        for other in (b, c):
            assert a["size"] == other["size"] and torch.equal(a["lut"], other["lut"])
            assert torch.equal(a["domain_min"], other["domain_min"]) and torch.equal(a["domain_max"], other["domain_max"])
        assert torch.equal(iv.VRGDG_LUTS._apply_cube_lut(x, a["lut"], a["domain_min"], a["domain_max"]),
                           oracle.apply_cube_lut(x, b["lut"], b["domain_min"], b["domain_max"]))
