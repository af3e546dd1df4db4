"""CPU oracle for the post-processing hot path — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference` legs may import this
module; the product (comfyui-vrgamedevgirl_b200/) never does and has no CPU execution path.

Each function restates, with the same torch / numpy calls in the same order, what one reference function
computes (citations are file:line into the reference tree), so that on a CPU it produces bit-identical
tensors.  Pinning: tests/golden/*.npz were produced by executing the reference's own source
(oracle/ref_harness.py, AST-extracted exactly like the reference's tests do) and
tests/test_oracle_golden.py checks this restatement against them; where a checkout of the reference is found
(oracle/ref_harness.py: VRGDG_REFERENCE_ROOT) the same test also compares against the live reference code.

Parity status
  * grain / unsharp / laplacian / sobel / 3D LUT / cube parser / palette LUT / u8 codecs: PINNED by the
    reference's source.
  * kornia.color.rgb_to_lab / lab_to_rgb (nodes.py:98,108,115): kornia is an unpinned, un-vendored
    dependency (requirements.txt:1) that is not installed here -> formulas restated from the published
    kornia implementation; "parity unpinned" for that sub-step (cross-checked against an independent float64
    CIE evaluation in tests/test_oracle_golden.py).
"""
import os

import math

import numpy as np
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------------------------------
# film grain
# --------------------------------------------------------------------------------------------------
def grain_mix(noise, saturation_mix):
    """nodes.py:53-57 (same lines in VRGDG_LUTVideoTools.py:273-276): scale R/B, mix with the G plane."""
    g = noise.clone()
    g[..., 0] *= 2.0
    g[..., 2] *= 3.0
    gray = g[..., 1].unsqueeze(-1).repeat(*([1] * (g.ndim - 1)), 3)
    return saturation_mix * g + (1.0 - saturation_mix) * gray


def film_grain(images, grain_intensity, saturation_mix, batch_size=4, noise=None):
    """FastFilmGrain.apply_grain, nodes.py:41-66 (CPU device).  `noise` (same shape) replaces randn_like."""
    step = batch_size if batch_size > 0 else images.shape[0]
    chunks = []
    for i in range(0, images.shape[0], step):
        batch = images[i:i + step]
        z = torch.randn_like(batch) if noise is None else noise[i:i + step]
        mixed = grain_mix(z, saturation_mix)
        chunks.append((batch + mixed * grain_intensity).clamp(0.0, 1.0))
    return torch.cat(chunks, dim=0)


def film_grain_tensor(image_tensor, grain_intensity=0.04, saturation_mix=0.5, seed=None):
    """_apply_film_grain_tensor, VRGDG_LUTVideoTools.py:262-277 (device="cpu")."""
    intensity = max(0.0, min(1.0, float(grain_intensity)))
    saturation = max(0.0, min(1.0, float(saturation_mix)))
    gen = None
    if seed not in (None, ""):
        gen = torch.Generator(device=image_tensor.device)
        gen.manual_seed(int(seed))
    z = torch.randn(image_tensor.shape, dtype=image_tensor.dtype, device=image_tensor.device, generator=gen)
    return (image_tensor + grain_mix(z, saturation) * intensity).clamp(0.0, 1.0)


def seeded_grain_noise(shape_hw3, seed, frame_start, count, dtype=torch.float32):
    """the per-frame generators of _apply_seeded_grain, VRGDG_StandaloneVideoEnhancerNodes.py:265-269."""
    frames = []
    for offset in range(count):
        gen = torch.Generator(device="cpu")
        gen.manual_seed((int(seed) + int(frame_start) + offset) & 0x7FFFFFFF)
        frames.append(torch.randn(shape_hw3, generator=gen, device="cpu", dtype=dtype))
    return torch.stack(frames, dim=0)


def seeded_grain(images, intensity, saturation_mix, seed, frame_start):
    """_apply_seeded_grain, VRGDG_StandaloneVideoEnhancerNodes.py:261-275."""
    if intensity <= 0:
        return images
    z = seeded_grain_noise(tuple(images.shape[1:]), seed, frame_start, images.shape[0], images.dtype)
    mixed = torch.stack([grain_mix(f, saturation_mix) for f in z], dim=0)
    return (images + mixed * intensity).clamp(0.0, 1.0)


# --------------------------------------------------------------------------------------------------
# 3x3 stencils
# --------------------------------------------------------------------------------------------------
def _edge_padded(images):
    img = images.contiguous().numpy()
    return img, np.pad(img, ((0, 0), (1, 1), (1, 1), (0, 0)), mode="edge")


def unsharp_numpy(images, strength):
    """FastUnsharpSharpen CPU path nodes.py:182-209 == _apply_unsharp numpy path EnhancerNodes.py:241-258."""
    img, p = _edge_padded(images)
    blur = (p[:, 0:-2, 0:-2] + p[:, 0:-2, 1:-1] + p[:, 0:-2, 2:] +
            p[:, 1:-1, 0:-2] + p[:, 1:-1, 1:-1] + p[:, 1:-1, 2:] +
            p[:, 2:, 0:-2] + p[:, 2:, 1:-1] + p[:, 2:, 2:]) / 9.0
    out = img + strength * (img - blur)
    np.clip(out, 0.0, 1.0, out=out)
    return torch.from_numpy(out)


def unsharp_torch(images, strength):
    """use_gpu=True path (device stubbed to CPU): nodes.py:166-177, EnhancerNodes.py:236-239."""
    x = images.permute(0, 3, 1, 2)
    blur = F.avg_pool2d(x, kernel_size=3, stride=1, padding=1)
    return (x + strength * (x - blur)).clamp(0.0, 1.0).permute(0, 2, 3, 1)


def laplacian_numpy(images, strength):
    """FastLaplacianSharpen CPU path nodes.py:266-289 (adds neighbours - 4*centre: reference quirk D5)."""
    img, p = _edge_padded(images)
    lap = (p[:, 1:-1, 0:-2] + p[:, 0:-2, 1:-1] + p[:, 2:, 1:-1] + p[:, 1:-1, 2:] - 4.0 * img)
    out = img + strength * lap
    np.clip(out, 0.0, 1.0, out=out)
    return torch.from_numpy(out)


def laplacian_torch(images, strength):
    """nodes.py:244-261."""
    x = images.permute(0, 3, 1, 2)
    k = torch.tensor([[0, -1, 0], [-1, 4, -1], [0, -1, 0]], dtype=torch.float32).expand(3, 1, 3, 3)
    edges = F.conv2d(x, k, padding=1, groups=3)
    return (x + strength * edges).clamp(0.0, 1.0).permute(0, 2, 3, 1)


def sobel_numpy(images, strength):
    """FastSobelSharpen CPU path nodes.py:357-384."""
    img, p = _edge_padded(images)
    gx = (-p[:, 0:-2, 0:-2] - 2 * p[:, 1:-1, 0:-2] - p[:, 2:, 0:-2] +
          p[:, 0:-2, 2:] + 2 * p[:, 1:-1, 2:] + p[:, 2:, 2:])
    gy = (-p[:, 0:-2, 0:-2] - 2 * p[:, 0:-2, 1:-1] - p[:, 0:-2, 2:] +
          p[:, 2:, 0:-2] + 2 * p[:, 2:, 1:-1] + p[:, 2:, 2:])
    out = img + strength * np.sqrt(gx * gx + gy * gy)
    np.clip(out, 0.0, 1.0, out=out)
    return torch.from_numpy(out)


def sobel_torch(images, strength):
    """nodes.py:324-352."""
    x = images.permute(0, 3, 1, 2)
    sx = torch.tensor([[-1, 0, 1], [-2, 0, 2], [-1, 0, 1]], dtype=torch.float32).expand(3, 1, 3, 3)
    sy = torch.tensor([[-1, -2, -1], [0, 0, 0], [1, 2, 1]], dtype=torch.float32).expand(3, 1, 3, 3)
    gx = F.conv2d(x, sx, padding=1, groups=3)
    gy = F.conv2d(x, sy, padding=1, groups=3)
    edges = torch.sqrt(gx * gx + gy * gy + 1e-6)
    return (x + strength * edges).clamp(0.0, 1.0).permute(0, 2, 3, 1)


def effects_batch(images, settings, frame_start=0):
    """_apply_effects_batch on CPU, EnhancerNodes.py:278-294: unsharp (numpy path) then seeded grain."""
    batch = images
    if settings.get("sharpen_enabled", True):
        s = float(settings.get("sharpen_strength", 0.5))
        if s > 0:
            batch = unsharp_numpy(batch, s)
    if settings.get("grain_enabled", False):
        batch = seeded_grain(batch, float(settings.get("grain_intensity", 0.04)), float(settings.get("saturation_mix", 0.5)),
                             int(settings.get("seed", 42)), int(frame_start))
    return batch


# --------------------------------------------------------------------------------------------------
# CIE Lab (kornia.color restatement — parity unpinned, see module docstring)
# --------------------------------------------------------------------------------------------------
def rgb_to_lab(image):
    """kornia.color.rgb_to_lab on NCHW float tensors (call sites nodes.py:98,108)."""
    lin = torch.where(image > 0.04045, torch.pow((image + 0.055) / 1.055, 2.4), image / 12.92)
    r, g, b = lin[..., 0, :, :], lin[..., 1, :, :], lin[..., 2, :, :]
    x = 0.412453 * r + 0.357580 * g + 0.180423 * b
    y = 0.212671 * r + 0.715160 * g + 0.072169 * b
    z = 0.019334 * r + 0.119193 * g + 0.950227 * b
    xyz = torch.stack([x, y, z], dim=-3)
    white = torch.tensor([0.95047, 1.0, 1.08883], device=xyz.device, dtype=xyz.dtype)[..., :, None, None]
    xyz_n = torch.div(xyz, white)
    thr = 0.008856
    power = torch.pow(xyz_n.clamp(min=thr), 1 / 3.0)
    scale = 7.787 * xyz_n + 4.0 / 29.0
    f = torch.where(xyz_n > thr, power, scale)
    fx, fy, fz = f[..., 0, :, :], f[..., 1, :, :], f[..., 2, :, :]
    return torch.stack([(116.0 * fy) - 16.0, 500.0 * (fx - fy), 200.0 * (fy - fz)], dim=-3)


def lab_to_rgb(image, clip=True):
    """kornia.color.lab_to_rgb (call site nodes.py:115)."""
    L, a, b_ = image[..., 0, :, :], image[..., 1, :, :], image[..., 2, :, :]
    fy = (L + 16.0) / 116.0
    fx = (a / 500.0) + fy
    fz = (fy - (b_ / 200.0)).clamp(min=0.0)
    fxyz = torch.stack([fx, fy, fz], dim=-3)
    power = torch.pow(fxyz, 3.0)
    scale = (fxyz - 4.0 / 29.0) / 7.787
    xyz = torch.where(fxyz > 0.2068966, power, scale)
    white = torch.tensor([0.95047, 1.0, 1.08883], device=xyz.device, dtype=xyz.dtype)[..., :, None, None]
    xyz = xyz * white
    x, y, z = xyz[..., 0, :, :], xyz[..., 1, :, :], xyz[..., 2, :, :]
    r = 3.2404813432005266 * x + -1.5371515162713185 * y + -0.4985363261688878 * z
    g = -0.9692549499965682 * x + 1.8759900014898907 * y + 0.0415559265582928 * z
    b = 0.0556466391351772 * x + -0.2040413383665112 * y + 1.0573110696453443 * z
    lin = torch.stack([r, g, b], dim=-3)
    thr = 0.0031308
    rgb = torch.where(lin > thr, 1.055 * torch.pow(lin.clamp(min=thr), 1 / 2.4) - 0.055, 12.92 * lin)
    return torch.clamp(rgb, min=0.0, max=1.0) if clip else rgb


def color_match(images, reference_image, match_strength, batch_size=1):
    """ColorMatchToReference.match_color, nodes.py:91-124, on CPU (autocast is a no-op for CPU tensors)."""
    imgs = images.permute(0, 3, 1, 2)
    ref = reference_image.permute(0, 3, 1, 2)
    ref_lab = rgb_to_lab(ref)
    ref_mean = ref_lab.mean(dim=[2, 3], keepdim=True)
    ref_std = ref_lab.std(dim=[2, 3], keepdim=True) + 1e-5
    outs = []
    for i in range(0, imgs.shape[0], batch_size):
        lab = rgb_to_lab(imgs[i:i + batch_size])
        mean = lab.mean(dim=[2, 3], keepdim=True)
        std = lab.std(dim=[2, 3], keepdim=True) + 1e-5
        matched = (lab - mean) / std * ref_std + ref_mean
        blended = match_strength * matched + (1.0 - match_strength) * lab
        outs.append(lab_to_rgb(blended))
    return torch.cat(outs, dim=0).clamp(0.0, 1.0).permute(0, 2, 3, 1)


def lab_moments_f64(images):
    """float64 raw LAB sums [B,7] = {n, S1[3], S2[3]} of fp32 LAB values: what vrgdg_lab_moments accumulates."""
    lab = rgb_to_lab(images.permute(0, 3, 1, 2)).double()
    n = float(lab.shape[2] * lab.shape[3])
    s1 = lab.sum(dim=[2, 3])
    s2 = (lab * lab).sum(dim=[2, 3])
    return torch.cat([torch.full((lab.shape[0], 1), n, dtype=torch.float64), s1, s2], dim=1)


# --------------------------------------------------------------------------------------------------
# 3D LUT
# --------------------------------------------------------------------------------------------------
def parse_cube(path):
    """VRGDG_LUTS._parse_cube_file, VRGDG_IV_Adjustments.py:222-282."""
    size = None
    dmin = np.array([0.0, 0.0, 0.0], dtype=np.float32)
    dmax = np.array([1.0, 1.0, 1.0], dtype=np.float32)
    vals = []
    with open(path, "r", encoding="utf-8", errors="ignore") as fh:
        for raw in fh:
            line = raw.strip()
            if not line or line.startswith("#"):
                continue
            up = line.upper()
            if up.startswith("TITLE "):
                continue
            if up.startswith("LUT_1D_SIZE"):
                raise ValueError(f"1D LUTs are not supported: {os.path.basename(path)}")
            tok = line.split()
            if up.startswith("LUT_3D_SIZE"):
                if len(tok) != 2:
                    raise ValueError(f"Invalid LUT_3D_SIZE line in {path}")
                size = int(tok[1])
                continue
            if up.startswith("DOMAIN_MIN") or up.startswith("DOMAIN_MAX"):
                if len(tok) != 4:
                    raise ValueError(f"Invalid {tok[0]} line in {path}")
                arr = np.array([float(tok[1]), float(tok[2]), float(tok[3])], dtype=np.float32)
                if up.startswith("DOMAIN_MIN"):
                    dmin = arr
                else:
                    dmax = arr
                continue
            if len(tok) != 3:
                continue
            vals.extend(float(t) for t in tok)
    if size is None:
        raise ValueError(f"Missing LUT_3D_SIZE in {path}")
    expected = size * size * size * 3
    if len(vals) != expected:
        raise ValueError(f"Invalid LUT data length in {path}. Expected {expected} floats, got {len(vals)}.")
    lut = torch.from_numpy(np.asarray(vals, dtype=np.float32).reshape(size, size, size, 3))
    return {"size": size, "lut": lut, "domain_min": torch.from_numpy(dmin), "domain_max": torch.from_numpy(dmax)}


def apply_cube_lut(image, lut, domain_min, domain_max):
    """VRGDG_LUTS._apply_cube_lut, VRGDG_IV_Adjustments.py:289-343."""
    if image.ndim != 4 or image.shape[-1] < 3:
        raise ValueError("VRGDG_LUTS expects IMAGE input shaped like [batch, height, width, channels].")
    src = image[..., :3].to(dtype=torch.float32)
    span = torch.clamp(domain_max - domain_min, min=1e-6)
    norm = torch.clamp((src - domain_min) / span, 0.0, 1.0)
    top = lut.shape[0] - 1
    coords = norm * top
    r, g, b = coords[..., 0], coords[..., 1], coords[..., 2]
    r0, g0, b0 = torch.floor(r).long(), torch.floor(g).long(), torch.floor(b).long()
    r1, g1, b1 = torch.clamp(r0 + 1, max=top), torch.clamp(g0 + 1, max=top), torch.clamp(b0 + 1, max=top)
    fr, fg, fb = (r - r0.float()).unsqueeze(-1), (g - g0.float()).unsqueeze(-1), (b - b0.float()).unsqueeze(-1)
    c00 = lut[b0, g0, r0] * (1.0 - fb) + lut[b1, g0, r0] * fb
    c01 = lut[b0, g1, r0] * (1.0 - fb) + lut[b1, g1, r0] * fb
    c10 = lut[b0, g0, r1] * (1.0 - fb) + lut[b1, g0, r1] * fb
    c11 = lut[b0, g1, r1] * (1.0 - fb) + lut[b1, g1, r1] * fb
    c0 = c00 * (1.0 - fg) + c01 * fg
    c1 = c10 * (1.0 - fg) + c11 * fg
    rgb = torch.clamp(c0 * (1.0 - fr) + c1 * fr, 0.0, 1.0)
    if image.shape[-1] == 3:
        return rgb.to(dtype=image.dtype)
    out = image.clone()
    out[..., :3] = rgb.to(dtype=image.dtype)
    return out


def apply_lut(image, lut_data, strength):
    """VRGDG_LUTS.apply_lut on CPU, VRGDG_IV_Adjustments.py:349-361 (== _apply_lut_tensor LUTVideoTools.py:172-185)."""
    dmin = lut_data["domain_min"].to(dtype=image.dtype)
    dmax = lut_data["domain_max"].to(dtype=image.dtype)
    out = apply_cube_lut(image, lut_data["lut"], dmin, dmax)
    blend = max(0.0, min(10.0, float(strength))) / 10.0
    if blend <= 0.0:
        return image
    if blend < 1.0:
        return (image * (1.0 - blend)) + (out * blend)
    return out


def palette_lut(colors_rgb, lut_size):
    """_build_palette_lut, VRGDG_IV_Adjustments.py:75-105; colors_rgb: float32 [n,3] (already parsed)."""
    palette = np.asarray(colors_rgb, dtype=np.float32)
    axis = np.linspace(0.0, 1.0, int(lut_size), dtype=np.float32)
    blue, green, red = np.meshgrid(axis, axis, axis, indexing="ij")
    source = np.stack([red, green, blue], axis=-1)
    luma = (0.2126 * source[..., 0]) + (0.7152 * source[..., 1]) + (0.0722 * source[..., 2])
    if palette.shape[0] == 1:
        target = np.empty(luma.shape + (3,), dtype=np.float32)
        target[...] = palette[0]
    else:
        pos = np.linspace(0.0, 1.0, palette.shape[0], dtype=np.float32)
        flat = luma.reshape(-1)
        target = np.stack([np.interp(flat, pos, palette[:, c]) for c in range(3)], axis=-1)
        target = target.reshape(luma.shape + (3,)).astype(np.float32)
    tl = (0.2126 * target[..., 0]) + (0.7152 * target[..., 1]) + (0.0722 * target[..., 2])
    scale = luma / np.maximum(tl, 1e-6)
    target = np.clip(target * scale[..., None], 0.0, 1.0)
    chroma = source - luma[..., None]
    out = np.clip((target * 0.82) + ((target + chroma) * 0.18), 0.0, 1.0)
    return torch.from_numpy(out.astype(np.float32))


# --------------------------------------------------------------------------------------------------
# "adjust" (temperature / tint / exposure / contrast / saturation / tonal masks / clarity / sharpen / fade / vignette)
# --------------------------------------------------------------------------------------------------
ADJUST_FIELDS = {"temperature": (-100.0, 100.0), "tint": (-100.0, 100.0), "saturation": (-100.0, 100.0), "exposure": (-100.0, 100.0),
                 "contrast": (-100.0, 100.0), "highlights": (-100.0, 100.0), "shadows": (-100.0, 100.0), "whites": (-100.0, 100.0),
                 "blacks": (-100.0, 100.0), "sharpen": (0.0, 100.0), "clarity": (-100.0, 100.0), "vignette": (0.0, 100.0), "fade": (0.0, 100.0)}


def normalize_adjust_settings(settings=None):
    """_normalize_adjust_settings, VRGDG_LUTVideoTools.py:280-304."""
    settings = settings if isinstance(settings, dict) else {}
    out = {"enabled": settings.get("enabled", True) is not False}
    for key, (lo, hi) in ADJUST_FIELDS.items():
        try:
            v = float(settings.get(key, 0.0))
        except Exception:
            v = 0.0
        out[key] = max(lo, min(hi, v))
    return out


def _luma(t):
    return (t[..., 0:1] * 0.2126) + (t[..., 1:2] * 0.7152) + (t[..., 2:3] * 0.0722)


def adjust(image_tensor, settings=None):
    """_apply_adjust_tensor on CPU, VRGDG_LUTVideoTools.py:307-391."""
    a = normalize_adjust_settings(settings)
    src = image_tensor.clamp(0.0, 1.0)
    if not a["enabled"]:
        return src
    out = src + torch.tensor([a["temperature"] / 400.0 - a["tint"] / 900.0, a["tint"] / 450.0, -a["temperature"] / 400.0 - a["tint"] / 900.0],
                             dtype=src.dtype).view(1, 1, 1, 3)
    out = out * (2.0 ** (a["exposure"] / 100.0))
    out = (out - 0.5) * (1.0 + (a["contrast"] / 100.0)) + 0.5
    gray = _luma(out).repeat(1, 1, 1, 3)
    out = gray + (out - gray) * (1.0 + (a["saturation"] / 100.0))
    luma = _luma(out)
    out = out + torch.clamp((luma - 0.55) / 0.45, 0.0, 1.0) * (a["highlights"] / 220.0)
    out = out + torch.clamp((0.45 - luma) / 0.45, 0.0, 1.0) * (a["shadows"] / 220.0)
    out = out + torch.clamp((luma - 0.75) / 0.25, 0.0, 1.0) * (a["whites"] / 240.0)
    out = out + torch.clamp((0.25 - luma) / 0.25, 0.0, 1.0) * (a["blacks"] / 240.0)
    clarity, sharpen = a["clarity"] / 100.0, a["sharpen"] / 100.0
    if abs(clarity) > 0.001 or sharpen > 0.001:
        x = out.permute(0, 3, 1, 2)
        h, w = int(x.shape[2]), int(x.shape[3])
        if abs(clarity) > 0.001:
            k = min(9, h if h % 2 else h - 1, w if w % 2 else w - 1)
            blur = x if k < 3 else F.avg_pool2d(F.pad(x, (k // 2,) * 4, mode="reflect"), kernel_size=k, stride=1)
            ln = x[:, 0:1] * 0.2126 + x[:, 1:2] * 0.7152 + x[:, 2:3] * 0.0722
            mid = 1.0 - torch.clamp(torch.abs(ln - 0.5) / 0.5, 0.0, 1.0)
            x = x + (x - blur) * clarity * 1.55 * (0.35 + mid * 0.65)
        if sharpen > 0.001:
            fine = F.avg_pool2d(F.pad(x, (1, 1, 1, 1), mode="replicate"), kernel_size=3, stride=1)
            x = x + (x - fine) * sharpen * 5.0
        out = x.permute(0, 2, 3, 1)
    fade = a["fade"] / 100.0
    if fade > 0.0:
        out = out * (1.0 - fade * 0.35) + fade * 0.18
    vig = a["vignette"] / 100.0
    if vig > 0.0:
        h, w = out.shape[1], out.shape[2]
        yy = torch.linspace(-1.0, 1.0, h, dtype=out.dtype).view(1, h, 1, 1)
        xx = torch.linspace(-1.0, 1.0, w, dtype=out.dtype).view(1, 1, w, 1)
        dist = torch.sqrt((xx * xx) + (yy * yy))
        out = out * (1.0 - torch.clamp((dist - 0.35) / 1.05, 0.0, 1.0) * vig * 0.75)
    return out.clamp(0.0, 1.0)


# --------------------------------------------------------------------------------------------------
# resize / restore around the enhancer (VRGDG_VideoEnhanceNodes.py:45-106, :408-414)
# --------------------------------------------------------------------------------------------------
INTERPOLATIONS = {"Nearest": "nearest", "Bilinear": "bilinear", "Bicubic (recommended)": "bicubic", "Area": "area"}


def resize_batch(images, target_width, target_height, fit_mode, resize_method):
    """_resize_batch, VRGDG_VideoEnhanceNodes.py:54-86."""
    if images.ndim != 4 or images.shape[0] < 1:
        raise ValueError("Video Enhance requires a non-empty IMAGE batch.")
    sh, sw = int(images.shape[1]), int(images.shape[2])
    tw, th = int(target_width), int(target_height)
    x = images[..., :3].permute(0, 3, 1, 2)
    mode = INTERPOLATIONS.get(str(resize_method), "bicubic")
    kw = {"mode": mode}
    if mode in ("bilinear", "bicubic"):
        kw["align_corners"] = False
    if fit_mode == "Stretch to dimensions":
        res = F.interpolate(x, size=(th, tw), **kw)
    else:
        scale = max(tw / sw, th / sh) if fit_mode == "Crop to fill" else min(tw / sw, th / sh)
        rw, rh = max(1, int(round(sw * scale))), max(1, int(round(sh * scale)))
        r = F.interpolate(x, size=(rh, rw), **kw)
        if fit_mode == "Crop to fill":
            left, top = max(0, (rw - tw) // 2), max(0, (rh - th) // 2)
            res = r[:, :, top:top + th, left:left + tw]
        else:
            pl = max(0, (tw - rw) // 2)
            pt = max(0, (th - rh) // 2)
            res = F.pad(r, (pl, max(0, tw - rw - pl), pt, max(0, th - rh - pt)), value=0.0)
    return res.permute(0, 2, 3, 1).clamp(0, 1)


def restore_batch(images, source_width, source_height, fit_mode, resize_method):
    """_restore_batch, VRGDG_VideoEnhanceNodes.py:89-106."""
    if fit_mode != "Fit with letterbox (preserve all)":
        return resize_batch(images, source_width, source_height, "Stretch to dimensions", resize_method)
    wh, ww = int(images.shape[1]), int(images.shape[2])
    scale = min(ww / source_width, wh / source_height)
    cw = min(ww, max(1, int(round(source_width * scale))))
    ch = min(wh, max(1, int(round(source_height * scale))))
    left, top = max(0, (ww - cw) // 2), max(0, (wh - ch) // 2)
    return resize_batch(images[:, top:top + ch, left:left + cw, :], source_width, source_height, "Stretch to dimensions", resize_method)


def restore_blend(originals, restored, strength):
    """VRGDG_VideoEnhanceNodes.py:408-414: lerp of the restored frames over the originals, clamp."""
    s = float(strength)
    return (originals * (1.0 - s) + restored * s).clamp(0, 1)


# --------------------------------------------------------------------------------------------------
# the enhancer's Lanczos4 resize of uint8 frames (_resize_frames, VRGDG_StandaloneVideoEnhancerNodes.py:213-230)
# The arithmetic lives in a dependency that is not vendored in the reference: OpenCV (cv2.resize, INTER_LANCZOS4; the pack pins
# no version, this image has opencv 4.13.0).  Restated from OpenCV's published algorithm (imgproc/resize.cpp: interpolateLanczos4,
# the 8-tap fixed-point tables with INTER_RESIZE_COEF_BITS = 11, HResizeLanczos4 / VResizeLanczos4 with border replication and
# FixedPtCast<int, uchar, 22>) and pinned bit-exactly against cv2 itself (tests/golden/lanczos.npz, make_golden.py).
# --------------------------------------------------------------------------------------------------
def lanczos4_coeffs(x):
    """interpolateLanczos4: 8 fp32 weights for the fractional offset x (an fp32 value)."""
    s45 = 0.70710678118654752440084436210485
    cs = ((1, 0), (-s45, -s45), (0, 1), (s45, -s45), (-1, 0), (s45, s45), (0, -1), (-s45, s45))
    f32 = np.float32
    y0 = float(-f32(f32(x) + f32(3))) * math.pi * 0.25           # (x+3) is a float sum in OpenCV; only then promoted to double
    s0, c0 = math.sin(y0), math.cos(y0)
    co, total = [], f32(0)
    for i in range(8):
        d = f32(f32(x) + f32(3) - f32(i))
        if abs(d) >= f32(1e-6):
            y = -float(d) * math.pi * 0.25
            c = f32((cs[i][0] * s0 + cs[i][1] * c0) / (y * y))
        else:
            c = f32(1e30)
        co.append(c)
        total = f32(total + c)
    inv = f32(f32(1) / total)
    return [f32(c * inv) for c in co]


def lanczos4_tables(ssize, dsize):
    """per destination index: first-tap source index (sx, taps are sx-3 .. sx+4) and the 8 weights as saturated shorts (x 2048)."""
    scale = 1.0 / (dsize / ssize)                                   # resize(): scale_x = 1. / inv_scale_x, doubles
    ofs = np.zeros(dsize, np.int32)
    coef = np.zeros((dsize, 8), np.int16)
    for d in range(dsize):
        fx = np.float32((d + 0.5) * scale - 0.5)
        sx = math.floor(float(fx))
        ofs[d] = sx
        for k, c in enumerate(lanczos4_coeffs(np.float32(fx - np.float32(sx)))):
            coef[d, k] = max(-32768, min(32767, int(np.rint(np.float32(c * np.float32(2048))))))   # saturate_cast<short>(cvRound)
    return ofs, coef


def resize_lanczos4_u8(frame, out_w, out_h):
    """cv2.resize(frame, (out_w, out_h), interpolation=cv2.INTER_LANCZOS4) for a uint8 [H,W,C] frame."""
    sh, sw = frame.shape[:2]
    xo, xa = lanczos4_tables(sw, int(out_w))
    yo, ya = lanczos4_tables(sh, int(out_h))
    src = frame.astype(np.int32)
    taps = np.arange(-3, 5)
    xi = np.clip(xo[:, None] + taps[None, :], 0, sw - 1)
    yi = np.clip(yo[:, None] + taps[None, :], 0, sh - 1)
    h = np.zeros((sh, int(out_w), frame.shape[2]), np.int32)
    for k in range(8):
        h += src[:, xi[:, k], :] * xa[:, k].astype(np.int32)[None, :, None]
    v = np.zeros((int(out_h), int(out_w), frame.shape[2]), np.int32)
    for k in range(8):
        v += h[yi[:, k]] * ya[:, k].astype(np.int32)[:, None, None]
    return np.clip((v + (1 << 21)) >> 22, 0, 255).astype(np.uint8)


def resize_frames(frames, output_width, output_height):
    """_resize_frames, VRGDG_StandaloneVideoEnhancerNodes.py:213-230: frames already at the output size pass through."""
    ow, oh = max(1, int(output_width)), max(1, int(output_height))
    return [f if (f.shape[1] == ow and f.shape[0] == oh) else resize_lanczos4_u8(f, ow, oh) for f in frames]


# --------------------------------------------------------------------------------------------------
# uint8 BGR wire format
# --------------------------------------------------------------------------------------------------
def frames_to_tensor(frames_bgr_u8):
    """_frames_to_tensor, VRGDG_LUTVideoTools.py:736-743 (cv2.COLOR_BGR2RGB == channel reversal)."""
    rgb = np.ascontiguousarray(np.asarray(frames_bgr_u8)[..., ::-1])
    return torch.from_numpy(rgb.astype(np.float32) / 255.0)


def tensor_to_frames(tensor):
    """_tensor_to_frames, VRGDG_LUTVideoTools.py:746-752: clip(x*255) TRUNCATED to uint8, RGB->BGR."""
    arr = np.clip(tensor.detach().cpu().numpy() * 255.0, 0, 255).astype(np.uint8)
    return np.ascontiguousarray(arr[..., ::-1])


# --------------------------------------------------------------------------------------------------
# compositions used by the benchmark configs (reference nodes applied one after another)
# --------------------------------------------------------------------------------------------------
def chain_grain_lut_unsharp(images, noise, grain_intensity, saturation_mix, lut_data, lut_strength, sharpen_strength):
    """config 2: FastFilmGrain -> VRGDG_LUTS -> FastUnsharpSharpen(use_gpu=False)."""
    x = film_grain(images, grain_intensity, saturation_mix, batch_size=0, noise=noise)
    x = apply_lut(x, lut_data, lut_strength)
    return unsharp_numpy(x, sharpen_strength)


def chain_full(images, noise, grain_intensity, saturation_mix, reference_image, match_strength, lut_data, lut_strength,
               sharpen_strength):
    """config 4: grain -> colour match -> LUT -> unsharp."""
    x = film_grain(images, grain_intensity, saturation_mix, batch_size=0, noise=noise)
    x = color_match(x, reference_image, match_strength, batch_size=1)
    x = apply_lut(x, lut_data, lut_strength)
    return unsharp_numpy(x, sharpen_strength)


def hist_counts(images):
    """256-bin counts per frame and RGB channel: bin = min(floor(clip(v,0,1) * 256), 255) evaluated in fp32.  int64 [B,3,256]."""
    x = images.detach().cpu().float().numpy()
    u = np.clip(x, np.float32(0.0), np.float32(1.0)) * np.float32(256.0)
    k = np.minimum(u.astype(np.int64), 255)
    B = x.shape[0]
    out = np.zeros((B, 3, 256), dtype=np.int64)
    for b in range(B):
        for c in range(3):
            out[b, c] = np.bincount(k[b, ..., c].ravel(), minlength=256)
    return torch.from_numpy(out)


def histmatch_tables(frame_counts, ref_counts):
    """Edge tables T[0..256] = ref_CDF^-1(frame_CDF(edge)) with both CDFs piecewise linear over the bin edges.  NOT a restatement of
    reference code (the reference has no histogram colour match, SURVEY D1): this IS the specification of the extension (parity
    unpinned).  float32 [B,3,257]."""
    fc = frame_counts.numpy().astype(np.int64)
    rc = ref_counts.numpy().astype(np.int64)
    B = fc.shape[0]
    T = np.zeros((B, 3, 257), dtype=np.float32)
    for b in range(B):
        for c in range(3):
            cf = np.cumsum(fc[b, c])
            cr = np.cumsum(rc[0 if rc.shape[0] == 1 else b, c])
            nf, nr = int(cf[-1]), int(cr[-1])
            for e in range(257):
                if nf == 0 or nr == 0:
                    T[b, c, e] = np.float32(e / 256.0)
                    continue
                cq = 0 if e == 0 else int(cf[e - 1])
                g = lambda i: (0 if i == 0 else int(cr[i - 1])) * nf          # edge values of the reference CDF, scaled: exact integers
                rhs = cq * nr
                ilo = next(i for i in range(257) if g(i) >= rhs)
                if g(ilo) == rhs:                                              # q lies ON edges ilo..ihi (plateau): inverse closest to the source edge
                    ihi = max(i for i in range(ilo, 257) if g(i) <= rhs)
                    T[b, c, e] = np.float32(np.float64(min(max(e, ilo), ihi)) / np.float64(256.0))
                else:                                                          # strictly inside the rising segment of bin j
                    j = ilo - 1
                    q = np.float64(cq) / np.float64(nf)
                    prev = np.float64(cr[j - 1]) / np.float64(nr) if j > 0 else np.float64(0.0)
                    cur = np.float64(cr[j]) / np.float64(nr)
                    frac = (q - prev) / (cur - prev)
                    T[b, c, e] = np.float32((np.float64(j) + frac) / np.float64(256.0))
    return torch.from_numpy(T)


def hist_match(images, reference_image, strength):
    """Histogram / CDF colour transfer (extension; see histmatch_tables): out = clip(x*(1-t) + map(x)*t), fp32, one rounding per op."""
    x = images.detach().cpu().float().numpy()
    T = histmatch_tables(hist_counts(images), hist_counts(reference_image)).numpy()
    t = np.float32(strength)
    omt = np.float32(1.0 - float(strength))
    u = np.clip(x, np.float32(0.0), np.float32(1.0)) * np.float32(256.0)
    k = np.minimum(u.astype(np.int64), 255)
    w = u - k.astype(np.float32)
    out = np.empty_like(x)
    for b in range(x.shape[0]):
        for c in range(3):
            t0 = T[b, c][k[b, ..., c]]
            dt = (T[b, c][1:] - T[b, c][:-1]).astype(np.float32)[k[b, ..., c]]
            m = (w[b, ..., c].astype(np.float64) * dt.astype(np.float64) + t0.astype(np.float64)).astype(np.float32)     # one FMA: exact product, one rounding
            out[b, ..., c] = np.clip(x[b, ..., c] * omt + m * t, np.float32(0.0), np.float32(1.0))
    return torch.from_numpy(out)


def temporal_sharpen(frames, strength, prev_frame=None, next_frame=None):
    """configs[4] temporal 3-frame unsharp.  NOT a restatement of reference code: the reference has no temporal operator (SURVEY D4),
    so this NumPy function IS the specification (parity unpinned):
        out[t] = clip(x[t] + s * (x[t] - (x[t-1] + x[t] + x[t+1]) / 3), 0, 1), fp32, frames outside the clip replicated."""
    x = frames.detach().cpu().float().numpy()
    first = x[:1] if prev_frame is None else prev_frame.detach().cpu().float().numpy().reshape(x[:1].shape)
    last = x[-1:] if next_frame is None else next_frame.detach().cpu().float().numpy().reshape(x[:1].shape)
    prev = np.concatenate([first, x[:-1]], axis=0)
    nxt = np.concatenate([x[1:], last], axis=0)
    mean = ((prev + x) + nxt) / np.float32(3.0)
    out = x + np.float32(strength) * (x - mean)
    return torch.from_numpy(np.clip(out, 0.0, 1.0).astype(np.float32))


def lab_reference_f64(rgb):
    """Independent float64 CIE evaluation (numpy, textbook formulas) used only to sanity-check rgb_to_lab."""
    c = np.asarray(rgb, dtype=np.float64)
    lin = np.where(c > 0.04045, ((c + 0.055) / 1.055) ** 2.4, c / 12.92)
    M = np.array([[0.412453, 0.357580, 0.180423], [0.212671, 0.715160, 0.072169], [0.019334, 0.119193, 0.950227]])
    xyz = lin @ M.T / np.array([0.95047, 1.0, 1.08883])
    f = np.where(xyz > 0.008856, np.cbrt(np.maximum(xyz, 0.008856)), 7.787 * xyz + 4.0 / 29.0)
    return np.stack([116 * f[..., 1] - 16, 500 * (f[..., 0] - f[..., 1]), 200 * (f[..., 1] - f[..., 2])], axis=-1)
