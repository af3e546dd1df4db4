"""Shared test helpers: synthetic frames and golden loading."""
import os
import re

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
LUTS = os.path.join(ROOT, "comfyui-vrgamedevgirl_b200", "LUTS")


def white_frames(B, H, W, seed=1, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, H, W, 3, generator=g).to(dtype)


def natural_frames(B, H, W, seed=0, dtype=torch.float32, device="cpu"):
    """Spatially coherent frames: 4 octaves of bilinearly upsampled uniform noise + 2% white noise (SURVEY 8d, dist. N)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    acc = torch.zeros(B, 3, H, W)
    amp, tot = 1.0, 0.0
    for o in range(4):
        gh, gw = 8 * 2 ** o + 1, 15 * 2 ** o + 1
        base = torch.rand(B, 3, gh, gw, generator=g)
        acc += amp * torch.nn.functional.interpolate(base, size=(H, W), mode="bilinear", align_corners=True)
        tot += amp
        amp *= 0.5
    acc = acc / tot
    acc = acc + 0.02 * (torch.rand(B, 3, H, W, generator=g) - 0.5)
    off = torch.tensor([0.03, 0.0, -0.03]).view(1, 3, 1, 1)
    return (acc + off).clamp(0, 1).permute(0, 2, 3, 1).contiguous().to(dtype).to(device)


GOLDEN_FILE_BYTES = 1000000      # no stored vector file is larger than this: save_golden spreads the arrays over more files


def load_golden(name, directory=GOLDEN):
    """The arrays of tests/golden/<name>.npz and of its continuation files <name>_part<k>.npz."""
    out = {}
    for f in sorted(os.listdir(directory)):
        if f == name + ".npz" or re.fullmatch(re.escape(name) + r"_part\d+\.npz", f):
            with np.load(os.path.join(directory, f), allow_pickle=False) as z:
                out.update({k: z[k] for k in z.files})
    return out


def save_golden(name, arrays, directory=GOLDEN, limit=GOLDEN_FILE_BYTES):
    """np.savez_compressed `arrays` as <name>.npz, spread round-robin over <name>_part2.npz, _part3.npz, ... when one file would be
    larger than `limit` bytes.  load_golden(name) returns them as one dict again."""
    keys = list(arrays)
    for f in os.listdir(directory):
        if re.fullmatch(re.escape(name) + r"_part\d+\.npz", f):
            os.remove(os.path.join(directory, f))
    for n in range(1, len(keys) + 1):
        paths = [os.path.join(directory, name + (".npz" if i == 0 else "_part%d.npz" % (i + 1))) for i in range(n)]
        for i, path in enumerate(paths):
            np.savez_compressed(path, **{k: arrays[k] for k in keys[i::n]})
        if all(os.path.getsize(p) <= limit for p in paths):
            return paths
        for path in paths[1:]:
            os.remove(path)
    raise ValueError("one array of %s is larger than %d bytes compressed" % (name, limit))


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


# ---- large LUTs (64^3 / 65^3: 28 of the 40 tables the reference ships) ------------------------------------------------------
# Generated instead of committed (a 65^3 .cube is 7 MB of text): float64 arithmetic with +, -, *, / and clip only, printed with
# %.6f, so every machine writes the same file; tests/golden/lut_big.npz holds the SHA-256 of the parsed float32 table.
def big_lut_table(size):
    ax = np.linspace(0.0, 1.0, size, dtype=np.float64)
    b, g, r = np.meshgrid(ax, ax, ax, indexing="ij")                 # file order: red fastest
    rgb = np.stack([r, g, b], axis=-1)
    y = rgb[..., 0:1] * 0.2126 + rgb[..., 1:2] * 0.7152 + rgb[..., 2:3] * 0.0722
    w = np.clip((y - 0.15) / 0.7, 0.0, 1.0)
    x = rgb * (np.array([0.88, 1.02, 1.10]) * (1.0 - w) + np.array([1.10, 1.0, 0.88]) * w)
    x = 0.5 + (x - 0.5) * 1.15
    x = x + 0.05 * x * (1.0 - x) * (size / 64.0)                      # size-dependent term: the two tables differ in more than sampling
    return np.clip(x, 0.0, 1.0).reshape(-1, 3)


BIG_LUT_HEADERS = {
    64: ["# vrgdg-b200 test table (tests/helpers.py::big_lut_table)", 'TITLE "big 64"', "", "LUT_3D_SIZE 64", "", "DOMAIN_MIN 0.0 0.0 0.0",
         "DOMAIN_MAX 1.0 1.0 1.0", ""],
    65: ['TITLE "big 65"', "LUT_3D_SIZE 65", "DOMAIN_MIN 0 0 0", "DOMAIN_MAX 1 1 1"],       # integer DOMAIN lines, as 4 reference files have
}


def write_big_cube(path, size):
    rows = big_lut_table(size)
    with open(path, "w", encoding="utf-8") as fh:
        for line in BIG_LUT_HEADERS[size]:
            fh.write(line + "\n")
        fh.write("\n".join("%.6f %.6f %.6f" % (a, b, c) for a, b, c in rows))
        fh.write("\n")
    return path
