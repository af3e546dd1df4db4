import importlib, os, sys, json, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
pkg = importlib.import_module("comfyui-vrgamedevgirl_b200")
from helpers import LUTS, natural_frames
nv, ops = pkg._native, pkg.ops
dev = torch.device("cuda", 0)
lut = pkg.VRGDG_LUTS._parse_cube_file(os.path.join(LUTS, "B200 Vintage 33.cube"))
B,H,W=32,2160,3840
x = natural_frames(8, H, W, seed=1, device=dev).repeat(B // 8, 1, 1, 1).contiguous()
out = torch.empty_like(x)
ref_sums = ops.lab_moments(natural_frames(1, H, W, seed=9, device=dev))
def timeit(fn, iters=8, warm=3):
    for _ in range(warm): fn()
    ts=[]
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
    ts.sort(); return ts[len(ts)//2]
for name, kw in (("grain_cm_lut (k_point apply)", dict(grain=dict(intensity=0.04, saturation_mix=0.5, seed=42), lut=dict(lut_data=lut, strength=10.0))),
                 ("cm_lut (k_point apply)", dict(lut=dict(lut_data=lut, strength=10.0))),
                 ("cm_lut_unsharp (k_tile apply, no grain)", dict(lut=dict(lut_data=lut, strength=10.0), stencil=dict(op=nv.STENCIL_BOX_UNSHARP, strength=0.5)))):
    c = pkg.chain.PostChain(colormatch=dict(ref_sums=ref_sums, strength=1.0), device=dev, **kw)
    for serial in (False, True):
        c.serial = serial
        ms = timeit(lambda: c(x, out=out))
        print(json.dumps({"chain": name, "serial": serial, "ms": round(ms,3), "GPx/s": round(B*H*W/ms/1e6,1)}), flush=True)
