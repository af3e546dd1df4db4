"""bench.py — headline benchmark of the post-processing hot path (driver contract: DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Headline workload = the configuration BASELINE.json's metric is quoted on ("grain+LUT+colormatch+sharpen chain at 4K"), i.e. the
per-GPU shard of configs[3]: grain(I=.04, s=.5, seed 42) -> colour match(t=1, one 4K reference frame) -> 33^3 .cube LUT ->
unsharp(.5) on 128 x 3840x2160 fp32 frames per GPU, synthesised on the device (weak scaling: every rank owns 128 frames).
One "step" = one pass of the chain over the rank's frames:
    reference moments (k_lab_moments on the rank's row shard + ONE NCCL all-gather of 56 bytes per rank, dist.py)
    -> vrgdg_chain_cm_apply, per group of 8 frames: k_lab_moments (grain drawn, forward Lab, statistics, (fx,fy,fz) planes stored)
       -> k_moments_final -> k_colormatch_params -> k_tile (colour match from the planes + LUT + unsharp);
       the statistics pass of group g+1 runs concurrently with the apply pass of group g (two internal streams, split register file)
  value : MP/s, frames resident in HBM (CUDA events around K steps on the launching stream, max over ranks)
  e2e   : MP/s through the public API (PostChain.run_host) from pinned HOST frames to pinned HOST frames on a stated sub-batch,
          H2D and D2H copies inside the timed region; e2e.stock_nodes = the same chain as four unchanged ComfyUI nodes
  extra : configs[1] (64 x 1080p fp16, grain + LUT + unsharp), "grain + LUT + unsharp at 4K fp32", configs[2] (colour match alone: LAB
          transfer and histogram mode, reference statistics gathered every step), configs[4] (temporal sharpen), each with its own roofline
  --impl reference : the reference's CPU path for the same chain (oracle port of the reference nodes, so the reference's own
          source is not needed) on all host cores, rank 0 only, 2 frames per step, --steps timed steps
"""
import argparse
import importlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def host_threads():
    """Threads for the CPU arm: one per PHYSICAL core (torch's own default; measured on the GPU box: 128 SMT threads run the
    reference chain 3x slower than 64)."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:
        n = None
    return int(n or max(1, (os.cpu_count() or 2) // 2))


if "reference" in sys.argv:      # the CPU arm uses every core; torchrun would otherwise pin OMP_NUM_THREADS=1
    os.environ["OMP_NUM_THREADS"] = str(host_threads())
    os.environ["MKL_NUM_THREADS"] = str(host_threads())

import torch  # noqa: E402

PKG = "comfyui-vrgamedevgirl_b200"
LUT_FILE = os.path.join(ROOT, PKG, "LUTS", "B200 Vintage 33.cube")
GRAIN = dict(intensity=0.04, saturation_mix=0.5, seed=42)
SHARPEN = 0.5
METRIC = "megapixels/sec (grain+LUT+colormatch+sharpen chain) at 4K"
H4K, W4K = 2160, 3840
FRAMES_4K = int(os.environ.get("VRGDG_BENCH_FRAMES", "128"))       # per GPU (configs[3]: 1024 frames over 8 GPUs)
E2E_FRAMES = 16                                                      # sub-batch of the end-to-end leg (1.6 GB each way)
STOCK_FRAMES = 4                                                     # sub-batch of the stock-node leg
WORKLOAD = ("configs[3] per-GPU shard: grain -> colour match (one 4K reference, t=1) -> 33^3 .cube LUT -> unsharp, "
            "%d x 3840x2160 fp32 frames per GPU" % FRAMES_4K)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_traffic(key):
    """dram bytes per launch of a kernel from the committed ncu capture (profiles/dominant_kernel.json), with a staleness flag:
    the capture is only valid for the kernel sources it was taken from (content hash of csrc/ + the header)."""
    path = os.path.join(ROOT, "profiles", "dominant_kernel.json")
    if not os.path.exists(path):
        return None, None
    with open(path) as fh:
        d = json.load(fh).get(key)
    if not d:
        return None, None
    try:
        cur = importlib.import_module(PKG + ".build")._source_hash()
    except Exception:
        cur = None
    return d.get("dram_bytes_per_launch"), {"capture": d.get("capture"), "traffic_stale": bool(cur is None or d.get("src_hash") != cur)}


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled every 10 ms during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80, "sw_power_cap": 0x4}
        while not self.stop_flag.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def device_natural_frames(n, h, w, seed, dtype, dev):
    """helpers.natural_frames (SURVEY 8d distribution N: 4 octaves of bilinearly upsampled uniform noise + 2 % white noise),
    generated on the device; every frame gets its own gain / offset so that per-frame colour statistics differ (config 3)."""
    g = torch.Generator(device=dev).manual_seed(1000 + seed)
    acc = torch.zeros(n, 3, h, w, device=dev)
    amp, tot = 1.0, 0.0
    for o in range(4):
        base = torch.rand(n, 3, 8 * 2 ** o + 1, 15 * 2 ** o + 1, generator=g, device=dev)
        acc += amp * torch.nn.functional.interpolate(base, size=(h, w), mode="bilinear", align_corners=True)
        tot += amp
        amp *= 0.5
    acc /= tot
    acc += 0.02 * (torch.rand(n, 3, h, w, generator=g, device=dev) - 0.5)
    acc += torch.tensor([0.03, 0.0, -0.03], device=dev).view(1, 3, 1, 1)
    gain = 0.8 + 0.4 * torch.rand(n, 1, 1, 1, generator=g, device=dev)
    off = 0.1 * (torch.rand(n, 3, 1, 1, generator=g, device=dev) - 0.5)
    return (acc * gain + off).clamp_(0, 1).permute(0, 2, 3, 1).contiguous().to(dtype)


DUMP_PIXELS = 1 << 21          # sampled output pixels over all ranks: 2 Mi x 3 channels x 4 B = 24 MiB
DUMP_CROP = 256                # side of the full-resolution corner crops (the stencil's replicated border is in them)


def headline_outputs(out, ref_sums, rank, world):
    """What the last headline step returned, small enough to store: a fixed, seeded sample of the output pixels (the same
    positions on every run and every build), full-resolution corner crops of the rank's first and last frame, and the
    gathered reference statistics.  float32 / float64 host arrays keyed by file name."""
    B, H, W, C = out.shape
    g = torch.Generator().manual_seed(7 + rank)
    idx = torch.randint(0, B * H * W, (max(1, DUMP_PIXELS // world),), generator=g).sort().values
    arrays = {"pixels": out.view(-1, C)[idx.to(out.device)], "first_frame_top_left": out[0, :DUMP_CROP, :DUMP_CROP],
              "last_frame_bottom_right": out[-1, -DUMP_CROP:, -DUMP_CROP:], "ref_sums": ref_sums}
    return {"rank%d_%s" % (rank, k): v.cpu().numpy() for k, v in arrays.items()}


def tile_frames(base, total):
    """`total` frames from the distinct `base` frames (repeated; a per-frame offset keeps every frame's statistics distinct)"""
    n = base.shape[0]
    x = base.repeat((total + n - 1) // n, 1, 1, 1)[:total].contiguous()
    x += (torch.arange(total, device=x.device, dtype=torch.float32).view(-1, 1, 1, 1) * (0.02 / max(total, 1))).to(x.dtype)
    return x.clamp_(0, 1)


# ------------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own nodes (oracle port) for the same chain
# ------------------------------------------------------------------------------------------------------------------------
def cpu_full_chain(frames, steps, threads=None):
    """grain -> colour match -> LUT -> unsharp (numpy path) on `frames` 4K fp32 frames.  Returns (MP/s, best seconds, threads)."""
    import vrgdg_oracle as oracle
    from helpers import natural_frames
    if threads:
        torch.set_num_threads(threads)
    x = natural_frames(frames, H4K, W4K, seed=0)
    ref = natural_frames(1, H4K, W4K, seed=99)
    lut = oracle.parse_cube(LUT_FILE)
    best = None
    for _ in range(steps):
        torch.manual_seed(123)
        t0 = time.perf_counter()
        a = oracle.film_grain(x, GRAIN["intensity"], GRAIN["saturation_mix"], batch_size=4)
        b = oracle.color_match(a, ref, 1.0, 1)
        c = oracle.apply_lut(b, lut, 10.0)
        oracle.unsharp_numpy(c, SHARPEN)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return frames * H4K * W4K / 1e6 / best, best, torch.get_num_threads()


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    threads = host_threads()
    torch.set_num_threads(threads)
    sample_frames = 2
    import vrgdg_oracle as oracle
    from helpers import natural_frames
    x = natural_frames(sample_frames, H4K, W4K, seed=0)
    ref = natural_frames(1, H4K, W4K, seed=99)
    lut = oracle.parse_cube(LUT_FILE)

    def step():
        a = oracle.film_grain(x, GRAIN["intensity"], GRAIN["saturation_mix"], batch_size=4)
        b = oracle.color_match(a, ref, 1.0, 1)
        c = oracle.apply_lut(b, lut, 10.0)
        return oracle.unsharp_numpy(c, SHARPEN)
    step()
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    mps = sample_frames * H4K * W4K / 1e6 / dt
    sample = ("%d x 3840x2160 fp32 frames per step through the reference CPU nodes FastFilmGrain -> ColorMatchToReference -> VRGDG_LUTS -> "
              "FastUnsharpSharpen (numpy path), oracle port" % sample_frames)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(mps, 3), "unit": "MP/s", "n_gpus": args.gpus, "steps": steps, "warmup": 1,
        "ms_per_step": round(dt * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": round(mps, 3), "unit": "MP/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(mps, 3), "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------------------
def run_b200(args):
    rank, world, local = dist_env()
    pkg = importlib.import_module(PKG)
    numa_cpus = pkg._runtime.bind_to_gpu_numa(local)        # before any pinned allocation / first touch
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist = None
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    nv = pkg._native
    nv.load_library()
    vdist = importlib.import_module(PKG + ".dist")
    peak, peak_src = measured_peaks()
    lut = pkg.VRGDG_LUTS._parse_cube_file(LUT_FILE)
    stencil = dict(op=nv.STENCIL_BOX_UNSHARP, strength=SHARPEN, border=nv.BORDER_REPLICATE)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup):
        """W untimed + K timed calls bracketed by barrier + synchronize; device time from CUDA events on the launching stream."""
        for _ in range(warmup):
            fn()
        barrier()
        l0 = nv.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps, nv.launch_count() - l0

    # ---- headline: configs[3] shard, frames synthesised on the device ----
    first = rank * FRAMES_4K                                  # absolute index of this rank's first frame (keys the grain)
    x = tile_frames(device_natural_frames(8, H4K, W4K, seed=rank, dtype=torch.float32, dev=dev), FRAMES_4K)
    out = torch.empty_like(x)
    ref = device_natural_frames(1, H4K, W4K, seed=4242, dtype=torch.float32, dev=dev)      # the same reference frame on every rank
    chain = pkg.chain.PostChain(grain=GRAIN, colormatch=dict(ref_sums=vdist.reference_sums_distributed(ref), strength=1.0),
                                lut=dict(lut_data=lut, strength=10.0), stencil=stencil, device=dev)
    npix = FRAMES_4K * H4K * W4K
    warm = max(args.warmup, 3)

    def step():
        # the path's one collective: reference rows sharded over the ranks, 7 doubles all-gathered, folded in rank order
        chain.set_reference(ref_sums=vdist.reference_sums_distributed(ref))
        chain(x, first_frame=first, out=out)

    sampler = ClockSampler(local)
    for _ in range(warm):
        step()
    barrier()
    sampler.start()
    ms_step, launches = timed(step, args.steps, 0)
    sampler.stop_flag.set()
    # taken before the schedules and extra lines below overwrite `out`
    dump = headline_outputs(out, chain._ref_sums, rank, world) if args.dump_outputs else None
    value = world * npix / 1e6 / (ms_step / 1e3)
    tile_path = nv.last_tile_path()
    ref_sums_identical = True
    if dist is not None:                                      # every rank holds bit-identical reference statistics
        mine = chain._ref_sums.reshape(-1).contiguous()
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        ref_sums_identical = all(torch.equal(a, allr[0]) for a in allr)
    # the other schedules of the same chain, a few steps each (explains the headline; identical results up to fp32 rounding)
    alt = {}
    if not args.no_extra:
        alt_steps = max(2, min(args.steps, 5))
        chain.serial = True
        alt["f_planes_serial_one_call_ms"], _ = timed(step, alt_steps, 1)    # same kernels one after the other: what the concurrent schedule hides
        chain.serial = False
        chain.recompute = True
        alt["recompute_one_call_ms"], _ = timed(step, alt_steps, 1)          # pass 2 re-reads the frames, redraws the grain, repeats the forward Lab
        chain.split, chain.timing = True, []
        alt["recompute_three_calls_ms"], _ = timed(step, alt_steps, 1)       # round-1 schedule: statistics / parameters / apply as separate entry points
        seg = chain.timing
        alt["three_calls_moments_pass_ms"] = max_over_ranks(sum(a.elapsed_time(b) for a, b, _, _ in seg) / len(seg))
        alt["three_calls_apply_pass_ms"] = max_over_ranks(sum(c.elapsed_time(d) for _, _, c, d in seg) / len(seg))
        chain.recompute, chain.split, chain.timing = False, False, None
        alt = {k: round(v, 4) for k, v in alt.items()}

    def roofline(alg_bytes, ms, extra=None):
        ach = alg_bytes / (ms / 1e3) / 1e9
        d = {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4), "peak_source": peak_src,
             "algorithmic_bytes_per_launch": alg_bytes}
        d.update(extra or {})
        return d

    # ---- extra lines: the gather-bound chains without colour match ----
    extras = {}
    if not args.no_extra:
        ex_steps = max(3, min(args.steps, 10))
        x4 = x[:32]
        o4 = out[:32]
        c4 = pkg.chain.PostChain(grain=GRAIN, lut=dict(lut_data=lut, strength=10.0), stencil=stencil, device=dev)
        ms4, _ = timed(lambda: c4(x4, first_frame=first, out=o4), ex_steps, 3)
        n4 = 32 * H4K * W4K
        extras["grain_lut_unsharp_4k_f32"] = {
            "workload": "fused grain + 33^3 LUT + unsharp, 32 x 3840x2160 fp32 frames per GPU, one k_tile launch per step",
            "value": round(world * n4 / 1e6 / (ms4 / 1e3), 1), "unit": "MP/s", "ms_per_step": round(ms4, 4), "steps": ex_steps,
            "roofline": roofline(n4 * 24, ms4, {"kernel": "k_tile<float, grain|lut>"})}
        x2 = tile_frames(device_natural_frames(8, 1080, 1920, seed=rank, dtype=torch.float16, dev=dev), 64)
        o2 = torch.empty_like(x2)
        ms2, _ = timed(lambda: c4(x2, first_frame=rank * 64, out=o2), ex_steps, 3)
        n2 = 64 * 1080 * 1920
        tr2, st2 = recorded_traffic("configs1_f16")
        extras["configs1_grain_lut_unsharp_1080p_f16"] = {
            "workload": "configs[1]: fused grain + 33^3 LUT + unsharp, 64 x 1920x1080 fp16 frames per GPU, one k_tile launch per step",
            "value": round(world * n2 / 1e6 / (ms2 / 1e3), 1), "unit": "MP/s", "ms_per_step": round(ms2, 4), "steps": ex_steps,
            "roofline": roofline(n2 * 12, ms2, dict({"kernel": "k_tile<half, grain|lut>", "traffic": tr2}, **(st2 or {})))}
        del x2, o2, c4
        # configs[2]: colour match alone on 4K fp32 frames (256 frames over 8 GPUs = 32 per GPU) against one reference frame, the reference
        # statistics gathered over NCCL inside every step: (a) the reference's algorithm (LAB mean / std transfer, nodes.py:91-124),
        # (b) the histogram / CDF mode BASELINE.json words it as (labelled extension, parity unpinned)
        cm_only = pkg.chain.PostChain(colormatch=dict(ref_sums=vdist.reference_sums_distributed(ref), strength=1.0), device=dev)

        def cm_step():
            cm_only.set_reference(ref_sums=vdist.reference_sums_distributed(ref))
            cm_only(x4, first_frame=first, out=o4)
        ms3, _ = timed(cm_step, ex_steps, 3)
        extras["configs2_colormatch_lab_4k_f32"] = {
            "workload": "configs[2] per-GPU shard, the reference's LAB mean/std transfer: 32 x 3840x2160 fp32 frames per GPU vs one 4K reference frame "
                        "(rows sharded, 56-byte all-gather per step), vrgdg_chain_cm_apply (statistics pass + f-planes, apply pass)",
            "value": round(world * n4 / 1e6 / (ms3 / 1e3), 1), "unit": "MP/s", "ms_per_step": round(ms3, 4), "steps": ex_steps,
            "roofline": roofline(n4 * 24, ms3, {"kernel": "k_lab_moments<float, store f-planes> + k_point<float, colormatch-from-f>", "moved_bytes_per_pixel": 48})}

        def hist_step():
            ref_counts = vdist.reference_histogram_distributed(ref)
            tables = pkg.ops.histmatch_tables(pkg.ops.hist_counts(x4), ref_counts)
            pkg.ops.histmatch_apply(x4, tables, 1.0, 0.0)
        ms3h, _ = timed(hist_step, ex_steps, 3)
        extras["configs2_colormatch_histogram_4k_f32"] = {
            "workload": "configs[2] per-GPU shard, histogram / CDF transfer (extension without a reference counterpart; parity unpinned): 32 x 3840x2160 "
                        "fp32 frames per GPU vs one 4K reference frame (rows sharded, all-gather of 3 x 256 counters per rank per step)",
            "value": round(world * n4 / 1e6 / (ms3h / 1e3), 1), "unit": "MP/s", "ms_per_step": round(ms3h, 4), "steps": ex_steps,
            "roofline": roofline(n4 * 24, ms3h, {"kernel": "k_hist_counts<float> + k_histmatch_tables + k_histmatch_apply<float>", "moved_bytes_per_pixel": 36})}
        del cm_only
        # configs[4]: temporal 3-frame sharpen, 512 x 1080p fp32 frames over 4 GPUs = 128 frames per GPU (labelled extension:
        # the reference has no temporal operator); at N > 1 every step exchanges one halo frame per shard boundary (NCCL send/recv)
        x5 = tile_frames(device_natural_frames(8, 1080, 1920, seed=100 + rank, dtype=torch.float32, dev=dev), 128)

        def temporal_step():
            prev, nxt = vdist.exchange_halo_frames(x5)
            pkg.ops.temporal_sharpen(x5, SHARPEN, prev, nxt)
        ms5, _ = timed(temporal_step, ex_steps, 3)
        n5 = 128 * 1080 * 1920
        extras["configs4_temporal_sharpen_1080p_f32"] = {
            "workload": "configs[4] per-GPU shard: temporal 3-frame unsharp, 128 x 1920x1080 fp32 frames per GPU, one halo frame per shard boundary "
                        "(extension without a reference counterpart; parity unpinned)",
            "value": round(world * n5 / 1e6 / (ms5 / 1e3), 1), "unit": "MP/s", "ms_per_step": round(ms5, 4), "steps": ex_steps,
            "roofline": roofline(n5 * 24, ms5, {"kernel": "k_temporal3<float>"})}
        del x5

    # ---- end to end through the public API: pinned host frames -> pinned host frames (sub-batch) ----
    nE = min(E2E_FRAMES, FRAMES_4K)
    host_in = torch.empty((nE,) + tuple(x.shape[1:]), dtype=x.dtype, pin_memory=True)
    host_in.copy_(x[:nE])
    host_out = torch.empty_like(host_in, pin_memory=True)      # pinned once, reused every step
    e2e_steps = max(1, min(args.steps, 5))
    chunk = int(os.environ.get("VRGDG_BENCH_CHUNK", "1"))       # measured: 1 frame per chunk 3838 MP/s, 2 frames 3690 (shorter pipeline fill / drain)

    def e2e_step():
        chain.set_reference(ref_sums=vdist.reference_sums_distributed(ref))
        return chain.run_host(host_in, chunk_frames=chunk, first_frame=first, out=host_out)
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    checksum = 0.0
    for _ in range(e2e_steps):
        res = e2e_step()
        checksum += float(res[0, 0, 0, 0])                     # the device->host result is read on the host
    torch.cuda.synchronize(dev)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps)
    e2e_value = world * nE * H4K * W4K / 1e6 / (e2e_ms / 1e3)
    e2e_bytes = host_in.numel() * host_in.element_size()

    def copy_gbs(dst, src):
        torch.cuda.synchronize(dev)
        t = time.perf_counter()
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize(dev)
        return src.numel() * src.element_size() / (time.perf_counter() - t) / 1e9
    d_tmp = torch.empty_like(host_in, device=dev)
    copy_gbs(d_tmp, host_in)
    h2d, d2h = copy_gbs(d_tmp, host_in), copy_gbs(host_out, d_tmp)
    del d_tmp

    # ---- the same chain as four unchanged ComfyUI nodes on pageable host tensors (what a saved workflow pays) ----
    stock = None
    if not args.no_extra:
        nS = min(STOCK_FRAMES, FRAMES_4K)
        hx, hr = x[:nS].cpu(), ref.cpu()
        nodes = (pkg.FastFilmGrain(), pkg.ColorMatchToReference(), pkg.VRGDG_LUTS(), pkg.FastUnsharpSharpen())

        def stock_step():
            a = nodes[0].apply_grain(hx, GRAIN["intensity"], GRAIN["saturation_mix"], 4)[0]
            b = nodes[1].match_color(a, hr, 1.0, 1)[0]
            c = nodes[2].apply_lut(b, os.path.basename(LUT_FILE), "auto", 10.0)[0]
            return nodes[3].apply_unsharp(c, SHARPEN, False)[0]
        for _ in range(2):        # steady state of a workflow that is run repeatedly: torch's pinned-memory cache holds the staging and result blocks
            r = stock_step()
        del r
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            r = stock_step()
            checksum += float(r[0, 0, 0, 0])
        torch.cuda.synchronize(dev)
        st_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / 3)
        stock = {"value": round(world * nS * H4K * W4K / 1e6 / (st_ms / 1e3), 1), "unit": "MP/s", "ms_per_step": round(st_ms, 2), "frames_per_gpu": nS,
                 "api": "FastFilmGrain -> ColorMatchToReference -> VRGDG_LUTS -> FastUnsharpSharpen node classes, pageable host frames in, "
                        "host tensors between the nodes and out (what an unchanged workflow pays), third to fifth run of the workflow"}

    if rank == 0:
        alg = npix * 24                                       # 12 B read + 12 B written per fp32 pixel, SURVEY 8(d)
        tr, st = recorded_traffic("headline_apply")
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": "MP/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_gpu": FRAMES_4K, "height": H4K, "width": W4K, "frame_dtype": "f32", "lut": os.path.basename(LUT_FILE),
                       "distribution": "natural-like (4 octaves of upsampled noise + 2% white), per-frame gain / offset",
                       "parallelism": "frame-sharded dp%d; colour-match reference rows sharded, one 56-byte all-gather per step" % world,
                       "collective": ("nccl all_gather inside every step" if world > 1 else "none at N=1 (single rank computes the whole reference frame)"),
                       "ref_sums_identical_on_all_ranks": ref_sums_identical,
                       "l2": "input (12.7 GB per GPU) and output are each far larger than L2 (126 MB); no flush needed", "tile_path": tile_path,
                       "numa_bound_cpus": len(numa_cpus) if numa_cpus else None},
            "roofline": dict(roofline(alg, ms_step, {
                "kernel": "the whole step: k_lab_moments<float, grain, store f-planes> + k_moments_final + k_colormatch_params + "
                          "k_tile<float, colormatch-from-f | lut, unsharp>, 16 groups of 8 frames (vrgdg_chain_cm_apply); "
                          "per-kernel shares: profiles/ launch list",
                "moved_bytes_per_pixel": 48, "algorithmic_bytes_per_pixel": 24,
                "limiter": "not HBM: the statistics pass is bound by instruction issue / the XU (MUFU) pipe (Philox + Box-Muller, six fractional "
                           "powers per pixel), the apply pass by the L1 data pipe (three 32-byte lane accesses per pixel for the LUT cell, 83 % busy); "
                           "the two passes of neighbouring frame groups run concurrently (pipelined schedule); HBM carries 48 B/px at ~0.4 of its "
                           "peak: see profiles/README.md",
                "traffic": tr}), **(st or {})),
            "schedules_ms_per_step": dict({"f_planes_pipelined_one_call (headline)": round(ms_step, 4)}, **alt),
            "e2e": {"value": round(e2e_value, 1), "unit": "MP/s", "h2d_bytes_per_step": e2e_bytes, "d2h_bytes_per_step": e2e_bytes,
                    "ms_per_step": round(e2e_ms, 3), "steps": e2e_steps, "frames_per_gpu": nE,
                    "api": "PostChain.run_host(pinned 4K fp32 frames, chunk_frames=%d), sub-batch of %d frames per GPU" % (chunk, nE),
                    "achieved_gbs_each_way": round(e2e_bytes / (e2e_ms / 1e3) / 1e9, 2), "h2d_gbs": round(h2d, 1), "d2h_gbs": round(d2h, 1),
                    "stock_nodes": stock},
            "extra": extras,
            "gpu_launches": launches,
            "clocks": sampler.result(),
        }
        if world == 1 and not args.no_cpu:
            mps, secs, threads = cpu_full_chain(1, steps=2)
            line["cpu_baseline"] = {"value": round(mps, 3), "unit": "MP/s", "cores": threads, "kind": "port",
                                    "sample": "1 x 3840x2160 fp32 frame, best of 2, oracle port of FastFilmGrain -> ColorMatchToReference -> VRGDG_LUTS -> "
                                              "FastUnsharpSharpen (%.1f s)" % secs}
        print(json.dumps(line))
    if dump is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra lines and the stock-node leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps write a fixed sample of the last headline step's outputs "
                                                          "to DIR/<name>.npy (float32 / float64, under 40 MB), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs stores the B200 path's outputs; --impl reference has none to store")
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
        run_b200(args)


if __name__ == "__main__":
    main()
