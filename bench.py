#!/usr/bin/env python
"""bench.py -- headline benchmark of the Lanczos hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): 1920x1080 -> 3840x2160 RGB8, 2x, Lanczos-3.  One "step" is one pass of
the hot path over a batch of `--frames` distinct synthetic frames per GPU, ONE kernel launch (the batch is ~2 GB
per GPU, far larger than the 126 MB L2, so every step streams from HBM).  Weak scaling: each GPU gets its own
batch; no data-path collective; NCCL is used only for the barrier and the max-over-ranks of the step time.

The kernel's speed depends on pixel values (the exact path re-evaluates samples the reference may truncate
differently), so the batch is a 50/50 MIX: even frames image-like (SURVEY.md 8d ii: smooth + noise), odd frames
uniform noise (8d i, the input BASELINE.md section 3 names and the worst case).  `value`, `roofline`, `e2e` and
`cpu_baseline` are all measured on that mix with the default flags; `by_content` gives the two halves alone.

Prints ONE JSON line (see the contract in the task statement):
  value        whole-job output Mpix/s, inputs resident in HBM, device-timed (CUDA events)
  roofline     HBM roofline of the dominant kernel (the step IS one launch of it), same flags and content as value
  e2e          same metric through the host-buffer C-ABI call (pinned host memory, H2D+D2H inside)
  cpu_baseline the reference's own software path (oracle/_ref) on this box's host cores
  c3, c4, c5_bands  the other BASELINE configs at their literal batch sizes (256 frames sharded over the GPUs,
               1024/8 = 128 frames per GPU, one 16384^2 image in row bands)
`--impl reference` times the CPU path alone (rank 0; other ranks exit).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# name -> (in_w, in_h, out_w, out_h, channels, a, N, D, default frames per GPU per step, label)
WORKLOADS = {
    "c2": (1920, 1080, 3840, 2160, 3, 3, 2, 1, 64, "1920x1080->3840x2160 RGB8 2x Lanczos-3 (BASELINE configs[1])"),
    "c3": (2560, 1440, 3840, 2160, 4, 3, 3, 2, 256, "2560x1440->3840x2160 RGBA8 3/2 Lanczos-3, batch of 256 frames sharded over the GPUs (BASELINE configs[2])"),
    "c4": (3840, 2160, 7680, 4320, 3, 3, 2, 1, 128, "3840x2160->7680x4320 RGB8 2x Lanczos-3, 1024 frames over 8 GPUs = 128 frames per GPU (BASELINE configs[3])"),
}
# CPU sample of the headline workload: a 1920x135 band -> 3840x270 (1/8 frame), reference compiled for it
CPU_SAMPLE_CFG = (1920, 135, 3840, 270, 2, 1, 3, 3)


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def ncu_traffic_per_frame():
    """DRAM bytes per frame of the headline kernel from the committed `ncu --set full` capture (None if absent).
    A constant from profiles/traffic.json: ncu cannot run inside the timed benchmark."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            t = json.load(fh)
        return float(t["dram_bytes_per_frame"]), t.get("source", "profiles/traffic.json")
    except Exception:
        return None, None


class ClockSampler:
    """Samples nvidia-smi clocks and throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        # median of the upper half = clocks under load (idle samples before/after drag the plain median down)
        med = sm[(len(sm) * 3) // 4] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# the reference's own CPU path (the one place outside tests/ that executes oracle/)
# ------------------------------------------------------------------------------------------------------
def run_reference_cpu(steps, warmup, threads=None):
    """The reference's own software path (full_TB.h:29-96 compiled into oracle/_ref) on host cores, on the same
    50/50 content mix as the GPU arm: even threads image-like bands, odd threads uniform noise."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle_py as O
    kind = "reference"
    cfg = CPU_SAMPLE_CFG
    iw, ih, ow, oh, n, d, a, c = cfg
    cores = threads or os.cpu_count() or 1
    have_ref = os.path.exists(O.ref_path(cfg))
    if not have_ref:
        kind = "port"

    def band(t):
        noise = O.xorshift_bytes(c * ih * iw, O.SEED + t).reshape(c, ih, iw)
        if t % 2 == 1:
            return noise
        yy, xx = np.mgrid[0:ih, 0:iw]
        img = np.stack([128 + 90 * np.sin(0.05 * xx + ch + 0.3 * t) * np.cos(0.037 * yy) for ch in range(c)])
        return np.ascontiguousarray(np.clip(img + ((noise.astype(np.int32) & 15) - 8), 0, 255).astype(np.uint8))

    imgs = [band(t) for t in range(cores)]

    def one(t):
        if have_ref:
            O.ref_expected_planar(imgs[t], cfg)
        else:  # literal per-tap-sin restatement, single thread per call like the reference
            O.expected_planar(imgs[t], ow, oh, a, n, d, fast=False)

    def step():
        ths = [threading.Thread(target=one, args=(t,)) for t in range(cores)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()

    if have_ref:
        O.ref_lib(cfg)
    for _ in range(max(0, warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    px = steps * cores * ow * oh
    sample = (f"{cores} threads x {steps} steps, each thread one 1920x135->3840x270 RGB8 band (1/8 of a frame; even threads "
              f"image-like, odd threads uniform noise: the GPU arm's 50/50 mix) through "
              f"{'oracle/_ref (reference full_TB.h:29-96 compiled as is)' if have_ref else 'the oracle literal port'}")
    return {"value": px / dt / 1e6, "unit": "Mpix/s", "cores": cores, "kind": kind, "sample": sample,
            "seconds": dt, "ms_per_step": dt / steps * 1e3}


# ------------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------------
class Ctx:
    """torch / NCCL plumbing of one rank."""

    def __init__(self, rank, local_rank, world):
        import torch
        self.torch = torch
        self.rank, self.local_rank, self.world = rank, local_rank, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.gen = torch.Generator(device=self.dev)
        self.gen.manual_seed(0x9E3779B9 + rank)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def timed(self, fn, steps, warm=3):
        """K calls of fn bracketed by barrier + synchronize, CUDA events on the launching stream, max over ranks.
        Returns ms per call."""
        torch = self.torch
        for _ in range(warm):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def fill_frames(ctx, d_in, content, frame0=0):
    """Synthetic frames in place: image-like = 128 + 90 sin(0.05x + c + 0.3f) cos(0.037y) + U[-8,7] (SURVEY.md 8d ii),
    noise = uniform bytes (8d i), mix = even frames image-like, odd frames noise."""
    torch = ctx.torch
    F, H, W, C = d_in.shape
    yy = torch.arange(H, device=ctx.dev, dtype=torch.float32).view(H, 1, 1)
    xx = torch.arange(W, device=ctx.dev, dtype=torch.float32).view(1, W, 1)
    cc = torch.arange(C, device=ctx.dev, dtype=torch.float32).view(1, 1, C)
    for f in range(F):
        if content == "noise" or (content == "mix" and f % 2 == 1):
            d_in[f] = torch.randint(0, 256, (H, W, C), dtype=torch.uint8, device=ctx.dev, generator=ctx.gen)
        else:
            base = 128 + 90 * torch.sin(0.05 * xx + cc + 0.3 * (frame0 + f)) * torch.cos(0.037 * yy)
            base += torch.randint(-8, 8, (H, W, C), device=ctx.dev, generator=ctx.gen)
            d_in[f] = base.clamp_(0, 255).to(torch.uint8)
    torch.cuda.synchronize()


def bench_batch(ctx, lz, name, frames, steps, flags=0, contents=("mix",)):
    """One BASELINE batch config on this rank's GPU: `frames` frames per GPU, one launch per step.
    Returns {content: ms per step} (max over ranks) plus the kernel id."""
    torch = ctx.torch
    iw, ih, ow, oh, ch, a, sn, sd, _, _ = WORKLOADS[name]
    d_in = torch.empty((frames, ih, iw, ch), dtype=torch.uint8, device=ctx.dev)
    d_out = torch.empty((frames, oh, ow, ch), dtype=torch.uint8, device=ctx.dev)

    def step():
        lz.upscale_batch_device(d_in, d_out, a=a, scale_n=sn, scale_d=sd, flags=flags)

    res = {}
    for content in contents:
        fill_frames(ctx, d_in, content)
        step()
        torch.cuda.synchronize()
        res[content] = ctx.timed(step, steps)
    st = lz.stats()
    del d_in, d_out
    torch.cuda.empty_cache()
    return res, st["kernel_id"], st["kernel_launches"]


DUMP_BYTES = 64 << 20


def dump_outputs(path, d_out):
    """--dump-outputs: the uint8 output batch [F][H][W][C] as float32 in path/output.npy, whole when it fits in
    DUMP_BYTES, else the same seeded sample of pixel positions (ascending raster order) in every frame, shape
    [F][P][C].  The inputs are seeded too, so two builds run with the same arguments can be compared value for value."""
    import numpy as np
    import torch
    F, H, W, C = d_out.shape
    per_frame = max(1, DUMP_BYTES // (4 * F * C))
    if H * W <= per_frame:
        out = d_out
    else:
        pos = torch.randperm(H * W, generator=torch.Generator().manual_seed(0))[:per_frame].sort().values
        out = d_out.reshape(F, H * W, C).index_select(1, pos.to(d_out.device))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "output.npy"), out.cpu().numpy().astype(np.float32))


def summarise_batch(name, frames, n_gpus, ms, peak):
    iw, ih, ow, oh, ch = WORKLOADS[name][:5]
    algo = frames * (iw * ih * ch + ow * oh * ch)
    out = {}
    for content, t in ms.items():
        out[content] = {"value": n_gpus * frames * ow * oh / (t * 1e-3) / 1e6, "unit": "Mpix/s", "ms_per_step": t,
                        "roofline_frac": algo / (t * 1e-3) / 1e9 / peak}
    return out


def bench_bands(ctx, lz, size, steps, contents=("image_like",)):
    """BASELINE configs[4]: one size x size RGB8 image upscaled x1.7 (17/10, out = floor(in*17/10)), output rows
    split into one band per GPU, each GPU holding only its own input rows + halo.  Strong scaling: the image is
    fixed, value = its output pixels / max-over-ranks step time."""
    torch = ctx.torch
    from lanczos_hls_b200.sharding import band_range
    iw = ih = size
    ow = oh = size * 17 // 10
    desc = lz.make_desc(iw, ih, ow, oh, 3, 3, 17, 10)
    r0, r1 = band_range(oh, ctx.rank, ctx.world)
    in0, inn = lz.band_input_rows(desc, r0, r1 - r0)
    d_in = torch.empty((inn, iw, 3), dtype=torch.uint8, device=ctx.dev)
    d_out = torch.empty((r1 - r0, ow, 3), dtype=torch.uint8, device=ctx.dev)

    def step():
        lz.upscale_band_device(desc, d_in, d_out, r0, r1 - r0, in0, inn)

    res = {}
    for content in contents:
        if content == "noise":
            d_in.copy_(torch.randint(0, 256, (inn, iw, 3), dtype=torch.uint8, device=ctx.dev, generator=ctx.gen))
        else:
            yy = torch.arange(in0, in0 + inn, device=ctx.dev, dtype=torch.float32).view(inn, 1, 1)
            xx = torch.arange(iw, device=ctx.dev, dtype=torch.float32).view(1, iw, 1)
            cc = torch.arange(3, device=ctx.dev, dtype=torch.float32).view(1, 1, 3)
            for a0 in range(0, inn, 1024):       # in slabs: the float temporaries of a 16384-wide band are large
                a1 = min(inn, a0 + 1024)
                d_in[a0:a1] = (128 + 90 * torch.sin(0.05 * xx + cc) * torch.cos(0.037 * yy[a0:a1])
                               + torch.randint(-8, 8, (a1 - a0, iw, 3), device=ctx.dev, generator=ctx.gen)).clamp_(0, 255).to(torch.uint8)
        step()
        torch.cuda.synchronize()
        res[content] = ctx.timed(step, steps)
    st = lz.stats()
    geo = {"iw": iw, "ih": ih, "ow": ow, "oh": oh, "in0": in0, "inn": inn, "r0": r0, "r1": r1}
    return res, st, geo, (d_in, d_out, step)


def bands_line(args, ctx, lz):
    """--workload c5: the row-band config as its own JSON line (strong scaling)."""
    torch = ctx.torch
    steps = args.steps
    sampler = ClockSampler(ctx.local_rank)
    if ctx.rank == 0:
        sampler.start()
        time.sleep(0.3)
    res, st, geo, (d_in, d_out, step) = bench_bands(ctx, lz, args.band_size, steps, contents=("image_like", "noise"))
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, d_out.unsqueeze(0))      # the noise band, the last content timed
    # a band step takes a few ms: keep the same kernel running (untimed) until the 50 ms clock sampler has seen it
    t_load = time.perf_counter()
    while time.perf_counter() - t_load < 0.5:
        step()
        torch.cuda.synchronize()
    clocks = sampler.stop() if ctx.rank == 0 else None
    iw, ih, ow, oh, inn = geo["iw"], geo["ih"], geo["ow"], geo["oh"], geo["inn"]
    rows = geo["r1"] - geo["r0"]
    # end to end: the band's input rows from pinned host memory, the band's output rows back to it
    lz.bind_host_to_device(ctx.local_rank)
    hin = lz.PinnedBuffer(inn * iw * 3)
    hout = lz.PinnedBuffer(rows * ow * 3)
    hin.array[:] = d_in.reshape(-1).cpu().numpy()
    h_in_t = torch.from_numpy(hin.array).view(inn, iw, 3)
    h_out_t = torch.from_numpy(hout.array).view(rows, ow, 3)
    e_steps = max(2, min(steps, 4))
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(e_steps):
        d_in.copy_(h_in_t, non_blocking=True)
        step()
        h_out_t.copy_(d_out, non_blocking=True)
    torch.cuda.synchronize()
    te = ctx.max_over_ranks(time.perf_counter() - t0)
    if ctx.rank != 0:
        return
    peak, peak_src = measured_hbm_peak()
    algo = iw * ih * 3 + ow * oh * 3
    ms = res["image_like"]
    achieved = algo / ctx.world / (ms * 1e-3) / 1e9      # per GPU (bands are equal to within one row)
    line = {
        "metric": "output Mpix/s", "value": ow * oh / (ms * 1e-3) / 1e6, "unit": "Mpix/s", "n_gpus": ctx.world,
        "steps": steps, "warmup": 3, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32 (f64 exact re-evaluation near integers)", "data": "synthetic",
        "config": {"workload": f"single {iw}x{ih} -> {ow}x{oh} RGB8 x1.7 (17/10) image, one row band per GPU with halo rows "
                               "(BASELINE configs[4])", "content": "image_like", "kernel_id": st["kernel_id"],
                   "l2": f"inputs larger than L2: {algo / ctx.world / 1e6:.0f} MB streamed per GPU per step"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "peak_source": peak_src, "kernel": "main kernel of the band (whole step: includes the top-rows kernel in band 0)",
                     "algorithmic_bytes_per_launch": algo / ctx.world},
        "by_content": {k: {"value": ow * oh / (v * 1e-3) / 1e6, "ms_per_step": v} for k, v in res.items()},
        "cpu_baseline": None,
        "e2e": {"value": ow * oh * e_steps / te / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": inn * iw * 3,
                "d2h_bytes_per_step": rows * ow * 3, "steps": e_steps,
                "api": "pinned host band -> lanczos_b200_upscale_band -> pinned host band"},
        "gpu_launches": st["kernel_launches"] * steps, "clocks": clocks,
    }
    print(json.dumps(line), flush=True)


def pcie_ceiling(ctx, hin, hout, d_in, d_out):
    """Plain pinned copies of the e2e buffers, both directions at once on two streams: the platform's ceiling for
    any host-buffer path on this rank while the other ranks do the same (max over ranks of the time)."""
    torch = ctx.torch
    s_up, s_dn = torch.cuda.Stream(device=ctx.dev), torch.cuda.Stream(device=ctx.dev)
    h_in_t, h_out_t = torch.from_numpy(hin.array), torch.from_numpy(hout.array)
    di, do = d_in.reshape(-1)[: hin.nbytes], d_out.reshape(-1)[: hout.nbytes]

    def both():
        with torch.cuda.stream(s_up):
            di.copy_(h_in_t, non_blocking=True)
        with torch.cuda.stream(s_dn):
            h_out_t.copy_(do, non_blocking=True)

    both()
    ctx.barrier()
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        both()
    torch.cuda.synchronize()
    dt = ctx.max_over_ranks(time.perf_counter() - t0) / reps
    return {"h2d_gbs": hin.nbytes / dt / 1e9, "d2h_gbs": hout.nbytes / dt / 1e9, "seconds_per_step_at_ceiling": dt,
            "how": "plain pinned cudaMemcpyAsync of the same buffers, H2D and D2H concurrently on two streams, slowest rank"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=0, help="frames per GPU per step (0 = workload default)")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS) + ["c5"],
                    help="c2 = headline (BASELINE configs[1]); c5 = one large image in row bands (BASELINE configs[4])")
    ap.add_argument("--band-size", type=int, default=16384, help="c5: input side length")
    ap.add_argument("--content", default="mix", choices=["mix", "noise", "image_like"],
                    help="mix (default) = even frames image-like (SURVEY 8d ii), odd frames uniform noise (8d i)")
    ap.add_argument("--e2e-frames", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the c3 / c4 / c5_bands / single-frame sub-benchmarks")
    ap.add_argument("--flags", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the output of the last one to DIR/output.npy (float32, see "
                         "dump_outputs); with several GPUs only rank 0's frames, each rank's being seeded differently")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's output: not with --impl reference")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and args.gpus > 1 and args.impl == "ours":
        # launched directly: re-exec under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    n_gpus = world

    if args.impl == "reference":
        if rank != 0:
            return
        steps = args.steps
        res = run_reference_cpu(steps, min(args.warmup, 2))
        line = {
            "impl": "reference", "metric": "output Mpix/s", "value": res["value"], "unit": "Mpix/s",
            "n_gpus": n_gpus, "steps": steps, "warmup": min(args.warmup, 2), "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS["c2"][9], "content": "mix", "sample": res["sample"]},
            "cpu_baseline": {"value": res["value"], "unit": "Mpix/s", "cores": res["cores"], "kind": res["kind"], "sample": res["sample"]},
            "e2e": {"value": res["value"], "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line), flush=True)
        return

    import numpy as np
    import torch
    import lanczos_hls_b200 as lz

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    ctx = Ctx(rank, local_rank, world)
    lz.lib()
    if args.workload == "c5":
        bands_line(args, ctx, lz)
        ctx.close()
        return

    name = args.workload
    IN_W, IN_H, OUT_W, OUT_H, CH, A, SN, SD, DEF_FRAMES, WORKLOAD = WORKLOADS[name]
    if name == "c3" and args.frames <= 0:
        args.frames = max(1, DEF_FRAMES // n_gpus)       # 256 frames sharded over the GPUs
    F = args.frames if args.frames > 0 else DEF_FRAMES
    algo_per_frame = IN_W * IN_H * CH + OUT_W * OUT_H * CH      # 31,104,000 for c2 (SURVEY.md 8d)
    px_per_frame = OUT_W * OUT_H
    warmup = max(args.warmup, 3)
    dev = ctx.dev
    peak, peak_src = measured_hbm_peak()

    d_in = torch.empty((F, IN_H, IN_W, CH), dtype=torch.uint8, device=dev)
    d_out = torch.empty((F, OUT_H, OUT_W, CH), dtype=torch.uint8, device=dev)

    def step(flags=args.flags):
        lz.upscale_batch_device(d_in, d_out, a=A, scale_n=SN, scale_d=SD, flags=flags)

    # the two halves alone, then the mix (which stays in d_in for everything that follows)
    by_content = {}
    others = [c for c in ("image_like", "noise") if c != args.content]
    for content in others:
        fill_frames(ctx, d_in, content)
        step()
        torch.cuda.synchronize()
        t = ctx.timed(step, max(3, min(args.steps, 20)))
        by_content[content] = {"value": n_gpus * F * px_per_frame / (t * 1e-3) / 1e6, "unit": "Mpix/s", "ms_per_step": t,
                               "roofline_frac": F * algo_per_frame / (t * 1e-3) / 1e9 / peak}
    fill_frames(ctx, d_in, args.content)
    step()
    step(args.flags | lz.FLAG_NO_ALIAS)   # builds the second plan (tables + upload) outside every timed region
    torch.cuda.synchronize()
    step()
    launches_per_step = lz.stats()["kernel_launches"]
    kernel_id = lz.stats()["kernel_id"]
    for _ in range(warmup):
        step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    ctx.barrier()
    ms_per_step = ctx.max_over_ranks(e0.elapsed_time(e1)) / args.steps
    ms_local = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_out)       # before the tolerance-mode steps below overwrite d_out
    value = n_gpus * F * px_per_frame / (ms_per_step * 1e-3) / 1e6
    by_content[args.content] = {"value": value, "unit": "Mpix/s", "ms_per_step": ms_per_step,
                                "roofline_frac": F * algo_per_frame / (ms_local * 1e-3) / 1e9 / peak}

    # ---- tolerance mode of the north star ("at most 1 LSB, exact-match fraction stated"): V pass in plain fp32 ----
    tol = None
    if not (args.flags & lz.FLAG_TOLERANCE_1LSB):
        tflags = args.flags | lz.FLAG_TOLERANCE_1LSB
        ref_out = d_out.clone() if F * px_per_frame * CH <= (4 << 30) else None
        if ref_out is not None:
            step()
            ref_out.copy_(d_out)
        tol_ms = ctx.timed(lambda: step(tflags), args.steps)
        tol = {"flag": "LANCZOS_FLAG_TOLERANCE_1LSB", "value": n_gpus * F * px_per_frame / (tol_ms * 1e-3) / 1e6,
               "unit": "Mpix/s", "ms_per_step": tol_ms, "content": args.content,
               "roofline_frac": F * algo_per_frame / (tol_ms * 1e-3) / 1e9 / peak,
               "note": "H pass bit-exact, V pass plain fp32: every byte within 1 LSB of the reference"}
        if ref_out is not None:
            neq = (d_out != ref_out)
            tol["exact_match_fraction"] = 1.0 - neq.float().mean().item()
            tol["max_abs_diff"] = int((d_out.to(torch.int16) - ref_out.to(torch.int16)).abs().max().item())
            del neq, ref_out

    # ---- BASELINE configs[1] read literally: ONE frame per call (lanczos_b200_upscale), the frames of the batch in
    # turn so the working set stays larger than L2; on one stream and round-robin over four ----
    single = None
    if not args.no_extra:
        import ctypes as C
        L = lz.lib()
        desc = lz.make_desc(IN_W, IN_H, OUT_W, OUT_H, CH, A, SN, SD, flags=args.flags)
        in_fs, out_fs = d_in.stride(0), d_out.stride(0)
        in0, out0 = d_in.data_ptr(), d_out.data_ptr()
        ptrs = [(C.c_void_p(in0 + f * in_fs), C.c_void_p(out0 + f * out_fs)) for f in range(F)]
        streams = [torch.cuda.Stream(device=dev) for _ in range(4)]
        sp = [C.c_void_p(st.cuda_stream) for st in streams]
        dref = C.byref(desc)
        single = {"call": "lanczos_b200_upscale, one frame per launch, frames of the batch in turn", "content": args.content}
        rounds = max(2, min(args.steps, 10))
        desc_ind = lz.make_desc(IN_W, IN_H, OUT_W, OUT_H, CH, A, SN, SD, flags=args.flags | lz.FLAG_INDEPENDENT)
        image_like = ptrs[0::2] if args.content == "mix" else ptrs     # even frames of the mix are the image-like ones
        for key, ns, dr, pp in (("streams_1", 1, dref, ptrs), ("streams_4", 4, dref, ptrs),
                                ("streams_1_independent_flag", 1, C.byref(desc_ind), ptrs),
                                ("image_like_frames_streams_1", 1, dref, image_like),
                                ("image_like_frames_streams_1_independent_flag", 1, C.byref(desc_ind), image_like)):
            def run():
                i = 0
                for _ in range(rounds):
                    for pi, po in pp:
                        L.lanczos_b200_upscale(dr, pi, po, local_rank, sp[i % ns])
                        i += 1
            run()
            ctx.barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(streams[0])
            for st in streams[1:ns]:
                st.wait_event(s0)
            run()
            for st in streams[1:ns]:
                streams[0].wait_stream(st)
            s1.record(streams[0])
            ctx.barrier()
            us = ctx.max_over_ranks(s0.elapsed_time(s1)) * 1e3 / (rounds * len(pp))
            single[key] = {"value": n_gpus * px_per_frame / (us * 1e-6) / 1e6, "unit": "Mpix/s", "us_per_frame": us}
        single["independent_flag"] = ("LANCZOS_FLAG_INDEPENDENT: the caller declares the frames independent; calls on ONE stream are "
                                      "launched with programmatic dependent launch and overlap like the frames of a batch")

    clocks = sampler.stop() if rank == 0 else None      # sampled over the timed device loops above

    # ---- end to end through the host-buffer C-ABI call (pinned host memory) ----
    e2e = None
    if not args.no_e2e:
        Fe = min(args.e2e_frames, F)
        numa_cpus = lz.bind_host_to_device(local_rank)      # pinned buffers below land next to this rank's GPU
        hin = lz.PinnedBuffer(Fe * IN_H * IN_W * CH)
        hout = lz.PinnedBuffer(Fe * OUT_H * OUT_W * CH)
        hin.array[:] = d_in[:Fe].reshape(-1).cpu().numpy()
        h_in = hin.array.reshape(Fe, IN_H, IN_W, CH)
        h_out = hout.array.reshape(Fe, OUT_H, OUT_W, CH)
        e_steps = max(3, min(args.steps, 8))
        lz.upscale(h_in, OUT_W, OUT_H, a=A, scale_n=SN, scale_d=SD, flags=args.flags, device=local_rank, out=h_out)
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            lz.upscale(h_in, OUT_W, OUT_H, a=A, scale_n=SN, scale_d=SD, flags=args.flags, device=local_rank, out=h_out)
        torch.cuda.synchronize()
        dt = ctx.max_over_ranks(time.perf_counter() - t0)
        ceiling = pcie_ceiling(ctx, hin, hout, d_in, d_out)
        e2e = {"value": n_gpus * Fe * e_steps * px_per_frame / dt / 1e6, "unit": "Mpix/s",
               "h2d_bytes_per_step": Fe * IN_H * IN_W * CH, "d2h_bytes_per_step": Fe * OUT_H * OUT_W * CH,
               "frames_per_step": Fe, "steps": e_steps, "ms_per_step": dt / e_steps * 1e3, "content": args.content,
               "api": "lanczos_b200_upscale_host (pinned host buffers, 3 streams)",
               "numa_bound_cpus": len(numa_cpus) if numa_cpus else 0,
               "pcie_ceiling": ceiling, "pcie_ceiling_gbs": ceiling["h2d_gbs"] + ceiling["d2h_gbs"],
               "frac_of_pcie_ceiling": ceiling["seconds_per_step_at_ceiling"] / (dt / e_steps)}
        hin.free()
        hout.free()

    del d_in, d_out
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs at their literal batch sizes (device-timed, same 50/50 mix) ----
    extra = {}
    if not args.no_extra and name == "c2":
        sub_steps = max(3, min(args.steps, 10))
        for sub in ("c3", "c4"):
            frames = max(1, WORKLOADS[sub][8] // n_gpus) if sub == "c3" else WORKLOADS[sub][8]
            ms, kid, _ = bench_batch(ctx, lz, sub, frames, sub_steps, flags=args.flags, contents=("mix", "image_like"))
            extra[sub] = {"workload": WORKLOADS[sub][9], "frames_per_gpu": frames, "kernel_id": kid,
                          "scaling": "strong (256 frames in total)" if sub == "c3" else "weak (128 frames per GPU)",
                          "by_content": summarise_batch(sub, frames, n_gpus, ms, peak)}
            extra[sub].update(extra[sub]["by_content"]["mix"])
        res, st, geo, keep = bench_bands(ctx, lz, args.band_size, max(3, min(args.steps, 5)), contents=("image_like", "noise"))
        del keep
        torch.cuda.empty_cache()
        algo5 = geo["iw"] * geo["ih"] * 3 + geo["ow"] * geo["oh"] * 3
        extra["c5_bands"] = {"workload": f"single {geo['iw']}x{geo['ih']} -> {geo['ow']}x{geo['oh']} RGB8 x1.7 (17/10), one row band per GPU "
                                         "with its own halo rows (BASELINE configs[4])", "scaling": "strong", "kernel_id": st["kernel_id"],
                             "by_content": {k: {"value": geo["ow"] * geo["oh"] / (v * 1e-3) / 1e6, "unit": "Mpix/s", "ms_per_step": v,
                                                "roofline_frac_per_gpu": algo5 / n_gpus / (v * 1e-3) / 1e9 / peak} for k, v in res.items()}}
        extra["c5_bands"].update(extra["c5_bands"]["by_content"]["image_like"])

    if rank != 0:
        ctx.close()
        return

    achieved = F * algo_per_frame / (ms_local * 1e-3) / 1e9
    traffic_pf, traffic_src = ncu_traffic_per_frame() if name == "c2" else (None, None)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic_pf * F if traffic_pf else None, "traffic_source": traffic_src, "peak_source": peak_src,
                "kernel": "main fused H->V kernel = the whole step (one launch per step, same flags and content as `value`)",
                "kernel_ms": ms_local, "algorithmic_bytes_per_launch": F * algo_per_frame,
                "by_content": {k: v["roofline_frac"] for k, v in by_content.items()}}
    cpu = None
    if n_gpus == 1 and not args.no_cpu_baseline and name == "c2":
        r = run_reference_cpu(2, 0)
        cpu = {"value": r["value"], "unit": "Mpix/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
    line = {
        "metric": "output Mpix/s", "value": value, "unit": "Mpix/s", "n_gpus": n_gpus, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if name == "c3" else "weak",
        "vs_baseline": None, "dtype": "f32 (f64 exact re-evaluation near integers)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_gpu_per_step": F, "content": args.content,
                   "content_note": "mix = even frames image-like (smooth + noise), odd frames uniform noise; see by_content",
                   "l2": f"inputs larger than L2: {F * algo_per_frame / 1e6:.0f} MB streamed per GPU per step",
                   "kernel_id": kernel_id, "flags": args.flags},
        "by_content": by_content,
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "tolerance_mode": tol,
        "single_frame_launches": single,
        "gpu_launches": launches_per_step * args.steps, "clocks": clocks,
    }
    line.update(extra)
    print(json.dumps(line), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
