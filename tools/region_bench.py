#!/usr/bin/env python3
"""Windows of the output image on the GPU: what they cost, and that they cost the whole-image path nothing.

  python tools/region_bench.py [--parent DIR] [--repeats R] [--steps K] [--warmup W] [--iters I]

1. With --parent (a built checkout of another commit): bench.py's `value` for this tree and that one, alternated R
   times (bench.py --gpus 1 --steps K --warmup W, its CPU baseline, end-to-end and extra sub-benchmarks off).  The
   spread between repeats of the same tree is the noise a difference has to exceed.
2. Output Gpix/s of windows through lanczos_b200_upscale_region (device buffers, CUDA events around I calls):
   - a 3840x2160 window of 3840x2160 -> 7680x4320 RGB (2x, Lanczos-3), with a left edge on the 16-byte grid (the
     static-phase kernel) and one pixel off it (the fallback);
   - a 1920x1080 viewport of a 16384x16384 RGB image at 2x, against the full-width band over the same rows (what a
     caller had to compute before windows existed), which is also checked to contain the viewport bit for bit.
The card's name and power limit are printed with the numbers.  One JSON line per measurement.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def bench_value(tree, steps, warmup):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--no-cpu-baseline", "--no-e2e", "--no-extra"]
    out = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    if out.returncode != 0 or not lines:
        raise RuntimeError("bench.py failed in %s: %s" % (tree, out.stderr[-2000:]))
    return json.loads(lines[-1])["value"]


def compare_bench(parent, repeats, steps, warmup):
    vals = {"this": [], "parent": []}
    for _ in range(repeats):
        for name, tree in (("parent", parent), ("this", ROOT)):
            vals[name].append(bench_value(tree, steps, warmup))
    res = {k: {"values": v, "median": statistics.median(v), "spread": max(v) - min(v)} for k, v in vals.items()}
    res["change"] = res["this"]["median"] / res["parent"]["median"] - 1
    return res


def image(torch, h, w, c, seed):
    """Image-like content on the device: 128 + 90 sin(0.05 x + c) cos(0.037 y) + U[-8, 7], row blocks at a time."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty((h, w, c), dtype=torch.uint8, device="cuda")
    x = torch.arange(w, device="cuda", dtype=torch.float32)
    for r0 in range(0, h, 2048):
        y = torch.arange(r0, min(h, r0 + 2048), device="cuda", dtype=torch.float32)[:, None]
        for ch in range(c):
            v = 128 + 90 * torch.sin(0.05 * x + ch)[None, :] * torch.cos(0.037 * y)
            v = v + torch.randint(-8, 8, v.shape, device="cuda", generator=g)
            out[r0:r0 + len(y), :, ch] = v.clamp(0, 255).to(torch.uint8)
    return out


def word_rect(rect, iw, c):
    """The rect widened to the right, inside the image, until its rows are whole 32-bit words (what the fast kernels
    read through their tensor map)."""
    ix, iy, w, h = rect
    while (w * c) % 4 and ix + w < iw:
        w += 1
    return ix, iy, w, h


def time_calls(torch, fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def window_rate(torch, lz, desc, full, x0, y0, w, h, iters):
    """(ms per call, output Gpix/s, kernel id, output) of one window of `full` (a device [H][W][C] image)."""
    ih, iw, c = full.shape
    ix, iy, riw, rih = word_rect(lz.region_input_rect(desc, x0, y0, w, h), iw, c)
    d_in = full[iy:iy + rih, ix:ix + riw]
    d_out = torch.empty((h, w, c), dtype=torch.uint8, device="cuda")
    ms = time_calls(torch, lambda: lz.upscale_region_device(desc, d_in, d_out, x0, y0, ix, iy), iters)
    torch.cuda.synchronize()
    lz.upscale_region_device(desc, d_in, d_out, x0, y0, ix, iy)
    torch.cuda.synchronize()
    return ms, w * h / (ms * 1e-3) / 1e9, lz.stats()["kernel_id"], d_out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", help="built checkout of the commit to compare bench.py against")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    import torch
    import lanczos_hls_b200 as lz
    gpu = card()
    print(json.dumps({"card": gpu}), flush=True)
    if args.parent:
        print(json.dumps({"bench_py": compare_bench(args.parent, args.repeats, args.steps, args.warmup), "card": gpu}),
              flush=True)

    # 3840x2160 window of config 4: 3840x2160 -> 7680x4320 RGB, 2x
    iw, ih, c = 3840, 2160, 3
    full = image(torch, ih, iw, c, 1)
    desc = lz.make_desc(iw, ih, 2 * iw, 2 * ih, c, 3, 2, 1)
    whole = torch.empty((2 * ih, 2 * iw, c), dtype=torch.uint8, device="cuda")
    lz.upscale_device(full, whole, 3, 2, 1)
    for label, x0 in (("aligned", 1920), ("unaligned", 1921)):
        ms, gpix, kid, out = window_rate(torch, lz, desc, full, x0, 1080, 3840, 2160, args.iters)
        same = bool(torch.equal(out, whole[1080:1080 + 2160, x0:x0 + 3840]))
        print(json.dumps({"case": "config 4 window 3840x2160, %s left edge (x0 = %d)" % (label, x0), "ms": ms,
                          "output_gpix_s": gpix, "kernel_id": kid, "equals_whole_image": same, "card": gpu}), flush=True)
    del full, whole

    # 1920x1080 viewport of a 16384^2 RGB image at 2x, against the full-width band over the same rows
    side = 16384
    full = image(torch, side, side, c, 2)
    desc = lz.make_desc(side, side, 2 * side, 2 * side, c, 3, 2, 1)
    y0, w, h = 12345, 1920, 1080
    ms_b, gpix_b, kid_b, band = window_rate(torch, lz, desc, full, 0, y0, 2 * side, h, args.iters)
    for label, x0 in (("aligned", 20000), ("unaligned", 20001)):
        ms_v, gpix_v, kid_v, view = window_rate(torch, lz, desc, full, x0, y0, w, h, args.iters)
        same = bool(torch.equal(view, band[:, x0:x0 + w]))
        print(json.dumps({"case": "viewport 1920x1080 of 16384^2 RGB at 2x, %s left edge (x0 = %d, y0 = %d)" % (label, x0, y0),
                          "window": {"ms": ms_v, "output_gpix_s": gpix_v, "kernel_id": kid_v},
                          "full_width_band": {"ms": ms_b, "output_gpix_s": gpix_b, "kernel_id": kid_b,
                                              "viewport_gpix_s": w * h / (ms_b * 1e-3) / 1e9},
                          "speedup": ms_b / ms_v, "window_equals_band_crop": same, "card": gpu}), flush=True)


if __name__ == "__main__":
    main()
