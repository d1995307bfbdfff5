"""Every kernel instance the library compiles, launched at least once and checked against the reference.

Each template instance (a kernel family x channels x ratio x taps x exact/tolerance mode x 64/32-bit output stores) is
separate machine code with its own branches and register allocation, so a bug can live in one instance only.  CASES
maps every instance, as `nm -C` prints it, to a call that launches it:

  - the CPU test reads the symbols of the built library and requires that the set of kernels equals the keys of CASES,
    so a new instance without a case (or a case for an instance that no longer exists) fails without a GPU;
  - the GPU test runs each case and asserts the kernel id the library reports and, for the v6 family, which of its
    64-bit or 32-bit store variants the layout selects (restated from launch_v6, see st64()).

Content: for every specialised instance the near-tie H and V images of tests/test_near_ties.py for its ratio and `a`,
and a patchwork of image-like, noise and dark patches several strips wide and several segments tall.  Exact mode
(MODE 0) must be bit-exact against the oracle.  Tolerance mode (MODE 1) is checked against a float64 restatement of the
reference for what include/lanczos_b200.h promises: the row pass exact, phase-0 rows copies of their centre row, and
interpolated samples plain fp32 sums that may differ from the reference only next to an integer.  Every output buffer
is surrounded by canary bytes (before the base, in the row padding, between frames, after the last row) that must
survive the call.
"""
import collections
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import test_near_ties as NTT
from test_gpu_parity import patchwork_hwc

# ---- the cases -------------------------------------------------------------------------------------------------

Case = collections.namedtuple("Case", "family c a n d mode kid st64 bp")

# LZ6_CASE list of launch_v6 (lanczos_hls_b200/csrc/lanczos_v6.cu): kernel id, C, a, N, D, PH, KM
V6 = [(1, 3, 3, 2, 1, 8, 17), (2, 4, 3, 2, 1, 6, 17), (3, 4, 3, 3, 2, 4, 17), (4, 3, 2, 2, 1, 8, 0),
      (8, 1, 3, 2, 1, 24, 17), (9, 1, 3, 3, 2, 16, 17), (10, 1, 2, 2, 1, 24, 0)]
# LZD_CASE list of launch_dyn (lanczos_dyn.cu): kernel id, C, a, N, D
DYN = [(5, 3, 3, 17, 10), (6, 3, 3, 3, 2), (7, 3, 3, 3, 1), (11, 1, 3, 17, 10), (12, 3, 2, 3, 1), (13, 1, 2, 3, 1),
       (14, 3, 3, 4, 1), (15, 1, 3, 3, 1), (16, 3, 3, 5, 3), (17, 3, 3, 7, 4), (18, 2, 3, 2, 1), (19, 3, 4, 2, 1),
       (20, 3, 1, 2, 1), (21, 4, 3, 3, 1), (22, 4, 3, 4, 1), (23, 3, 2, 3, 2), (24, 1, 3, 4, 1)]
# HLS_CASE list of launch_hls (lanczos_hls.cu), bit precision 8: C, a, N, MASK
HLS_TILE = [(3, 3, 2, 4), (4, 3, 2, 4), (1, 3, 2, 4), (3, 2, 2, 0), (3, 3, 4, 4), (3, 2, 4, 0)]


def _cases():
    cases = {}
    for (kid, c, a, n, d, ph, km) in V6:
        for mode in (0, 1):
            for st in (True, False):
                sig = "lanczos_v6_kernel<%d, %d, %d, %d, %d, %d, %d, %s>" % (c, a, n, d, ph, km, mode, str(st).lower())
                cases[sig] = Case("v6", c, a, n, d, mode, kid, st, None)
    for (kid, c, a, n, d) in DYN:
        for mode in (0, 1):
            cases["lanczos_dyn_kernel<%d, %d, %d, %d, %d>" % (c, a, n, d, mode)] = Case("dyn", c, a, n, d, mode, kid, None, None)
    # FLAG_GENERIC_KERNEL, one ratio per channel count
    for (c, a, n, d) in [(1, 3, 4, 1), (2, 3, 5, 3), (3, 2, 17, 10), (4, 3, 7, 4)]:
        cases["lanczos_generic_kernel<%d>" % c] = Case("generic", c, a, n, d, 0, 0, None, None)
    # the in-place top rows of a dyn-kernel call with default flags: a second launch
    cases["lanczos_alias_rows_kernel"] = Case("alias", 3, 3, 3, 2, 0, 6, None, None)
    for (c, a, n, mask) in HLS_TILE:
        cases["lanczos_hls_tile_kernel<%d, %d, %d, %d>" % (c, a, n, mask)] = Case("hls", c, a, n, 1, 0, 101, None, 8)
    # configurations without a tiled instance: the generic HLS kernel
    for (c, a, n, bp) in [(1, 3, 3, 8), (2, 3, 2, 8), (3, 3, 2, 10), (4, 2, 2, 8)]:
        cases["lanczos_hls_kernel<%d>" % c] = Case("hls", c, a, n, 1, 0, 100, None, bp)
    # the packed-word stream shim unpacks and packs on the device around the upscale
    for sig in ("words_to_rgb_kernel", "rgb_to_words_kernel"):
        cases[sig] = Case("stream", 3, 3, 2, 1, 0, 1, None, None)
    return cases


CASES = _cases()

# host functions whose names end in _kernel: the Lanczos weight L(x) of plan.cpp
NOT_KERNELS = {"ref_kernel"}


def kernel_symbols(path):
    """Instance signatures (name<template arguments>) of every *_kernel symbol of the library, as `nm -C` prints them."""
    out = subprocess.run(["nm", "-C", path], capture_output=True, text=True, check=True).stdout
    sigs = set()
    for line in out.splitlines():
        m = re.search(r"(\w+_kernel)(<[^()]*>)?\(", line)
        if m and m.group(1) not in NOT_KERNELS:
            sigs.add(m.group(1) + (m.group(2) or ""))
    return sigs


def test_every_kernel_instance_has_a_case(lz):
    sigs = kernel_symbols(lz.lib_path())
    assert sigs == set(CASES), {"without a case": sorted(sigs - set(CASES)), "not in the library": sorted(set(CASES) - sigs)}
    assert len(sigs) == 79


def st64(row_bytes, out_pitch, out_addr, frames, out_frame_stride):
    """The store-width predicate of launch_v6 (lanczos_hls_b200/csrc/lanczos_v6.cu): 64-bit V-pass stores only when the
    output row bytes, the pitch, the base address and (batches) the frame stride are all multiples of 8."""
    return (row_bytes % 8 == 0 and out_pitch % 8 == 0 and out_addr % 8 == 0
            and (frames <= 1 or out_frame_stride % 8 == 0))


def test_store_predicate_of_the_layouts():
    """The layouts used below select the store variant they are meant to (the GPU test checks it on real addresses)."""
    for rb in (480, 1920, 83040):
        assert st64(rb, rb, 4096, 1, 0)
        assert not st64(rb, rb + 4, 4096, 1, 0)                 # pitch
        assert not st64(rb, rb, 4096 + 4, 1, 0)                 # base
        assert not st64(rb, rb, 4096, 3, rb * 10 + 4)           # batch
        assert st64(rb, rb, 4096, 1, rb * 10 + 4)               # a frame stride is not read for one frame
    assert not st64(189 * 4, 189 * 4, 4096, 1, 0)              # id 3 natural: 126 -> 189 pixels of 4 bytes
    assert not st64(252, 252, 4096, 1, 0)                      # id 9 natural: 168 -> 252 one-byte pixels


# ---- content ---------------------------------------------------------------------------------------------------

PATCH_H = 120                 # input rows of a patchwork (a multiple of every D served)
NATURAL_W = {3: 126, 9: 168}  # widths whose output rows end in half a 64-bit word (the last lane stores one word)


def patch_width(c, n, d):
    """Input width of a patchwork: whole 32-bit input words, output rows a multiple of 8 bytes but not of a 256-byte
    strip (a partial last strip), at least three strips."""
    w = d
    while True:
        ob = w * n // d * c
        if w % d == 0 and (w * c) % 4 == 0 and ob % 8 == 0 and ob % 256 != 0 and ob >= 700:
            return w
        w += d


def patchwork(oracle, c, n, d, seed, w=None):
    w = w or patch_width(c, n, d)
    return patchwork_hwc(oracle, PATCH_H, w, c, seed=seed, band=13, col=37)


def contents(oracle, case):
    """(name, frames, planted windows, output layout) for a specialised instance.  The v6 32-bit-store instances get a
    layout that forces them: a padded pitch, an output base 4 bytes past an 8-byte boundary, a batch with an odd frame
    stride, or (ids 3 and 9) the natural width whose rows end in half a word."""
    c, a, n, d, kid = case.c, case.a, case.n, case.d, case.kid
    h, hp = _cached(("h", c, a, n, d), lambda: NTT.h_image(oracle, n, d, a, c, seed=100 + kid))
    v, vp = _cached(("v", c, a, n, d), lambda: NTT.v_image(oracle, n, d, a, c, seed=100 + kid))
    frames = [patchwork(oracle, c, n, d, seed=200 + kid + f) for f in range(3)]
    narrow = case.st64 is False
    out = [("near-tie H", [h], hp, "pitch" if narrow else "dense"),
           ("near-tie V", [v], vp, "base" if narrow else "dense"),
           ("patchwork", frames, [], "batch" if narrow else "dense")]
    if narrow and kid in NATURAL_W:
        out.append(("patchwork, natural width", [patchwork(oracle, c, n, d, seed=300 + kid, w=NATURAL_W[kid])], [], "natural"))
    return out


_CACHE = {"config": None}


def _cached(key, make):
    """Images and their references are shared by the cases of one configuration (adjacent in CASES); the cache holds
    one configuration at a time."""
    config = key[1:5]
    if _CACHE["config"] != config:
        _CACHE.clear()
        _CACHE["config"] = config
    if key not in _CACHE:
        _CACHE[key] = make()
    return _CACHE[key]


def oracle_ref(oracle, img, a, n, d, variant):
    ow, oh = oracle.out_dims(img.shape[1], img.shape[0], n, d)
    key = ("oracle", img.shape[2], a, n, d, img.shape, variant, oracle.fnv1a64(img))
    return _cached(key, lambda: oracle.upscale(img, ow, oh, a, n, d, variant=variant))


def restated(oracle, img, a, n, d):
    """Planar (reference, row pass, column sums) of the ping-pong (CLEAN) reference, in float64."""
    ow, oh = oracle.out_dims(img.shape[1], img.shape[0], n, d)
    key = ("restated", img.shape[2], a, n, d, img.shape, oracle.fnv1a64(img))
    return _cached(key, lambda: NTT.restate_planar(NTT.to_planar(img), ow, oh, a, n, d, clean=True, parts=True))


# ---- launching with canaries -----------------------------------------------------------------------------------

CANARY = 0xA7
LEAD = 64                     # canary bytes before the output base


def out_layout(layout, row_bytes, rows, frames):
    """(pitch, frame stride, offset of the base in the buffer, buffer bytes); two canary rows follow the last row."""
    pitch = row_bytes + (4 if layout == "pitch" else 0)
    fstride = pitch * rows + (4 if layout == "batch" else 0)
    lead = LEAD + (4 if layout == "base" else 0)
    return pitch, fstride, lead, lead + fstride * (frames - 1) + pitch * rows + 2 * pitch + 64


def launch(torch, lz, case, frames, layout, flags, stats=False):
    """Run one specialised-kernel call on `frames` (list of [H][W][C]); returns (outputs, stats).  Checks the kernel
    id, the store variant of v6 instances and every canary byte."""
    c, a, n, d = case.c, case.a, case.n, case.d
    ih, iw = frames[0].shape[:2]
    ow, oh = iw * n // d, ih * n // d
    nf = len(frames)
    in_pitch = -(-iw * c // 16) * 16              # the TMA kernels need 16-byte input rows
    src = np.zeros((nf, ih, in_pitch), np.uint8)
    for f, img in enumerate(frames):
        src[f, :, :iw * c] = img.reshape(ih, iw * c)
    d_in = torch.from_numpy(src).cuda()
    rb = ow * c
    pitch, fstride, lead, total = out_layout(layout, rb, oh, nf)
    buf = torch.full((total,), CANARY, dtype=torch.uint8, device="cuda")
    assert buf.data_ptr() % 16 == 0 and d_in.data_ptr() % 16 == 0
    out_addr = buf.data_ptr() + lead
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, in_pitch, pitch, flags)
    L = lz.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lz.enable_stats(stats)
    try:
        if nf == 1:
            rc = L.lanczos_b200_upscale(C.byref(desc), C.c_void_p(d_in.data_ptr()), C.c_void_p(out_addr), 0, stream)
        else:
            rc = L.lanczos_b200_upscale_batch(C.byref(desc), C.c_void_p(d_in.data_ptr()), C.c_void_p(out_addr), nf,
                                              ih * in_pitch, fstride, 0, stream)
        torch.cuda.synchronize()
        st = lz.stats()
    finally:
        lz.enable_stats(False)
    assert rc == 0, (rc, L.lanczos_b200_strerror(rc))
    assert st["kernel_id"] == case.kid, (st, case)
    if case.family == "v6":
        assert st64(rb, pitch, out_addr, nf, fstride) == case.st64, (layout, rb, pitch, out_addr % 8, fstride)
    host = buf.cpu().numpy()
    view = np.lib.stride_tricks.as_strided(host[lead:], shape=(nf, oh, rb), strides=(fstride, pitch, 1))
    outs = [np.array(view[f]).reshape(oh, ow, c) for f in range(nf)]
    canary = np.ones(total, bool)
    np.lib.stride_tricks.as_strided(canary[lead:], shape=(nf, oh, rb), strides=(fstride, pitch, 1))[...] = False
    hit = np.nonzero(canary & (host != CANARY))[0]
    assert len(hit) == 0, ("canary bytes overwritten", layout, len(hit), [(int(i) - lead) for i in hit[:8]])
    return outs, st


# ---- checks ----------------------------------------------------------------------------------------------------

def check_exact(torch, lz, oracle, case, name, frames, planted, layout):
    a, n, d = case.a, case.n, case.d
    got, st = launch(torch, lz, case, frames, layout, 0, stats=True)
    for f, img in enumerate(frames):
        want = oracle_ref(oracle, img, a, n, d, oracle.VERBATIM)
        bad = np.argwhere(got[f] != want)
        assert len(bad) == 0, (name, layout, "frame", f, len(bad), bad[:8].tolist())
    assert st["strict_samples"] >= NTT.strict_floor(planted), (name, st, NTT.strict_floor(planted))
    got, _ = launch(torch, lz, case, frames, layout, lz.FLAG_NO_ALIAS)
    for f, img in enumerate(frames):
        bad = np.argwhere(got[f] != oracle_ref(oracle, img, a, n, d, oracle.CLEAN))
        assert len(bad) == 0, (name, layout, "no alias, frame", f, len(bad), bad[:8].tolist())


# Tolerance mode sums the 2a vertical taps in fp32 from fp32 weights.  With bytes <= 255 and sum |w| < 1.3 the
# accumulated rounding error stays below the guards the exact path needs for the same sums -- about 1.3e-4 for the
# served ratios (DESIGN.md section 3) -- so a truncation can differ from the reference's only where the reference's
# double sum lies that close to an integer.  delta = 2^-10 (~9.8e-4) leaves a factor of 7 over that bound and is
# still far too tight for a rounding or a wrong-row bug, which move samples by up to 0.5 or more.
DELTA = 2.0 ** -10


def check_tolerance_clean(got, ref, mid, sums, n, d, what):
    """(a) phase-0 rows are the row pass at the centre row, byte for byte; (b) interpolated samples equal the reference
    except within DELTA of an integer, and there differ by 1 at most.  Returns the exact-match fraction."""
    g = NTT.to_planar(got)
    c, oh, ow = g.shape
    yy = np.arange(oh)
    ph0 = (yy * d) % n == 0
    bad = np.argwhere(g[:, ph0] != mid[:, yy[ph0] * d // n])
    assert len(bad) == 0, (what, "phase-0 rows are not copies of their centre rows", len(bad), bad[:8].tolist())
    rows = yy[~ph0]
    n_diff = n_all = 0
    for r0 in range(0, len(rows), 1024):
        rr = rows[r0:r0 + 1024]
        diff = g[:, rr].astype(np.int16) - ref[:, rr]
        s = sums[:, rr]
        near = np.abs(s - np.rint(s)) < DELTA
        wrong = (np.abs(diff) > 1) | ((diff != 0) & ~near)
        n_diff += int((diff != 0).sum())
        n_all += diff.size
        if wrong.any():
            i = np.argwhere(wrong)[:8]
            detail = [(int(ch), int(rr[y]), int(x), int(diff[ch, y, x]), float(s[ch, y, x])) for ch, y, x in i]
            pytest.fail("%s: interpolated samples off by more than fp32 rounding next to an integer allows: %d of %d "
                        "differ (exact-match fraction %.6f); (channel, row, column, diff, double sum): %s"
                        % (what, int(wrong.sum()), n_all, 1 - n_diff / n_all, detail))
    return 1 - n_diff / max(n_all, 1)


def check_tolerance(torch, lz, oracle, case, name, frames, layout):
    a, n, d = case.a, case.n, case.d
    got, _ = launch(torch, lz, case, frames, layout, lz.FLAG_TOLERANCE_1LSB | lz.FLAG_NO_ALIAS)
    for f, img in enumerate(frames):
        ref, mid, sums = restated(oracle, img, a, n, d)
        check_tolerance_clean(got[f], ref, mid, sums, n, d, "%s frame %d (%s)" % (name, f, layout))
    got, _ = launch(torch, lz, case, frames, layout, lz.FLAG_TOLERANCE_1LSB)
    for f, img in enumerate(frames):
        want = oracle_ref(oracle, img, a, n, d, oracle.VERBATIM)
        dev = np.abs(got[f].astype(np.int16) - want)
        assert dev.max() <= 1, (name, layout, "frame", f, int(dev.max()), np.argwhere(dev > 1)[:8].tolist())


def test_restatement_with_parts_equals_the_oracle(oracle):
    """The tolerance checks read the restatement's row pass and column sums: its output stays pinned to the oracle, its
    column sums quantise to its output, and the check accepts the promised result and rejects a rounding one."""
    for (c, a, n, d) in [(3, 3, 17, 10), (1, 2, 3, 1), (4, 3, 3, 2)]:
        img = patchwork(oracle, c, n, d, seed=7)[:40]
        ow, oh = oracle.out_dims(img.shape[1], img.shape[0], n, d)
        ref, mid, sums = NTT.restate_planar(NTT.to_planar(img), ow, oh, a, n, d, clean=True, parts=True)
        assert np.array_equal(NTT.to_interleaved(ref), oracle.upscale(img, ow, oh, a, n, d, variant=oracle.CLEAN))
        assert np.array_equal(NTT.NT.quantise(sums), ref)
        full = NTT.restate_planar(NTT.to_planar(img), ow, oh, a, n, d, clean=False, parts=True)[0]
        assert np.array_equal(NTT.to_interleaved(full), oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM))
        yy = np.arange(oh)
        ph0 = (yy * d) % n == 0
        promised = ref.copy()
        promised[:, ph0] = mid[:, yy[ph0] * d // n]
        assert check_tolerance_clean(NTT.to_interleaved(promised), ref, mid, sums, n, d, "promised") == 1.0
        rounded = promised.copy()
        rounded[:, ~ph0] = np.clip(np.floor(sums[:, ~ph0] + 0.5), 0, 255).astype(np.uint8)
        with pytest.raises(pytest.fail.Exception):
            check_tolerance_clean(NTT.to_interleaved(rounded), ref, mid, sums, n, d, "rounded")
        if d == 1:
            shifted = promised.copy()
            shifted[:, ph0] = mid[:, np.maximum(yy[ph0] * d // n - 1, 0)]
            with pytest.raises(AssertionError):
                check_tolerance_clean(NTT.to_interleaved(shifted), ref, mid, sums, n, d, "wrong centre row")


# ---- GPU -------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def run_small(torch, lz, img, ow, oh, case, flags):
    d_in = torch.from_numpy(img).cuda()
    d_out = torch.full((oh, ow, img.shape[2]), CANARY, dtype=torch.uint8, device="cuda")
    lz.upscale_device(d_in, d_out, a=case.a, scale_n=case.n, scale_d=case.d, flags=flags)
    torch.cuda.synchronize()
    return d_out.cpu().numpy(), lz.stats()


@pytest.mark.gpu
@pytest.mark.parametrize("sig", list(CASES))
def test_instance(torch_cuda, lz, oracle, sig):
    torch = torch_cuda
    case = CASES[sig]
    c, a, n, d = case.c, case.a, case.n, case.d
    if case.family in ("v6", "dyn"):
        for (name, frames, planted, layout) in contents(oracle, case):
            if case.mode == 0:
                check_exact(torch, lz, oracle, case, name, frames, planted, layout)
            else:
                check_tolerance(torch, lz, oracle, case, name, frames, layout)
    elif case.family == "generic":
        img = patchwork_hwc(oracle, 37, 61, c, seed=c, band=7, col=11)
        ow, oh = oracle.out_dims(61, 37, n, d)
        for flags, variant in ((0, oracle.VERBATIM), (lz.FLAG_NO_ALIAS, oracle.CLEAN)):
            got, st = run_small(torch, lz, img, ow, oh, case, lz.FLAG_GENERIC_KERNEL | flags)
            assert st["kernel_id"] == 0, st
            assert np.array_equal(got, oracle.upscale(img, ow, oh, a, n, d, variant=variant))
    elif case.family == "alias":
        img = patchwork(oracle, c, n, d, seed=9)
        got, st = launch(torch, lz, case, [img], "dense", 0)
        assert st["kernel_launches"] == 2 and st["alias_rows"] > 0, st
        assert np.array_equal(got[0], oracle_ref(oracle, img, a, n, d, oracle.VERBATIM))
    elif case.family == "hls":
        h, w = (30, 40) if c == 2 else (29, 67)
        img = patchwork_hwc(oracle, h, w, c, seed=50 + c, band=5, col=9)
        d_in = torch.from_numpy(img).cuda()
        d_out = torch.full((h * n, w * n, c), CANARY, dtype=torch.uint8, device="cuda")
        lz.upscale_hls_device(d_in, d_out, a=a, bit_precision=case.bp)
        torch.cuda.synchronize()
        assert lz.stats()["kernel_id"] == case.kid, lz.stats()
        assert np.array_equal(d_out.cpu().numpy(), oracle.hls_upscale(img, n, a, case.bp))
    else:  # stream
        img = patchwork_hwc(oracle, 36, 64, 3, seed=60, band=5, col=9)
        _, st = run_small(torch, lz, img, 128, 72, case, 0)
        device_launches = st["kernel_launches"]
        words = img[..., 0].astype(np.uint32) | (img[..., 1].astype(np.uint32) << 8) | (img[..., 2].astype(np.uint32) << 16)
        got = lz.lanczos_stream(words, 64, 36, 128, 72, a=a, scale_n=n, scale_d=d)
        st = lz.stats()
        assert st["kernel_id"] == case.kid and st["kernel_launches"] == device_launches + 2, st
        want = oracle.upscale(img, 128, 72, a, n, d).astype(np.uint32)
        assert np.array_equal(got.reshape(72, 128), want[..., 0] | (want[..., 1] << 8) | (want[..., 2] << 16))
