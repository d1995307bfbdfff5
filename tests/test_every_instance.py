"""Every kernel instance the library compiles, launched at least once and checked against the reference.

Each template instance (a kernel family x channels x ratio x taps x exact/tolerance mode x 64/32-bit output stores) is
separate machine code with its own branches and register allocation, so a bug can live in one instance only.  CASES
maps every instance, as `nm -C` prints it, to a call that launches it:

  - the CPU test reads the symbols of the built library and requires that the set of kernels equals the keys of CASES,
    so a new instance without a case (or a case for an instance that no longer exists) fails without a GPU;
  - the GPU test runs each case and asserts the kernel id the library reports and, for the v6 family, which of its
    64-bit or 32-bit store variants the layout selects (restated from launch_v6, see st64()).

Content: for every specialised instance the near-tie H and V images of tests/util.py for its ratio and `a`,
and a patchwork of image-like, noise and dark patches several strips wide and several segments tall.  Exact mode
(MODE 0) must be bit-exact against the oracle.  Tolerance mode (MODE 1) is checked against a float64 restatement of the
reference for what include/lanczos_b200.h promises: the row pass exact, phase-0 rows copies of their centre row, and
interpolated samples plain fp32 sums that may differ from the reference only next to an integer.  Every output buffer
is surrounded by canary bytes (before the base, in the row padding, between frames, after the last row) that must
survive the call.
"""
import collections
import re
import subprocess

import numpy as np
import pytest

from harness import CANARY, canary_call, canary_layout, device_upscale, overwritten, torch_cuda  # noqa: F401
from util import (INSTANCES, NT, h_image, interleaved, patchwork, patchwork_hwc, planar, restate_planar, strict_floor,
                  v_image)

# ---- the cases -------------------------------------------------------------------------------------------------

Case = collections.namedtuple("Case", "family c a n d mode kid st64 bp")


def _cases():
    cases = {}
    for i in INSTANCES:
        for mode in (0, 1):
            if i.family == "v6":
                for st in (True, False):
                    sig = "lanczos_v6_kernel<%d, %d, %d, %d, %d, %d, %d, %s>" % (i.c, i.a, i.n, i.d, i.ph, i.km, mode,
                                                                                  str(st).lower())
                    cases[sig] = Case("v6", i.c, i.a, i.n, i.d, mode, i.kid, st, None)
            elif i.family == "dyn":
                cases["lanczos_dyn_kernel<%d, %d, %d, %d, %d>" % (i.c, i.a, i.n, i.d, mode)] = Case(
                    "dyn", i.c, i.a, i.n, i.d, mode, i.kid, None, None)
    # FLAG_GENERIC_KERNEL, one ratio per channel count
    for (c, a, n, d) in [(1, 3, 4, 1), (2, 3, 5, 3), (3, 2, 17, 10), (4, 3, 7, 4)]:
        cases["lanczos_generic_kernel<%d>" % c] = Case("generic", c, a, n, d, 0, 0, None, None)
    # the in-place top rows of a dyn-kernel call with default flags: a second launch
    cases["lanczos_alias_rows_kernel"] = Case("alias", 3, 3, 3, 2, 0, 6, None, None)
    for i in INSTANCES:
        if i.family == "hls_tile":
            sig = "lanczos_hls_tile_kernel<%d, %d, %d, %d>" % (i.c, i.a, i.n, i.mask)
            cases[sig] = Case("hls", i.c, i.a, i.n, i.d, 0, i.kid, None, 8)
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
    """The layouts used below select the store variant they are meant to (the GPU test checks it on every layout it
    launches)."""
    for rb in (480, 1920, 83040):
        assert st64(rb, rb, 4096, 1, 0)
        assert not st64(rb, rb + 4, 4096, 1, 0)                 # pitch
        assert not st64(rb, rb, 4096 + 4, 1, 0)                 # base
        assert not st64(rb, rb, 4096, 3, rb * 10 + 4)           # batch
        assert st64(rb, rb, 4096, 1, rb * 10 + 4)               # a frame stride is not read for one frame
    assert not st64(189 * 4, 189 * 4, 4096, 1, 0)              # id 3 natural: 126 -> 189 pixels of 4 bytes
    assert not st64(252, 252, 4096, 1, 0)                      # id 9 natural: 168 -> 252 one-byte pixels


def test_canary_check_reports_every_byte_outside_the_output():
    """The check behind every canary_call: one byte changed in the lead, a row's padding, a frame gap or the tail is
    reported at its offset from the base; bytes of the output rows are not looked at."""
    rb, rows, frames = 12, 3, 2
    base, pitch, fstride, total = canary_layout(rb, rows, frames, 4, 5, 6)
    host = np.full(total, CANARY, np.uint8)
    out = np.lib.stride_tricks.as_strided(host[base:], shape=(frames, rows, rb), strides=(fstride, pitch, 1))
    out[...] = np.arange(out.size).reshape(out.shape)
    assert len(overwritten(host, base, frames, rows, rb, pitch, fstride)) == 0
    places = {"lead": (-base, -1), "row pad": (rb, pitch - 1, fstride + pitch + rb),
              "frame gap": (pitch * rows, fstride - 1), "tail": (fstride * frames, total - base - 1)}
    for where, offsets in places.items():
        for off in offsets:
            hit = host.copy()
            hit[base + off] ^= 0xFF
            assert overwritten(hit, base, frames, rows, rb, pitch, fstride).tolist() == [off], (where, off)


# ---- content ---------------------------------------------------------------------------------------------------

NATURAL_W = {3: 126, 9: 168}  # widths whose output rows end in half a 64-bit word (the last lane stores one word)


def contents(oracle, case):
    """(name, frames, planted windows, output layout) for a specialised instance.  The v6 32-bit-store instances get a
    layout that forces them: a padded pitch, an output base 4 bytes past an 8-byte boundary, a batch with an odd frame
    stride, or (ids 3 and 9) the natural width whose rows end in half a word."""
    c, a, n, d, kid = case.c, case.a, case.n, case.d, case.kid
    h, hp = _cached(("h", c, a, n, d), lambda: h_image(oracle, n, d, a, c, seed=100 + kid))
    v, vp = _cached(("v", c, a, n, d), lambda: v_image(oracle, n, d, a, c, seed=100 + kid))
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
    return _cached(key, lambda: restate_planar(planar(img), ow, oh, a, n, d, clean=True, parts=True))


# ---- launching with canaries -----------------------------------------------------------------------------------

# output layouts of contents(): canary_layout's base offset, row padding and frame gap
LAYOUTS = {"dense": (0, 0, 0), "natural": (0, 0, 0), "pitch": (0, 4, 0), "base": (4, 0, 0), "batch": (0, 0, 4)}


def launch(torch, lz, case, frames, layout, flags, stats=False):
    """Run one specialised-kernel call on `frames` (list of [H][W][C]), input rows padded to 16 bytes (the TMA kernels
    need them); returns (outputs, stats).  Checks the kernel id and the store variant of v6 instances."""
    c, a, n, d = case.c, case.a, case.n, case.d
    ih, iw = frames[0].shape[:2]
    ow, oh = iw * n // d, ih * n // d
    nf = len(frames)
    off, pad, gap = LAYOUTS[layout]
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, flags=flags)
    outs, st, _ = canary_call(torch, lz, desc, frames, "upscale" if nf == 1 else "upscale_batch", in_pad=(-iw * c) % 16,
                              out_off=off, out_pad=pad, out_gap=gap, stats=stats)
    assert st["kernel_id"] == case.kid, (st, case)
    if case.family == "v6":
        base, pitch, fstride, _ = canary_layout(ow * c, oh, nf, off, pad, gap)   # base: past a 256-byte boundary
        assert st64(ow * c, pitch, base, nf, fstride) == case.st64, (layout, ow * c, pitch, base % 8, fstride)
    return outs, st


# ---- checks ----------------------------------------------------------------------------------------------------

def check_exact(torch, lz, oracle, case, name, frames, planted, layout):
    a, n, d = case.a, case.n, case.d
    got, st = launch(torch, lz, case, frames, layout, 0, stats=True)
    for f, img in enumerate(frames):
        want = oracle_ref(oracle, img, a, n, d, oracle.VERBATIM)
        bad = np.argwhere(got[f] != want)
        assert len(bad) == 0, (name, layout, "frame", f, len(bad), bad[:8].tolist())
    assert st["strict_samples"] >= strict_floor(planted), (name, st, strict_floor(planted))
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
    g = planar(got)
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
        ref, mid, sums = restate_planar(planar(img), ow, oh, a, n, d, clean=True, parts=True)
        assert np.array_equal(interleaved(ref), oracle.upscale(img, ow, oh, a, n, d, variant=oracle.CLEAN))
        assert np.array_equal(NT.quantise(sums), ref)
        full = restate_planar(planar(img), ow, oh, a, n, d, clean=False, parts=True)[0]
        assert np.array_equal(interleaved(full), oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM))
        yy = np.arange(oh)
        ph0 = (yy * d) % n == 0
        promised = ref.copy()
        promised[:, ph0] = mid[:, yy[ph0] * d // n]
        assert check_tolerance_clean(interleaved(promised), ref, mid, sums, n, d, "promised") == 1.0
        rounded = promised.copy()
        rounded[:, ~ph0] = np.clip(np.floor(sums[:, ~ph0] + 0.5), 0, 255).astype(np.uint8)
        with pytest.raises(pytest.fail.Exception):
            check_tolerance_clean(interleaved(rounded), ref, mid, sums, n, d, "rounded")
        if d == 1:
            shifted = promised.copy()
            shifted[:, ph0] = mid[:, np.maximum(yy[ph0] * d // n - 1, 0)]
            with pytest.raises(AssertionError):
                check_tolerance_clean(interleaved(shifted), ref, mid, sums, n, d, "wrong centre row")


# ---- GPU -------------------------------------------------------------------------------------------------------

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
            got = device_upscale(torch, lz, img, ow, oh, a, n, d, flags=lz.FLAG_GENERIC_KERNEL | flags)
            assert lz.stats()["kernel_id"] == 0, lz.stats()
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
        device_upscale(torch, lz, img, 128, 72, a, n, d)
        device_launches = lz.stats()["kernel_launches"]
        words = img[..., 0].astype(np.uint32) | (img[..., 1].astype(np.uint32) << 8) | (img[..., 2].astype(np.uint32) << 16)
        got = lz.lanczos_stream(words, 64, 36, 128, 72, a=a, scale_n=n, scale_d=d)
        st = lz.stats()
        assert st["kernel_id"] == case.kid and st["kernel_launches"] == device_launches + 2, st
        want = oracle.upscale(img, 128, 72, a, n, d).astype(np.uint32)
        assert np.array_equal(got.reshape(72, 128), want[..., 0] | (want[..., 1] << 8) | (want[..., 2] << 16))
