"""Windows of the output image: lanczos_b200_region_input_rect, lanczos_b200_upscale_region and
lanczos_b200_upscale_host_region.

A window is any rectangle of the output.  Its pixels must equal the pixels at the same coordinates of the whole-image
result, bit for bit, computed from the input rect the window reads and nothing else:

  - CPU: the rect of region_input_rect against a restatement of the tap rule (rows are band_input_rows, every tap of
    every window pixel lies in the rect or outside the image, the rect is no wider than the taps plus the documented
    16-byte rounding of its first column), and the order in which the entry points check their arguments;
  - GPU: windows of every kernel family against the oracle's whole image, cropped.  Every call reads its rect from a
    tight copy inside a larger allocation of unrelated random bytes (a kernel that reads outside the rect gets wrong
    pixels) and writes into a buffer of canary bytes that must survive around the window.
"""
import ctypes as C
import math

import numpy as np
import pytest

from harness import (ERR_BAND, ERR_CUDA, ERR_DIMS, ERR_NULL, ERR_TAPS, NO_DEVICE, canary_call, in_thread,  # noqa: F401
                     torch_cuda)
from util import EMPTY, INSTANCES, h_image, patchwork, patchwork_hwc, tap0, v_image


# ---- the rect a window reads ----------------------------------------------------------------------------------

def needed_cols(iw, n, d, a, x0, w):
    """First and last input column that the output columns [x0, x0 + w) read, clipped to the image."""
    lo = max(0, tap0(x0, n, d, a))
    hi = min(iw - 1, tap0(x0 + w - 1, n, d, a) + 2 * a - 1)
    return lo, hi


def rect_windows(ow, oh, alias):
    """Corners, edges, interior and windows containing the in-place top rows, as (x0, y0, w, h)."""
    w, h = max(1, ow // 5), max(1, oh // 5)
    out = [(0, 0, w, h), (ow - w, 0, w, h), (0, oh - h, w, h), (ow - w, oh - h, w, h),      # corners
           (ow // 3, 0, w, 1), (0, oh // 3, 1, h), (ow - 1, oh // 2, 1, 1), (ow // 2, oh - 1, w, 1),   # edges
           (ow // 3 + 1, oh // 3, w, h), (ow // 2 - 3, oh // 2 + 1, 7, 3), (0, 0, ow, oh)]    # interior, whole
    if alias > 0:
        out += [(ow // 4 + 1, max(0, alias - 2), w, 4), (5, alias, 3, 2)]
    return out


RECT_RATIOS = [(2, 1), (3, 2), (17, 10), (7, 4), (9, 4)]


@pytest.mark.parametrize("n,d", RECT_RATIOS)
def test_region_input_rect(lz, n, d):
    for a in range(1, 5):
        for c in range(1, 5):
            iw, ih = 30 * d + 7, 20 * d + 3
            ow, oh = iw * n // d, ih * n // d
            desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d)
            step = 16 // math.gcd(16, c)
            for (x0, y0, w, h) in rect_windows(ow, oh, lz.alias_rows(desc)):
                ix, iy, iwr, ihr = lz.region_input_rect(desc, x0, y0, w, h)
                assert (iy, ihr) == lz.band_input_rows(desc, y0, h)
                assert 0 <= ix and ix + iwr <= iw and (ix * c) % 16 == 0
                xx = np.arange(x0, x0 + w)
                taps = tap0(xx, n, d, a)[:, None] + np.arange(2 * a)[None, :]
                inside = (taps >= 0) & (taps < iw)
                assert np.all(~inside | ((taps >= ix) & (taps < ix + iwr))), (n, d, a, c, x0, w)
                lo, hi = needed_cols(iw, n, d, a, x0, w)
                assert ix + iwr - 1 == hi and ix <= lo < ix + step and ix == lo // step * step, (n, d, a, c, x0, w)
            for bad in [(-1, 0, 4, 4), (0, -1, 4, 4), (ow - 3, 0, 4, 4), (0, oh - 3, 4, 4), (0, 0, 0, 4), (0, 0, 4, 0)]:
                with pytest.raises(lz.LanczosError) as e:
                    lz.region_input_rect(desc, *bad)
                assert e.value.code == ERR_BAND, bad


def region_calls(lz, desc, null=False, rect=(0, 0, 16, 16), frames=1):
    L = lz.lib()
    img = np.zeros(1 << 16, np.uint8)
    host = C.c_void_p(img.ctypes.data)
    buf = None if null else host
    d = C.byref(desc)
    ix, iy, iw, ih = rect
    return {
        "upscale_region": lambda: L.lanczos_b200_upscale_region(d, host, buf, 4, 4, 8, 8, ix, iy, iw, ih, frames, 0, 0,
                                                                NO_DEVICE, None),
        "upscale_host_region": lambda: L.lanczos_b200_upscale_host_region(d, host, buf, 4, 4, 8, 8, 0, NO_DEVICE),
    }


def test_error_order_of_region_entry_points(lz):
    """Like lanczos_b200_upscale_band: null buffers, then the device, then the descriptor, then the window and rect."""
    valid = lz.make_desc(16, 16, 32, 32, 3, 3, 2, 1)
    bad_a = lz.make_desc(16, 16, 32, 32, 3, 9, 2, 1)
    for name in ("upscale_region", "upscale_host_region"):
        assert in_thread(region_calls(lz, valid)[name]) == ERR_CUDA
        assert in_thread(region_calls(lz, bad_a)[name]) == ERR_CUDA
        assert in_thread(region_calls(lz, bad_a, null=True)[name]) == ERR_NULL
    # a rect that does not cover the window: the device is checked first
    assert in_thread(region_calls(lz, valid, rect=(4, 4, 2, 2))["upscale_region"]) == ERR_CUDA
    assert in_thread(region_calls(lz, valid, frames=-1)["upscale_region"]) == ERR_DIMS
    # the rect query has no device: the descriptor, then the window
    r = [C.c_int32() for _ in range(4)]
    L = lz.lib()
    assert L.lanczos_b200_region_input_rect(C.byref(bad_a), 0, 0, 4, 4, *[C.byref(v) for v in r]) == ERR_TAPS
    assert L.lanczos_b200_region_input_rect(C.byref(valid), 0, 0, 4, 4, None, *[C.byref(v) for v in r[1:]]) == ERR_NULL
    assert L.lanczos_b200_region_input_rect(C.byref(valid), 30, 0, 4, 4, *[C.byref(v) for v in r]) == ERR_BAND


# ---- GPU --------------------------------------------------------------------------------------------------------

def word_rect(rect, iw, c):
    """The rect widened to the right, inside the image, until its rows are whole 32-bit words (the fast kernels
    read the rect through a map of words)."""
    ix, iy, w, h = rect
    while (w * c) % 4 and ix + w < iw:
        w += 1
    return ix, iy, w, h


def run_region(torch, lz, desc, frames, win, rect=None, flags=None, stats=False, in_gap=0, out_gap=0, whole=False):
    """Window win = (x0, y0, w, h) of `frames` (list of [H][W][C] host images) through lanczos_b200_upscale_region
    (whole: the whole image through lanczos_b200_upscale, same buffers) with canary_call.  The rect (default:
    region_input_rect widened to whole words) has rows padded past the next 16 bytes; the window's rows are padded past
    the next 8.  `flags` replaces desc.flags.  Returns (windows, stats, launch)."""
    x0, y0, w, _ = win
    ih, iw, c = frames[0].shape
    rect = rect or word_rect(lz.region_input_rect(desc, *win), iw, c)
    if flags is not None:
        desc = lz.Desc.from_buffer_copy(desc)
        desc.flags = flags
    return canary_call(torch, lz, desc, frames, "upscale" if whole else "upscale_region", win=win, rect=rect, in_off=256,
                       in_pad=(-rect[2] * c) % 16 + 16, in_gap=in_gap, out_pad=(-w * c) % 8 + 8, out_gap=out_gap,
                       seed=x0 * 7919 + y0 * 31 + w + len(frames), stats=stats)


def full_frame(torch, lz, desc, img, flags):
    """The whole image through lanczos_b200_upscale with the padded pitches run_region uses: (output, stats, launch)."""
    ih, iw, c = img.shape
    return run_region(torch, lz, desc, [img], (0, 0, desc.out_w, desc.out_h), rect=(0, 0, iw, ih), flags=flags,
                      whole=True)


def crop(ref, win):
    x0, y0, w, h = win
    return ref[y0:y0 + h, x0:x0 + w]


GENERIC = 1 << 2   # LANCZOS_FLAG_GENERIC_KERNEL

# (name, channels, a, N, D, flags, kernel id of aligned windows, kernel id of unaligned windows)
DYN_IDS = {(i.c, i.a, i.n, i.d): i.kid for i in INSTANCES if i.family == "dyn"}
FAMILIES = ([("v6_%d" % i.kid, i.c, i.a, i.n, i.d, 0, i.kid, DYN_IDS.get((i.c, i.a, i.n, i.d), 0))
             for i in INSTANCES if i.family == "v6"]
            + [("dyn_%d" % i.kid, i.c, i.a, i.n, i.d, 0, i.kid, i.kid) for i in INSTANCES if i.family == "dyn"]
            + [("generic_c%d" % c, c, a, n, d, GENERIC, 0, 0) for (c, a, n, d) in [(1, 3, 4, 1), (2, 3, 5, 3), (3, 2, 17, 10),
                                                                                 (4, 3, 7, 4)]]
            + [("alias_rows", 3, 3, 3, 2, 0, 6, 6)])
FAMILY = {f[0]: f[1:] for f in FAMILIES}


def family_windows(ow, oh, c, n, d, alias):
    """(label, window, aligned): aligned windows start on the 16-byte grid of the output row, unaligned ones at an odd
    pixel off that grid whose phase is not 0."""
    step = 16 // math.gcd(16, c)
    xa = step * max(1, ow // (4 * step))                       # aligned, not 0
    xu = xa + 1
    while (xu * d) % n == 0 or (xu * c) % 16 == 0:
        xu += 2
    w = max(4, (ow // 3) // 4 * 4)
    h = max(3, oh // 4)
    y = oh // 3
    top = max(alias + 2, 3)
    return [("aligned", (xa, y, w, h), True), ("unaligned", (xu, y + 1, w, h), False),
            ("left edge", (0, y, w, h), True), ("right edge", (ow - w, y, w, h), None),
            ("top-left", (0, 0, w, h), True), ("top-right", (ow - w, 0, w, h), None),
            ("bottom-left", (0, oh - h, w, h), True), ("bottom-right", (ow - w, oh - h, w, h), None),
            ("bottom edge", (xu, oh - h, w, h), False),
            ("top rows aligned", (xa, 0, w, top), True), ("top rows unaligned", (xu, 1, w, top), False),
            ("1 pixel wide", (xu, y, 1, h), None), ("1 row tall", (xa, y, w, 1), None)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FAMILY))
def test_windows_of_every_family(torch_cuda, lz, oracle, name):
    torch = torch_cuda
    c, a, n, d, flags, kid_aligned, kid_unaligned = FAMILY[name]
    img = patchwork(oracle, c, n, d, seed=400 + c * 7 + n)
    ih, iw, _ = img.shape
    ow, oh = oracle.out_dims(iw, ih, n, d)
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, flags=flags)
    alias = lz.alias_rows(desc)
    for extra, variant in ((0, oracle.VERBATIM), (lz.FLAG_NO_ALIAS, oracle.CLEAN)):
        ref = oracle.upscale(img, ow, oh, a, n, d, variant=variant)
        for (label, win, aligned) in family_windows(ow, oh, c, n, d, alias):
            (got,), st, _ = run_region(torch, lz, desc, [img], win, flags=flags | extra)
            bad = np.argwhere(got != crop(ref, win))
            assert len(bad) == 0, (name, label, win, extra, len(bad), bad[:8].tolist())
            x0, y0, w, h = win
            if aligned is not None and (w * c) % 4 == 0:
                want = kid_aligned if aligned else kid_unaligned
                assert st["kernel_id"] == want, (name, label, win, st)
            if name == "alias_rows" and extra == 0 and y0 < alias:
                assert st["kernel_launches"] == 2 and st["alias_rows"] == min(alias, y0 + h) - y0, (label, st)
        # the whole image: the same output, kernel and launch report as the full-frame call
        want, want_st, want_ln = full_frame(torch, lz, desc, img, flags | extra)
        got, st, ln = run_region(torch, lz, desc, [img], (0, 0, ow, oh), flags=flags | extra)
        assert np.array_equal(got[0], want[0]) and np.array_equal(want[0], ref)
        assert (st, ln) == (want_st, want_ln)


@pytest.mark.gpu
@pytest.mark.parametrize("kid", [f[6] for f in FAMILIES if f[0].startswith(("v6", "dyn"))])
def test_strict_paths_at_column_offsets(torch_cuda, lz, oracle, kid):
    """The near-tie images of tests/util.py: the exact re-evaluation runs at a column offset, and is right."""
    torch = torch_cuda
    name = [f[0] for f in FAMILIES if f[6] == kid and f[0].startswith(("v6", "dyn"))][0]
    c, a, n, d, flags, _, _ = FAMILY[name]
    step = 16 // math.gcd(16, c)
    for img, _ in (h_image(oracle, n, d, a, c, seed=500 + kid), v_image(oracle, n, d, a, c, seed=500 + kid)):
        ih, iw, _ = img.shape
        ow, oh = oracle.out_dims(iw, ih, n, d)
        desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d)
        ref = oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM)
        x0 = step if name.startswith("v6") else 3          # v6 needs the 16-byte grid, dyn takes any column
        w = (ow - x0 - 1) // 4 * 4
        win = (x0, 1, w, oh - 2)
        (got,), st, _ = run_region(torch, lz, desc, [img], win, stats=True)
        bad = np.argwhere(got != crop(ref, win))
        assert len(bad) == 0, (name, win, len(bad), bad[:8].tolist())
        assert st["kernel_id"] == kid, (name, st)
        assert st["strict_samples"] > 0 or (n, d, a) in EMPTY, (name, st)   # EMPTY: the ratio has no near ties


# 2/1 RGB (v6 id 1), 3/2 RGBA (v6 id 3), 17/10 RGB (dyn id 5) and 17/10 RGB with a = 2 (generic only)
TILE_CASES = [(3, 3, 2, 1, 1), (4, 3, 3, 2, 3), (3, 3, 17, 10, 5), (3, 2, 17, 10, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("c,a,n,d,kid", TILE_CASES)
def test_tiles_assemble_to_the_whole_image(torch_cuda, lz, oracle, c, a, n, d, kid):
    torch = torch_cuda
    img = patchwork(oracle, c, n, d, seed=600 + n)
    ih, iw, _ = img.shape
    ow, oh = oracle.out_dims(iw, ih, n, d)
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d)
    want, want_st, _ = full_frame(torch, lz, desc, img, 0)
    assert want_st["kernel_id"] == kid
    step = 16 // math.gcd(16, c)
    cols = [0, step * (ow // (3 * step)), (2 * ow) // 3 | 1, ow]         # an aligned and an odd cut
    rows = [0, 2, oh // 3, (2 * oh) // 3 + 1, oh]                        # one cut inside the top rows
    got = np.zeros_like(want[0])
    for y0, y1 in zip(rows, rows[1:]):
        for x0, x1 in zip(cols, cols[1:]):
            win = (x0, y0, x1 - x0, y1 - y0)
            ix, iy, riw, rih = word_rect(lz.region_input_rect(desc, *win), iw, c)
            # the tile's own rect, as a tight copy with a 16-byte pitch
            rect = np.zeros((rih, -(-riw * c // 16) * 16), np.uint8)
            rect[:, :riw * c] = img[iy:iy + rih, ix:ix + riw].reshape(rih, riw * c)
            d_in = torch.as_strided(torch.from_numpy(rect).cuda(), (rih, riw, c), (rect.shape[1], c, 1))
            d_out = torch.empty((y1 - y0, x1 - x0, c), dtype=torch.uint8, device="cuda")
            lz.upscale_region_device(desc, d_in, d_out, x0, y0, ix, iy)
            torch.cuda.synchronize()
            got[y0:y1, x0:x1] = d_out.cpu().numpy()
    bad = np.argwhere(got != want[0])
    assert len(bad) == 0, (len(bad), bad[:8].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["v6_1", "dyn_5", "generic_c3"])
def test_batch_window_with_frame_strides(torch_cuda, lz, oracle, name):
    torch = torch_cuda
    c, a, n, d, flags, _, _ = FAMILY[name]
    frames = [patchwork(oracle, c, n, d, seed=700 + f) for f in range(3)]
    ih, iw, _ = frames[0].shape
    ow, oh = oracle.out_dims(iw, ih, n, d)
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, flags=flags)
    refs = [oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM) for img in frames]
    for win in [(16, 5, 160, 40), (33, 0, 100, 30)]:
        got, st, ln = run_region(torch, lz, desc, frames, win, in_gap=48, out_gap=12)
        assert ln["grid_z"] == 3, ln
        for f, ref in enumerate(refs):
            assert np.array_equal(got[f], crop(ref, win)), (name, win, f)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["v6_1", "v6_3", "dyn_5", "dyn_6"])
def test_tolerance_mode_window(torch_cuda, lz, oracle, name):
    """A window of the tolerance-mode result equals the same pixels of the whole image in that mode."""
    torch = torch_cuda
    c, a, n, d, _, kid, _ = FAMILY[name]
    img = patchwork(oracle, c, n, d, seed=800)
    ih, iw, _ = img.shape
    ow, oh = oracle.out_dims(iw, ih, n, d)
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d)
    flags = lz.FLAG_TOLERANCE_1LSB
    want, st, _ = full_frame(torch, lz, desc, img, flags)
    assert st["kernel_id"] == kid
    x0 = 48 // math.gcd(48, c) * 2 if name.startswith("v6") else 7   # v6 tolerance mode: the 48-byte grid
    for win in [(x0, 0, 64, oh), (x0, oh // 3, (ow - x0) // 4 * 4, oh // 3)]:
        (got,), st, _ = run_region(torch, lz, desc, [img], win, flags=flags)
        assert st["kernel_id"] == kid, (win, st)
        assert np.array_equal(got, crop(want[0], win)), win


@pytest.mark.gpu
def test_independent_flag_on_consecutive_windows(torch_cuda, lz, oracle):
    torch = torch_cuda
    c, a, n, d = 3, 3, 2, 1
    img = patchwork(oracle, c, n, d, seed=900)
    ih, iw, _ = img.shape
    ow, oh = oracle.out_dims(iw, ih, n, d)
    full = torch.from_numpy(np.ascontiguousarray(np.pad(img, ((0, 0), (0, (-iw) % 16), (0, 0))))).cuda()[:, :iw]
    wins = [(16, 0, 128, 60), (64, 50, 96, 70), (0, oh - 40, ow, 40)]
    outs = {}
    for flags in (0, lz.FLAG_INDEPENDENT):
        desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, flags=flags)
        res = []
        for (x0, y0, w, h) in wins:
            ix, iy, riw, rih = word_rect(lz.region_input_rect(desc, x0, y0, w, h), iw, c)
            d_out = torch.empty((h, w, c), dtype=torch.uint8, device="cuda")
            lz.upscale_region_device(desc, full[iy:iy + rih, ix:ix + riw], d_out, x0, y0, ix, iy)
            res.append(d_out)
        torch.cuda.synchronize()
        outs[flags] = [r.cpu().numpy() for r in res]
    ref = oracle.upscale(img, ow, oh, a, n, d)
    for win, g0, g1 in zip(wins, outs[0], outs[lz.FLAG_INDEPENDENT]):
        assert np.array_equal(g0, g1) and np.array_equal(g0, crop(ref, win)), win


@pytest.mark.gpu
@pytest.mark.parametrize("c,n,d", [(3, 2, 1), (3, 17, 10), (4, 3, 2)])
def test_torch_view_equals_tight_copy(torch_cuda, lz, oracle, c, n, d):
    torch = torch_cuda
    img = patchwork(oracle, c, n, d, seed=1000)
    ih, iw, _ = img.shape
    ow, oh = oracle.out_dims(iw, ih, n, d)
    desc = lz.make_desc(iw, ih, ow, oh, c, 3, n, d)
    full = torch.from_numpy(img).cuda()
    for (x0, y0, w, h) in [(16, 3, 100, 50), (37, 0, 64, 33)]:
        ix, iy, riw, rih = lz.region_input_rect(desc, x0, y0, w, h)
        view = full[iy:iy + rih, ix:ix + riw]
        a_out = torch.empty((h, w, c), dtype=torch.uint8, device="cuda")
        b_out = torch.empty((h, w, c), dtype=torch.uint8, device="cuda")
        lz.upscale_region_device(desc, view, a_out, x0, y0, ix, iy)
        lz.upscale_region_device(desc, view.contiguous(), b_out, x0, y0, ix, iy)
        torch.cuda.synchronize()
        want = crop(oracle.upscale(img, ow, oh, 3, n, d), (x0, y0, w, h))
        assert np.array_equal(a_out.cpu().numpy(), want) and np.array_equal(b_out.cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("iw,ih,c,n,d", [(61, 37, 3, 2, 1), (64, 40, 4, 3, 2), (57, 30, 1, 3, 1), (45, 25, 2, 2, 1)])
def test_host_region(lz, oracle, iw, ih, c, n, d):
    img = patchwork_hwc(oracle, ih, iw, c, seed=c, band=7, col=11)
    ow, oh = oracle.out_dims(iw, ih, n, d)
    ref = oracle.upscale(img, ow, oh, 3, n, d)
    for win in [(0, 0, ow, oh), (3, 1, 11, 7), (ow - 9, oh - 5, 9, 5), (ow // 2, 0, 1, oh)]:
        got = lz.upscale_region(img, ow, oh, *win, a=3, scale_n=n, scale_d=d)
        assert np.array_equal(got, crop(ref, win)), win
