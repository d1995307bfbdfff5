"""Every ratio the library accepts: the generic kernel, the alias-rows kernel and the host drivers.

The 24 specialised instances serve seven ratios and a few (channels, a) pairs each.  Every other call runs
lanczos_generic_kernel<C> (lanczos_generic.cu), and the in-place top rows of the reference's column pass run in
lanczos_alias_rows_kernel.  These tests run both at every reduced ratio N/D <= 16 the library accepts, with a = 1..4
and every channel count, on windows whose reference sums sit next to an integer under the generic kernel's own fp32
chain (tests/golden/near_ties_any_ratio.npz), on flat and dark patches, at ratios close to 1 where many top rows alias,
at output sizes unrelated to the ratio and on buffer layouts the specialised kernels decline.  The oracle stays the
truth: every byte must equal it.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

import test_near_ties as NTT
from util import dark_hwc, noise_hwc

NT = NTT.NT
HERE = os.path.dirname(os.path.abspath(__file__))
TIE, WRONG, NEAR = NT.TIE, NT.WRONG, NT.NEAR


def any_windows():
    z = np.load(os.path.join(HERE, "golden", "near_ties_any_ratio.npz"))
    return {k: z[k] for k in z.files}


ANY = any_windows()
INSTANCE_OF = {v: k for k, v in NTT.INSTANCES.items()}          # (C, a, N, D) -> kernel id


def reduced_ratios(limit):
    return [(n, d) for n in range(1, limit + 1) for d in range(1, n + 1) if math.gcd(n, d) == 1]


# ---- the reference's tables, restated ----------------------------------------------------------------------

def alias_restated(in_h, out_h, n, d, a):
    """(alias_rows, alias_in_rows) of the reference's in-place column pass (full_TB.h:67-77): going bottom-up, output
    row yy reads input rows first..first+2a-1 clipped to the image, and every one of them below yy already holds its
    final value.  Rows [0, alias_rows) read such a row; the emulation starts at the last row they read and needs the
    row pass of every input row the rows above that read."""
    def last(yy):
        return min(in_h - 1, yy * d // n + a)
    k = 1 + max([yy for yy in range(out_h) if last(yy) > yy], default=-1)
    top = max([last(yy) for yy in range(k)], default=-1)
    return k, 1 + max([last(yy) for yy in range(top + 1)], default=-1)


def band_restated(r0, rows, in_h, n, d, a, k, alias_in):
    """Input rows of an output band: its taps clipped to the image, from row 0 when it starts in the alias rows; a band
    entirely below the last input row reads one clamped row."""
    lo = min(in_h - 1, max(0, r0 * d // n - a + 1))
    hi = min(in_h - 1, (r0 + rows - 1) * d // n + a)
    if r0 < k:
        lo, hi = 0, max(hi, alias_in - 1)
    return lo, max(hi, lo) - lo + 1


# ---- CPU tests ---------------------------------------------------------------------------------------------

def accepted(lz, desc):
    try:
        lz.alias_rows(desc)
        return True
    except lz.LanczosError as e:
        assert e.code == -6, e
        return False


def test_float_floor_rejection_is_exactly_the_references(lz):
    """LANCZOS_ERR_RATIO_FLOAT happens exactly where the reference's floor((double)xx / ((double)N/D)) differs from
    xx*D/N for an output coordinate of either axis: at x0, the first such coordinate, an output length of x0 is
    accepted (coordinates stop at x0 - 1) and x0 + 1 is rejected."""
    misses = 0
    for (n, d) in reduced_ratios(64):
        x0 = NT.first_float_floor_miss(n, d)
        lengths = [4096] if x0 is None else [x0, x0 + 1]
        for length in lengths:
            want = x0 is None or length <= x0
            for (ow, oh) in ((length, 1), (1, length)):
                assert accepted(lz, lz.make_desc(1, 1, ow, oh, 1, 3, n, d)) == want, (n, d, ow, oh)
        misses += x0 is not None
    assert misses > 100
    assert [NT.first_float_floor_miss(n, d) for (n, d) in [(7, 3), (9, 7), (11, 10)]] == [35, 9, 33]
    # a ratio that is not reduced, and one taken from the widths (scale_n = 0), behave like the reduced ratio 7/3
    for (iw, ow, want) in [(15, 35, True), (18, 42, False)]:
        for (n, d) in [(7, 3), (14, 6), (0, 0)]:
            assert accepted(lz, lz.make_desc(iw, iw, ow, ow, 3, 3, n, d)) == want, (iw, ow, n, d)


def test_generic_windows_cover_the_sweep_and_sit_on_tile_edges():
    assert os.path.getsize(os.path.join(HERE, "golden", "near_ties_any_ratio.npz")) < 1 << 20
    cfgs = set(zip(ANY["n"].tolist(), ANY["d"].tolist(), ANY["a"].tolist()))
    assert cfgs <= set(NT.GENERIC_CONFIGS) and len(cfgs) > len(NT.GENERIC_CONFIGS) * 3 // 4
    for (n, d, a, xx) in zip(ANY["n"], ANY["d"], ANY["a"], ANY["coord"]):
        assert xx in NT.generic_coordinates(n, d) and xx % 64 in (0, 63) and xx % 32 in (0, 31), (n, d, a, xx)
    wrong = ANY["cls"] == WRONG
    assert wrong.sum() > 500 and (ANY["flags"][wrong] & NT.F_OFF_INTEGER).astype(bool).sum() > 100
    assert (ANY["cls"] == NEAR).sum() > 500


def test_generic_windows_keep_their_class(oracle):
    """Every stored window, re-evaluated from oracle_kernel and an exact emulation of the generic kernel's fp32
    chain, still has its recorded class, flags, nearest integer and distance."""
    for i in range(len(ANY["n"])):
        n, d, a, xx = (int(ANY[k][i]) for k in ("n", "d", "a", "coord"))
        cls, flags, k, dist = NT.classify_generic(ANY["win"][i], xx, n, d, a)
        assert (cls, flags, k, dist) == (ANY["cls"][i], ANY["flags"][i], ANY["k"][i], ANY["dist"][i]), (n, d, a, xx, i)
        if cls == WRONG:
            assert NT.WRONG_LO <= dist <= NT.WRONG_HI and flags & NT.F_WRONG_GENERIC
        else:
            assert cls == NEAR and dist <= NT.NEAR_TOL


NEAR_ONE = [(9, 8, 28), (17, 16, 52), (33, 32, 100), (65, 64, 196)]      # N, D, alias rows at a = 4


def test_alias_rows_and_band_rows_at_every_ratio(lz):
    """alias_rows and band_input_rows equal their restatement at the sweep ratios, near 1 and at 1/1 (whose alias
    input rows are the whole image), for bands from row 0, inside the alias rows, from alias_rows, and entirely below
    the last input row."""
    for (n, d, k) in NEAR_ONE:
        assert lz.alias_rows(lz.make_desc(8 * d, 8 * d, 8 * n, 8 * n, 1, 4, n, d)) == k
    cases = [(n, d, a, 3 * d + 5) for (n, d, a) in NT.GENERIC_CONFIGS]
    cases += [(n, d, 4, 4 * d) for (n, d, _) in NEAR_ONE] + [(1, 1, a, h) for a in (1, 4) for h in (32, 33)]
    for (n, d, a, in_h) in cases:
        out_h = in_h * n // d + 3 * n // d + 2 * a + 1                  # the last rows have no input row at all
        for flags in (0, 1):
            desc = lz.make_desc(16, in_h, 16, out_h, 1, a, n, d, flags=flags)
            k, alias_in = alias_restated(in_h, out_h, n, d, a) if flags == 0 else (0, 0)
            assert lz.alias_rows(desc) == k, (n, d, a, in_h, flags)
            if n == 1 and flags == 0:
                assert (k, alias_in) == (in_h - 1, in_h)
            below = next(yy for yy in range(out_h) if yy * d // n - a + 1 > in_h - 1)
            bands = [(0, max(1, k)), (0, out_h), (k, out_h - k), (below, out_h - below), (out_h - 1, 1)]
            if k > 2:
                bands.append((1, k - 2))
            for (r0, rows) in bands:
                got = lz.band_input_rows(desc, r0, rows)
                assert got == band_restated(r0, rows, in_h, n, d, a, k, alias_in), (n, d, a, in_h, flags, r0, rows)
            assert lz.band_input_rows(desc, below, 1) == (in_h - 1, 1)


# ---- GPU tests ---------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def patch_image(oracle, h, w, c, seed):
    """Top half dark noise (0..15), bottom half flat 8x8 blocks of extreme and middle values."""
    img = dark_hwc(oracle, h, w, c, seed=seed)
    vals = np.array([0, 255, 1, 254, 128, 127, 16, 200], np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    flat = vals[((yy // 8) * 3 + (xx // 8) + np.arange(c)[:, None, None]) % len(vals)]
    img[h // 2:] = np.transpose(flat, (1, 2, 0))[h // 2:]
    return img


def sweep_cases():
    """Every (N, D, a) of the generic windows with C rotating over 1..4 so that every (a, C) pair occurs; then the
    ratios close to 1 at a = 4, 1/1 on either side of the alias-rows kernel's 32-row cache, and 32/1 and 64/1."""
    cases = []
    ratios = sorted({(n, d) for (n, d, _) in NT.GENERIC_CONFIGS} | {(1, 1)})
    for r, (n, d) in enumerate(ratios):
        for a in range(1, 5):
            cases.append((n, d, a, 1 + (r + a) % 4, None))
    cases += [(n, d, 4, 1 + n % 4, None) for (n, d, _) in NEAR_ONE[1:]]
    cases += [(1, 1, 4, c, (40, h)) for c, h in ((3, 32), (1, 33), (4, 32))]
    cases += [(32, 1, 3, 3, (12, 9)), (64, 1, 2, 1, (8, 6))]
    return cases


SWEEP = sweep_cases()


def run_device(torch, lz, img, ow, oh, a, n, d, flags, stats):
    d_in = torch.from_numpy(img).cuda()
    d_out = torch.empty((oh, ow, img.shape[2]), dtype=torch.uint8, device="cuda")
    lz.enable_stats(stats)
    try:
        lz.upscale_device(d_in, d_out, a=a, scale_n=n, scale_d=d, flags=flags)
        torch.cuda.synchronize()
        st = lz.stats()
    finally:
        lz.enable_stats(False)
    return d_out.cpu().numpy(), st


def check_all_paths(torch, lz, oracle, img, planted, a, n, d, what):
    """Default dispatch and FLAG_GENERIC_KERNEL, each with the in-place top rows and with FLAG_NO_ALIAS: bit for bit,
    the expected kernel, and on the generic kernel every planted near and wrong-side window re-evaluated."""
    h, w, c = img.shape
    ow, oh = w * n // d, h * n // d
    kid = INSTANCE_OF.get((c, a, n, d), 0)                   # every image here has a layout the instances take
    for variant, alias_flag in ((oracle.VERBATIM, 0), (oracle.CLEAN, lz.FLAG_NO_ALIAS)):
        want = oracle.upscale(img, ow, oh, a, n, d, variant=variant)
        for generic in (False, True):
            got, st = run_device(torch, lz, img, ow, oh, a, n, d, alias_flag | (lz.FLAG_GENERIC_KERNEL if generic else 0),
                                 stats=True)
            assert st["kernel_id"] == (0 if generic else kid), (what, generic, st)
            bad = np.argwhere(got != want)
            assert len(bad) == 0, (what, "generic" if generic else "default", variant, len(bad), bad[:8].tolist())
            if st["kernel_id"] == 0:
                assert st["strict_samples"] >= NTT.strict_floor(planted, ANY), (what, st, NTT.strict_floor(planted, ANY))


@pytest.mark.gpu
@pytest.mark.parametrize("case", SWEEP, ids=lambda s: "%d_%d_a%d_c%d" % s[:4] + ("_%dx%d" % s[4] if s[4] else ""))
def test_every_ratio_bit_exact(torch_cuda, lz, oracle, case):
    n, d, a, c, size = case
    seed = 97 * n + 13 * d + a
    if size is None:
        img, hp = NTT.h_image(oracle, n, d, a, c, seed=seed, win=ANY)
        check_all_paths(torch_cuda, lz, oracle, img, hp, a, n, d, "H windows")
        in_h = max([NTT.tap0(int(x), n, d, a) + 2 * a for x in ANY["coord"][NTT.config_rows(n, d, a, ANY)]] + [64]) + 4
        ow = NTT.up_len(16 * d, n, d)
        top = lz.alias_rows(lz.make_desc(16 * d, in_h, ow, NTT.up_len(in_h, n, d), c, a, n, d))
        img, vp = NTT.v_image(oracle, n, d, a, c, seed=seed, nblk=8, win=ANY,
                              place=lambda i: int(ANY["coord"][i]) if ANY["coord"][i] >= max(top, 1) else None)
        check_all_paths(torch_cuda, lz, oracle, img, vp, a, n, d, "V windows")
        iw, ih = 16 * d * max(1, -(-256 * d // n) // (16 * d)), max(2 * a, 256 * d // n)
    else:
        iw, ih = size
        check_all_paths(torch_cuda, lz, oracle, noise_hwc(oracle, ih, iw, c, seed), [], a, n, d, "noise")
    check_all_paths(torch_cuda, lz, oracle, patch_image(oracle, ih, iw, c, seed), [], a, n, d, "dark and flat")


@pytest.mark.gpu
@pytest.mark.parametrize("case", [(n, d, 4, 1 + i) for i, (n, d, _) in enumerate(NEAR_ONE)] + [(1, 1, 4, 3), (1, 1, 3, 2)],
                         ids=lambda s: "%d_%d_a%d_c%d" % s)
def test_bands_through_the_alias_rows(torch_cuda, lz, oracle, case):
    """Bands that start or end inside the alias rows, at them and below them concatenate to the whole frame."""
    torch = torch_cuda
    n, d, a, c = case
    iw, ih = (16 * d, 4 * d) if n > 1 else (24, 40)
    ow, oh = iw * n // d, ih * n // d
    img = noise_hwc(oracle, ih, iw, c, seed=n)
    want = oracle.upscale(img, ow, oh, a, n, d)
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d)
    k = lz.alias_rows(desc)
    assert k > 8
    for cuts in ([0, k // 3, k - 1, k, k + 5, oh], [0, 1, k // 2, k + 1, oh], [0, oh]):
        cuts = sorted({min(r, oh) for r in cuts})
        out = np.zeros_like(want)
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            in0, inn = lz.band_input_rows(desc, r0, r1 - r0)
            d_in = torch.from_numpy(np.ascontiguousarray(img[in0:in0 + inn])).cuda()
            d_out = torch.zeros((r1 - r0, ow, c), dtype=torch.uint8, device="cuda")
            lz.upscale_band_device(desc, d_in, d_out, r0, r1 - r0, in0, inn)
            torch.cuda.synchronize()
            out[r0:r1] = d_out.cpu().numpy()
        bad = np.argwhere(out != want)
        assert len(bad) == 0, (cuts, len(bad), bad[:8].tolist())


# ---- raw launches with canaries ----------------------------------------------------------------------------

CANARY = 0x5C


def launch_raw(torch, lz, frames, ow, oh, a, n, d, in_off=0, in_pad=0, in_gap=0, out_off=0, out_pad=0, flags=0):
    """One call on device buffers laid out as asked: the input base `in_off` bytes past a 256-byte boundary, rows
    padded by `in_pad` bytes, frames `in_gap` bytes apart; the output likewise, surrounded by canary bytes.  Returns
    (outputs, kernel id) after checking every canary."""
    nf = len(frames)
    ih, iw, c = frames[0].shape
    in_pitch, out_pitch = iw * c + in_pad, ow * c + out_pad
    in_fs = in_pitch * ih + in_gap
    src = np.zeros(in_off + in_fs * nf + 64, np.uint8)
    for f, img in enumerate(frames):
        v = np.lib.stride_tricks.as_strided(src[in_off + f * in_fs:], shape=(ih, iw * c), strides=(in_pitch, 1))
        v[...] = img.reshape(ih, iw * c)
    out_fs = out_pitch * oh + 4
    lead = 64 + out_off
    total = lead + out_fs * nf + 2 * out_pitch + 64
    d_in = torch.from_numpy(src).cuda()
    buf = torch.full((total,), CANARY, dtype=torch.uint8, device="cuda")
    assert d_in.data_ptr() % 256 == 0 and buf.data_ptr() % 256 == 0
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, in_pitch, out_pitch, flags)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    L = lz.lib()
    rc = L.lanczos_b200_upscale_batch(C.byref(desc), C.c_void_p(d_in.data_ptr() + in_off),
                                      C.c_void_p(buf.data_ptr() + lead), nf, in_fs, out_fs, 0, stream)
    torch.cuda.synchronize()
    assert rc == 0, (rc, L.lanczos_b200_strerror(rc))
    kid = lz.stats()["kernel_id"]
    host = buf.cpu().numpy()
    rb = ow * c
    view = np.lib.stride_tricks.as_strided(host[lead:], shape=(nf, oh, rb), strides=(out_fs, out_pitch, 1))
    outs = [np.array(view[f]).reshape(oh, ow, c) for f in range(nf)]
    canary = np.ones(total, bool)
    np.lib.stride_tricks.as_strided(canary[lead:], shape=(nf, oh, rb), strides=(out_fs, out_pitch, 1))[...] = False
    hit = np.nonzero(canary & (host != CANARY))[0]
    assert len(hit) == 0, ("canary bytes overwritten", len(hit), [int(i) - lead for i in hit[:8]])
    return outs, kid


# (channels, a, N, D, input width, input height) of the generic kernel, one v6 and one dyn instance
FAMILIES = {"generic": (3, 3, 5, 4, 64, 40), "v6": (3, 3, 2, 1, 64, 40), "dyn": (3, 2, 3, 1, 48, 36)}


@pytest.mark.gpu
@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_output_size_independent_of_ratio_any_kernel(torch_cuda, lz, oracle, family):
    """Output widths below and far above in_w*N/D (columns with no tap inside the image), narrower than the input,
    and heights past in_h*N/D with a band entirely below the input: every kernel takes the sizes as loop bounds."""
    c, a, n, d, iw, ih = FAMILIES[family]
    kid = INSTANCE_OF.get((c, a, n, d), 0)
    img = noise_hwc(oracle, ih, iw, c, seed=5)
    full_w, full_h = iw * n // d, ih * n // d
    empty_w = (iw + a + 2) * n // d + 8                           # past this column no tap lies inside the image
    for (ow, oh) in [(full_w - 12, full_h), (empty_w // 4 * 4 + 16, full_h), (iw - 8, ih + 4), (full_w, full_h + 24 * n)]:
        outs, got_kid = launch_raw(torch_cuda, lz, [img], ow, oh, a, n, d)
        assert got_kid == kid, (family, ow, oh, got_kid)
        want = oracle.upscale(img, ow, oh, a, n, d)
        assert np.array_equal(outs[0], want), (family, ow, oh)
    # a band that lies entirely below the last input row
    ow, oh = full_w, full_h + 24 * n
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d)
    r0 = oh - 16
    assert r0 * d // n - a + 1 > ih - 1
    in0, inn = lz.band_input_rows(desc, r0, 16)
    assert (in0, inn) == (ih - 1, 1)
    torch = torch_cuda
    d_out = torch.zeros((16, ow, c), dtype=torch.uint8, device="cuda")
    lz.upscale_band_device(desc, torch.from_numpy(np.ascontiguousarray(img[in0:in0 + inn])).cuda(), d_out, r0, 16, in0, inn)
    torch.cuda.synchronize()
    assert np.array_equal(d_out.cpu().numpy(), oracle.upscale(img, ow, oh, a, n, d)[r0:])


# every clause of strip_layout_ok (fast_common.cuh) broken on its own, each a layout the API accepts
BROKEN = {
    "in_base+4": dict(in_off=4), "in_base+8": dict(in_off=8), "in_pitch%16=4": dict(in_pad=4),
    "in_frame_stride%16=4": dict(in_gap=4, frames=2), "out_base+1": dict(out_off=1), "out_base+2": dict(out_off=2),
    "odd_out_pitch": dict(out_pad=1),
}


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["v6", "dyn"])
@pytest.mark.parametrize("layout", sorted(BROKEN))
def test_layouts_the_instances_decline_fall_back(torch_cuda, lz, oracle, family, layout):
    c, a, n, d, iw, ih = FAMILIES[family]
    kid = INSTANCE_OF[(c, a, n, d)]
    kw = dict(BROKEN[layout])
    nf = kw.pop("frames", 1)
    frames = [noise_hwc(oracle, ih, iw, c, seed=f + 1) for f in range(nf)]
    frames[-1][: ih // 2] = dark_hwc(oracle, ih // 2, iw, c, seed=9)
    ow, oh = iw * n // d, ih * n // d
    for flags, variant in ((0, oracle.VERBATIM), (lz.FLAG_NO_ALIAS, oracle.CLEAN)):
        twin = {k: 16 for k in kw}                                          # the same offsets, aligned
        for args, want_kid in ((kw, 0), (twin, kid)):
            outs, got_kid = launch_raw(torch_cuda, lz, frames, ow, oh, a, n, d, flags=flags, **args)
            assert got_kid == want_kid, (family, layout, args, got_kid)
            for f, img in enumerate(frames):
                assert np.array_equal(outs[f], oracle.upscale(img, ow, oh, a, n, d, variant=variant)), (layout, args, f)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [  # in_w, in_h, out_w, out_h, N, D, a, C
    (15, 15, 35, 35, 7, 3, 3, 3), (15, 15, 35, 35, 7, 3, 3, 1), (7, 7, 9, 9, 9, 7, 2, 3), (33, 21, 41, 26, 5, 4, 3, 3),
    (31, 17, 77, 42, 5, 2, 4, 1), (45, 23, 120, 61, 8, 3, 1, 2), (29, 30, 58, 60, 2, 1, 3, 3),
], ids=lambda s: "%dx%d_%dx%d_%d_%d_a%d_c%d" % s)
def test_host_entry_points_accept_what_the_device_accepts(torch_cuda, lz, oracle, case):
    """The host drivers run odd widths on a widened image in their own buffers.  Columns the widening adds must not
    change which descriptors are accepted: 7/3 at 15 -> 35 and 9/7 at 7 -> 9 pass the reference's float floor on every
    coordinate the caller sees, but not on the added ones."""
    iw, ih, ow, oh, n, d, a, c = case
    img = noise_hwc(oracle, ih, iw, c, seed=iw)
    img[: ih // 2, : iw // 2] = dark_hwc(oracle, ih // 2, iw // 2, c, seed=3)
    want = oracle.upscale(img, ow, oh, a, n, d)
    dev, _ = run_device(torch_cuda, lz, img, ow, oh, a, n, d, 0, stats=False)
    assert np.array_equal(dev, want)
    assert np.array_equal(lz.upscale(img, ow, oh, a=a, scale_n=n, scale_d=d), want), "upscale"
    assert np.array_equal(lz.upscale_bands_multi_gpu(img, ow, oh, [0, 0], a=a, scale_n=n, scale_d=d), want), "bands"
    got = lz.lanczos_expected(NTT.to_planar(img), ow, oh, a=a, scale_n=n, scale_d=d)
    assert np.array_equal(got, oracle.expected_planar(NTT.to_planar(img), ow, oh, a, n, d)), "lanczos_expected"
