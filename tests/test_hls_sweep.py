"""The fixed-point "HLS mode" over everything it accepts: a = 1..4, integer ratios n up to 127 / a, bit precision
1..12, C = 1..4, any output size, pitched and batched layouts.

CPU: the LUT of every accepted (a, n, bp), and a plain numpy restatement of the HLS image path written from the
citations of oracle/hls_oracle.c (not from its loops), against that oracle per sample and per image.  GPU: both
kernels (the generic lanczos_hls_kernel<C>, kernel id 100, and the six lanczos_hls_tile_kernel instances, id 101)
through the C ABI on canary-checked buffers, bit for bit against oracle.hls_upscale."""
import ctypes as C

import numpy as np
import pytest

from harness import CANARY, ERR_DIMS, canary_call, canary_layout, torch_cuda  # noqa: F401
from util import INSTANCES, noise_hwc

ERR_RATIO = -5
TILES = {(i.c, i.a, i.n): i.mask for i in INSTANCES if i.family == "hls_tile"}   # bit precision 8 only
ACCEPTED = [(a, n, bp) for a in range(1, 5) for n in range(1, 127 // a + 1) for bp in range(1, 13)]


def checker(h, w, c):
    """0/255 checkerboard: every window alternates between the extremes, so the de-ring clamp binds from both sides."""
    yy, xx = np.mgrid[0:h, 0:w]
    return np.repeat((((yy + xx) % 2) * 255).astype(np.uint8)[:, :, None], c, axis=2)


def content(oracle, kind, h, w, c, seed=0):
    if kind == "noise":
        return noise_hwc(oracle, h, w, c, seed=seed)
    if kind == "checker":
        return checker(h, w, c)
    return np.full((h, w, c), {"flat0": 0, "flat255": 255}[kind], np.uint8)


# ---- the LUT ---------------------------------------------------------------------------------------------------

def test_lut_on_every_accepted_triple(lz, oracle):
    assert len(ACCEPTED) == 3156
    for (a, n, bp) in ACCEPTED:
        lut = lz.hls_lut(a, n, bp)
        assert np.array_equal(lut, oracle.hls_lut(a, n, bp)), (a, n, bp)
        # whole-pixel distances: L(0) = 1 exactly, L(k) = 0 up to the +-1e-17 residue of sin(k pi), floored
        assert lut[0] == 1 << bp, (a, n, bp)
        assert set(lut[n::n].tolist()) <= {-1, 0}, (a, n, bp)
        assert lut[a * n] == 0


def test_lut_rejections(lz, oracle):
    for a in (1, 2, 4):                          # a * n = 128: kernel_t(i) wraps (kernel.cpp:42)
        with pytest.raises(lz.LanczosError) as e:
            lz.hls_lut(a, 128 // a)
        assert e.value.code == ERR_RATIO
        with pytest.raises(ValueError):
            oracle.hls_lut(a, 128 // a)
    for bp in (0, 13):
        with pytest.raises(lz.LanczosError) as e:
            lz.hls_lut(3, 2, bp)
        assert e.value.code == ERR_DIMS
        with pytest.raises(ValueError):
            oracle.hls_lut(3, 2, bp)
    buf = (C.c_int32 * 7)()
    assert lz.lib().lanczos_b200_hls_lut(3, 2, 8, buf, 6) == ERR_DIMS     # a * n + 1 = 7 entries needed
    assert lz.lib().lanczos_b200_hls_lut(3, 2, 8, buf, 7) == 0


def test_lut_has_the_pattern_of_every_tile_instance(lz):
    """launch_hls_tile runs a tile instance only when lut[0] = 2^8 and lut[k n] = -1 exactly for the bits k of its
    MASK (0 elsewhere); otherwise the call silently goes to the generic kernel.  The library's own LUT must match."""
    assert len(TILES) == 6
    for (c, a, n), mask in TILES.items():
        lut = lz.hls_lut(a, n, 8)
        assert lut[0] == 256
        assert sum(1 << k for k in range(1, a + 1) if lut[k * n] == -1) == mask, (c, a, n)
        assert all(lut[k * n] == 0 for k in range(1, a + 1) if not (mask >> k) & 1)


# ---- a plain restatement of the HLS image path -----------------------------------------------------------------
# Written from the citations in oracle/hls_oracle.c's header: weights LUT[|out - in*n|] (kernel.cpp:50-67), vertical
# pass first (lanczos.cpp:96), exact products summed into num_el_t = ap_fixed<10+bp, 10> with AP_WRAP and clamped to
# the two central taps (worker.cpp:45-78), the same on the intermediates with every product floored to bp fraction
# bits (worker.cpp:81-115), clamp_to_byte (worker.cpp:118-130), zeros above / left of the image and the last row /
# column replicated below / right (worker.cpp:170-198, :239-275).  Everything is int64; the wrap is explicit.

def r_wrap(x, bp):
    """Two's-complement wrap to the 10 + bp bits of num_el_t.  Wrapping is a ring homomorphism, so wrapping the
    whole sum equals wrapping after every +=."""
    half = np.int64(1) << (9 + bp)
    return (np.asarray(x, np.int64) + half) % (2 * half) - half


def r_dering(acc, c0, c1):
    return np.minimum(np.maximum(acc, np.minimum(c0, c1)), np.maximum(c0, c1))


def r_mac1(v, k, a, bp):
    """First pass on bytes v[..., 2a] with weights k[..., 2a] (units 2^-bp): exact sum, wrap, clamp."""
    v = np.asarray(v, np.int64)
    acc = r_wrap((np.asarray(k, np.int64) * v).sum(-1), bp)
    return r_dering(acc, v[..., a - 1] << bp, v[..., a] << bp)


def r_mac2(v, k, a, bp):
    """Second pass on fixed-point v[..., 2a]: each product floored to bp fraction bits, summed, wrap, clamp."""
    v = np.asarray(v, np.int64)
    acc = r_wrap(np.floor_divide(np.asarray(k, np.int64) * v, np.int64(1) << bp).sum(-1), bp)
    return r_dering(acc, v[..., a - 1], v[..., a])


def r_to_byte(raw, bp):
    """byte_el_t(num_el_t): the integer part, toward zero like a C cast, wrapped to 8 bits."""
    raw = np.asarray(raw, np.int64)
    q = np.sign(raw) * (np.abs(raw) >> bp)
    return (q & 0xFF).astype(np.uint8)


def r_axis(out_len, in_len, n, a, lut):
    """(clamped source index, inside-or-replicated mask, weight) of every tap of every output coordinate."""
    o = np.arange(out_len)[:, None]
    src = o // n - a + 1 + np.arange(2 * a)[None, :]        # nominal input index; it also indexes the LUT
    return np.clip(src, 0, in_len - 1), src >= 0, lut[np.abs(o - src * n)]


def r_hls_upscale(img, n, a, bp, out_w, out_h, lut):
    h, w, c = img.shape
    iy, vy, ky = r_axis(out_h, h, n, a, lut)
    col = np.where(vy[:, :, None, None], img[iy], 0)                      # [out_h][2a][w][c]
    mid = r_mac1(np.moveaxis(col, 1, -1), ky[:, None, None, :], a, bp)    # [out_h][w][c]
    ix, vx, kx = r_axis(out_w, w, n, a, lut)
    row = np.where(vx[None, :, :, None], mid[:, ix], 0)                   # [out_h][out_w][2a][c]
    return r_to_byte(r_mac2(np.moveaxis(row, 2, -1), kx[None, :, None, :], a, bp), bp)


def test_restated_samples_equal_the_oracle(oracle):
    """r_mac1 / r_mac2 / r_to_byte against oracle_hls_mac1 / _mac2 / _to_byte: every LUT phase of a few ratios and
    random kernels, some large enough that the 10 integer bits of num_el_t wrap; windows of random bytes, flat runs
    and 0/255 extremes."""
    L = oracle.lib()
    i32p, u8p = C.POINTER(C.c_int32), C.POINTER(C.c_uint8)
    rng = np.random.default_rng(12)
    n_wrapped = 0
    for a in range(1, 5):
        taps = 2 * a
        for bp in range(1, 13):
            kernels = []
            for n in (1, 2, 3, 5):
                lut = oracle.hls_lut(a, n, bp)
                kernels += [lut[np.abs(ph - (np.arange(taps) - a + 1) * n)] for ph in range(n)]
            kernels += [rng.integers(-(1 << bp), 1 << bp, size=taps) for _ in range(3)]
            kernels += [rng.integers(-(1 << (bp + 3)), 1 << (bp + 3), size=taps) for _ in range(3)]   # wrap
            for k in kernels:
                k = np.ascontiguousarray(k, np.int32)
                kp = k.ctypes.data_as(i32p)
                v1 = rng.integers(0, 256, size=(6, taps)).astype(np.uint8)
                v1[1] = rng.integers(0, 256)
                v1[2] = rng.choice([0, 255], size=taps)
                v2 = rng.integers(0, 256 << bp, size=(6, taps)).astype(np.int32)
                v2[1] = rng.integers(0, 256 << bp)
                v2[2] = rng.choice([0, (256 << bp) - 1], size=taps)
                want1 = [L.oracle_hls_mac1(np.ascontiguousarray(v).ctypes.data_as(u8p), kp, a, bp) for v in v1]
                want2 = [L.oracle_hls_mac2(np.ascontiguousarray(v).ctypes.data_as(i32p), kp, a, bp) for v in v2]
                assert r_mac1(v1, k, a, bp).tolist() == want1, (a, bp, k.tolist())
                assert r_mac2(v2, k, a, bp).tolist() == want2, (a, bp, k.tolist())
                n_wrapped += int((np.abs((k.astype(np.int64) * v1).sum(-1)) >= 1 << (9 + bp)).sum())
                raw = np.array(want1 + want2 + rng.integers(-(512 << bp), 512 << bp, size=8).tolist() + [-1, 1])
                assert r_to_byte(raw, bp).tolist() == [L.oracle_hls_to_byte(int(x), bp) for x in raw], (a, bp)
    assert n_wrapped > 100      # the wrap is exercised, not only restated


def restate_cases():
    """A covering set: every (a, n, bp) of a = 1..4, n in {1, 2, 3, 5, 8, 127 // a}, bp in {1, 2, 7, 8, 12}, with C,
    the shape and the content cycling through their own lists.  Shapes (in_w, in_h, out_w(w, n), out_h(h, n)):
    1x1, inputs narrower than 2a, outputs wider and narrower than in x n, taller than in_h x n, and from in_h up."""
    shapes = [(1, 1, lambda w, n: w * n, lambda h, n: h * n),
              (None, 5, lambda w, n: w * n + n + 1, lambda h, n: h * n + 2 * n + 1),     # None: 2a - 1
              (7, 4, lambda w, n: max(1, w * n - n // 2 - 1), lambda h, n: h * n),
              (9, 6, lambda w, n: w * n, lambda h, n: h),
              (3, 2, lambda w, n: w * n + 1, lambda h, n: h * n + 1),
              (1, 3, lambda w, n: max(1, n - 1), lambda h, n: h * n + n)]
    kinds = ["noise", "checker", "flat0", "flat255", "noise"]
    cases = []
    i = 0
    for a in range(1, 5):
        for n in sorted({1, 2, 3, 5, 8, 127 // a}):
            for bp in (1, 2, 7, 8, 12):
                w, h, fw, fh = shapes[i % len(shapes)]
                w = 2 * a - 1 if w is None else w
                if n > 16:                               # keep the output small at the largest ratios
                    w, h = min(w, 2), min(h, 2)
                cases.append((a, n, bp, 1 + i % 4, w, h, fw(w, n), fh(h, n), kinds[i % len(kinds)]))
                i += 1
    return cases


def test_restated_images_equal_the_oracle(oracle):
    cases = restate_cases()
    assert {c[0] for c in cases} == {1, 2, 3, 4} and {c[3] for c in cases} == {1, 2, 3, 4}
    assert len({c[8] for c in cases}) == 4
    for (a, n, bp, c, w, h, ow, oh, kind) in cases:
        img = content(oracle, kind, h, w, c, seed=a * 1000 + n * 10 + bp)
        want = oracle.hls_upscale(img, n, a, bp, out_w=ow, out_h=oh)
        got = r_hls_upscale(img, n, a, bp, ow, oh, oracle.hls_lut(a, n, bp))
        assert want.shape == (oh, ow, c)
        assert np.array_equal(got, want), (a, n, bp, c, w, h, ow, oh, kind)


def crop_valid_rows(in_h, r0, r1, n, a):
    """Output rows [lo, hi) of the upscale of input rows [r0, r1) that equal rows n*r0 + lo .. n*r0 + hi of the whole
    image's upscale (integer scale n, out_h = in_h * n): those whose taps lie inside the crop.  At the image's own
    top or bottom the crop's border rule is the image's."""
    lo = 0 if r0 == 0 else (a - 1) * n
    hi = (r1 - r0) * n if r1 == in_h else (r1 - r0 - a) * n
    return lo, hi


def test_crop_rule(oracle):
    """The rule test_output_past_2_gib relies on, checked on a small image for every a."""
    for a in range(1, 5):
        img = noise_hwc(oracle, 40, 9, 3, seed=a)
        whole = oracle.hls_upscale(img, 3, a, 8)
        for (r0, r1) in [(0, 12), (10, 25), (28, 40), (0, 40)]:
            lo, hi = crop_valid_rows(40, r0, r1, 3, a)
            part = oracle.hls_upscale(img[r0:r1], 3, a, 8)
            assert np.array_equal(part[lo:hi], whole[3 * r0 + lo:3 * r0 + hi]), (a, r0, r1)


# ---- GPU: the parameter sweep ----------------------------------------------------------------------------------

def tile_geometry(c, a, n):
    """(TW, TH) of HlsGeo<C, A, N> in lanczos_hls.cu: the output tile of a tile instance."""
    tix = ((256 // c - (2 * a - 1)) // 4) * 4
    return tix * n, 12 * n


def kernel_of(c, a, n, bp):
    return 101 if bp == 8 and (c, a, n) in TILES else 100


def sweep_cells():
    """A covering array over a x n x bp x C: every (a, bp) pair of a = 1..4 and bp = 1..12, with n cycling through
    {1, 2, 3, 4, 5, 8, 127 // a} and C through 1..4 (so every (a, n) and (a, C) pair occurs), plus the six tile
    configurations at bp 8 and their generic neighbours (same C, a, n at bp 7 and 9; bp 8 at a C without a tile)."""
    cells = set()
    for a in range(1, 5):
        ns = [1, 2, 3, 4, 5, 8, 127 // a]
        for i, bp in enumerate(range(1, 13)):
            cells.add((a, ns[(i + a) % len(ns)], bp, 1 + (i + 2 * a) % 4))
    for (c, a, n) in TILES:
        cells |= {(a, n, 8, c), (a, n, 7, c), (a, n, 9, c)}
    cells |= {(3, 2, 8, 2), (2, 2, 8, 4), (3, 4, 8, 1), (2, 4, 8, 4), (4, 2, 8, 3), (1, 2, 8, 3), (3, 3, 8, 3)}
    return sorted(cells)


CELLS = sweep_cells()


def sweep_shapes(c, a, n, bp):
    """(in_w, in_h, out_w, out_h) that straddle the output tile of the kernel that runs: one tile -1, exactly one
    tile, +1 (each axis), less than one tile, and in x n just past one tile.  Inputs are the fewest pixels that cover
    the output, so most outputs are narrower or shorter than in x n.  The input of the small output is 3 columns
    wider than that (and up to 2 rows taller, keeping out_h >= in_h): the input's last column is not the one under
    the last output pixel."""
    tw, th = tile_geometry(c, a, n) if kernel_of(c, a, n, bp) == 101 else (64, 32)
    outs = [(tw - 1, th + 1), (tw, th), (tw + 1, th - 1)]
    shapes = [(-(-ow // n), -(-oh // n), ow, oh) for (ow, oh) in outs]
    ow, oh = max(1, tw // 3 - 1), max(1, th // 2 - 1)
    iw, ih = -(-(tw + 1) // n), -(-(th + 1) // n)
    return shapes + [(-(-ow // n) + 3, min(oh, -(-oh // n) + 2), ow, oh), (iw, ih, iw * n, ih * n)]


def run_hls(torch, lz, oracle, imgs, a, n, bp, ow, oh, **layout):
    """canary_call of upscale_hls on the frames `imgs`; asserts every frame against the oracle, returns kernel_id."""
    ih, iw, c = imgs[0].shape
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, 1)
    outs, st, _ = canary_call(torch, lz, desc, imgs, "upscale_hls", bit_precision=bp, **layout)
    for f, (img, out) in enumerate(zip(imgs, outs)):
        want = oracle.hls_upscale(img, n, a, bp, out_w=ow, out_h=oh)
        if not np.array_equal(out, want):
            bad = np.argwhere(out != want)
            raise AssertionError(("mismatch", (a, n, bp, c), (iw, ih, ow, oh), layout, "frame", f, len(bad),
                                  bad[:4].tolist()))
    return st["kernel_id"]


def test_sweep_covers_every_corner():
    assert {x[0] for x in CELLS} == {1, 2, 3, 4}
    assert {x[2] for x in CELLS} == set(range(1, 13))
    assert {x[3] for x in CELLS} == {1, 2, 3, 4}
    for a in range(1, 5):
        assert {x[1] for x in CELLS if x[0] == a} >= {1, 2, 3, 4, 5, 8, 127 // a}
        assert {x[2] for x in CELLS if x[0] == a} == set(range(1, 13))
        assert {x[3] for x in CELLS if x[0] == a} == {1, 2, 3, 4}
    assert {(c, a, n) for (a, n, bp, c) in CELLS if kernel_of(c, a, n, bp) == 101} == set(TILES)
    assert tile_geometry(3, 3, 2) == (160, 24)
    for (a, n, bp, c) in CELLS:
        for (iw, ih, ow, oh) in sweep_shapes(c, a, n, bp):
            assert oh >= ih and ow <= iw * n and oh <= ih * n, ((a, n, bp, c), (iw, ih, ow, oh))


@pytest.mark.gpu
@pytest.mark.parametrize("cell", CELLS, ids=lambda x: "a%d_n%d_bp%d_c%d" % x)
def test_sweep(torch_cuda, lz, oracle, cell):
    a, n, bp, c = cell
    for k, (iw, ih, ow, oh) in enumerate(sweep_shapes(c, a, n, bp)):
        for kind in ("noise", "checker"):
            img = content(oracle, kind, ih, iw, c, seed=k)
            kid = run_hls(torch_cuda, lz, oracle, [img], a, n, bp, ow, oh, seed=k)
            assert kid == kernel_of(c, a, n, bp), (cell, kid)


# ---- GPU: output sizes that are not in x n ---------------------------------------------------------------------

SIZE_CFGS = [(3, 3, 2, 8), (1, 3, 2, 8), (3, 2, 4, 8), (3, 3, 2, 10), (4, 4, 3, 12), (2, 1, 5, 5)]
NOT_IN_TIMES_N = {
    # out_w <= in_w * n: every tap column the kernels clamp lies inside the input
    "narrower": lambda iw, ih, n: [(iw * n - 2 * n - 1, ih * n), (iw * n - 1, ih * n - n + 1), (iw, ih * n + 1),
                                   (iw * n - n + 1, ih)],
    # replicated right columns and bottom rows
    "wider": lambda iw, ih, n: [(iw * n + 2 * n + 3, ih * n), (iw * n, ih * n + 3 * n + 2), (iw * n + 5, ih),
                                (iw * n + 1, ih * n + n - 1)],
}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(NOT_IN_TIMES_N))
@pytest.mark.parametrize("cfg", SIZE_CFGS, ids=lambda x: "c%d_a%d_n%d_bp%d" % x)
def test_output_sizes_that_are_not_in_times_n(torch_cuda, lz, oracle, cfg, kind):
    """Outputs narrower or wider than in x n, taller, and shorter down to out_h = in_h, for both kernels."""
    c, a, n, bp = cfg
    iw, ih = 97, 41
    for k, (ow, oh) in enumerate(NOT_IN_TIMES_N[kind](iw, ih, n)):
        img = noise_hwc(oracle, ih, iw, c, seed=k) if k % 2 == 0 else checker(ih, iw, c)
        kid = run_hls(torch_cuda, lz, oracle, [img], a, n, bp, ow, oh, seed=k)
        assert kid == kernel_of(c, a, n, bp)


# ---- GPU: layouts ------------------------------------------------------------------------------------------------

LAYOUT_CFGS = [(3, 3, 2, 8), (1, 3, 2, 8), (4, 3, 2, 8), (3, 2, 4, 8), (3, 3, 2, 10), (2, 4, 3, 12)]


def layout_size(c, a, n, bp):
    """An output width whose rows are whole words (so the pitch alone decides the word-store path) and end in a
    partial run of the tile kernel: one tile + 12 pixels wide, 1.5 tiles tall."""
    tw, th = tile_geometry(c, a, n) if kernel_of(c, a, n, bp) == 101 else (64, 32)
    iw = -(-(tw + 12) // n)
    while (iw * n * c) % 4:
        iw += 1
    return iw, -(-(th * 3 // 2) // n)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", LAYOUT_CFGS, ids=lambda x: "c%d_a%d_n%d_bp%d" % x)
def test_layouts(torch_cuda, lz, oracle, cfg):
    """Odd padded input pitch and an input base offset; output pitch = 0 and != 0 mod 4 at base offsets 0..3 (the
    tile kernel's word stores and its byte stores); frames with gaps between them and different content each."""
    c, a, n, bp = cfg
    iw, ih = layout_size(c, a, n, bp)
    ow, oh = iw * n, ih * n
    kid = kernel_of(c, a, n, bp)
    img = noise_hwc(oracle, ih, iw, c, seed=5)
    assert run_hls(torch_cuda, lz, oracle, [img], a, n, bp, ow, oh, in_off=3, in_pad=5, seed=1) == kid
    assert run_hls(torch_cuda, lz, oracle, [img], a, n, bp, ow, oh, in_off=1, in_pad=(-iw * c) % 16 + 16, seed=2) == kid
    for out_pad in (0, 4, 1, 3):                # (ow * c) % 4 == 0: pitch mod 4 = 0, 0, 1, 3
        for out_off in range(4):
            got = run_hls(torch_cuda, lz, oracle, [img], a, n, bp, ow, oh, out_off=out_off, out_pad=out_pad,
                          seed=out_off)
            assert got == kid
    frames = [noise_hwc(oracle, ih, iw, c, seed=10 + f) for f in range(3)] + [checker(ih, iw, c)]
    assert run_hls(torch_cuda, lz, oracle, frames, a, n, bp, ow, oh, in_off=2, in_pad=3, in_gap=7, out_off=1,
                   out_pad=2, out_gap=5, seed=3) == kid
    assert run_hls(torch_cuda, lz, oracle, frames, a, n, bp, ow, oh, in_gap=64, out_gap=256, seed=4) == kid


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [(3, 3, 2, 8), (3, 3, 2, 10)], ids=lambda x: "c%d_a%d_n%d_bp%d" % x)
def test_zero_frames_write_nothing(torch_cuda, lz, cfg):
    torch = torch_cuda
    c, a, n, bp = cfg
    iw, ih = 90, 30
    rb = iw * n * c
    base, pitch, fstride, total = canary_layout(rb, ih * n, 2, 0, 4, 16)
    d_in = torch.randint(0, 256, (4 * ih * iw * c,), dtype=torch.uint8, device="cuda")
    buf = torch.full((total,), CANARY, dtype=torch.uint8, device="cuda")
    d = lz.make_desc(iw, ih, iw * n, ih * n, c, a, n, 1, iw * c, pitch)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lz.lib().lanczos_b200_upscale_hls(C.byref(d), C.c_void_p(d_in.data_ptr()),
                                           C.c_void_p(buf.data_ptr() + base), bp, 0, 0, fstride, 0, stream)
    torch.cuda.synchronize()
    assert rc == 0
    assert (buf.cpu().numpy() == CANARY).all()


# ---- GPU: one frame past 2 GiB of output --------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("bp", [8, 10], ids=["tile_bp8", "generic_bp10"])
def test_output_past_2_gib(torch_cuda, lz, oracle, bp):
    """16384^2 RGB x2: 3 GiB of output, every byte offset past 2^31 in the lower third.  The output starts as CANARY;
    the first band, the band holding byte 2^31 and the last band are compared with the oracle run on input-row crops
    (crop_valid_rows), and the bytes after the output must stay CANARY."""
    torch = torch_cuda
    a, n, c, side = 3, 2, 3, 16384
    ow = oh = side * n
    row = ow * c
    assert oh * row > 1 << 31
    gen = torch.Generator(device="cuda").manual_seed(bp)
    d_in = torch.randint(0, 256, (side, side, c), generator=gen, dtype=torch.uint8, device="cuda")
    buf = torch.full((oh * row + 4096,), CANARY, dtype=torch.uint8, device="cuda")
    d_out = buf[:oh * row].view(oh, ow, c)
    try:
        lz.upscale_hls_device(d_in, d_out, a=a, bit_precision=bp)
        torch.cuda.synchronize()
        assert lz.stats()["kernel_id"] == (101 if bp == 8 else 100)
        assert (buf[oh * row:].cpu().numpy() == CANARY).all()
        y31 = (1 << 31) // row                   # the output row that holds byte 2^31
        for (r0, r1) in [(0, 12), (y31 // n - 6, y31 // n + 6), (side - 12, side)]:
            lo, hi = crop_valid_rows(side, r0, r1, n, a)
            want = oracle.hls_upscale(d_in[r0:r1].cpu().numpy(), n, a, bp)[lo:hi]
            got = d_out[n * r0 + lo:n * r0 + hi].cpu().numpy()
            assert np.array_equal(got, want), (bp, r0, r1, int((got != want).sum()))
            if r0 > 0 and r1 < side:
                assert n * r0 + lo <= y31 < n * r0 + hi
    finally:
        del d_in, d_out, buf
        torch.cuda.empty_cache()
