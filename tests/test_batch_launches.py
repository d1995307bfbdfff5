"""The batch launches bench.py times, checked against the oracle, and batches past CUDA's 65,535-frame grid limit.

Small calls run the headline kernels' latency plan: everything resident at once, a few chunks per segment.  The
batches bench.py times take the batch branch of the segment planner instead -- a few long segments over several waves
of CTAs, the noisy mode persisting over hundreds of chunks, output frames gigabytes into the buffer.  Each case here
runs such a batch, asserts from lanczos_b200_get_launch that it really is in that regime, and compares with the oracle:
a few whole frames, and in every frame the rows around every segment boundary and at the top and bottom.

Batches of more than 65,535 frames (or planes) run as frame groups, one launch each; those are checked frame by frame.
"""
import concurrent.futures

import numpy as np
import pytest

from harness import torch_cuda  # noqa: F401
from util import NEAR, NT, V_TOP, WIN, WRONG, config_rows, noise_hwc, planted_counts, smooth_hwc, strict_floor, v_image

CANARY = 0xA5
TAIL = 1 << 16          # canary bytes after the last output frame
EDGE_ROWS = 16          # top and bottom output rows checked in every frame
MAX_GRID_FRAMES = 65535

# name: (in_w, in_h, out_w, out_h, channels, a, N, D, frames, kernel id)
C2 = (1920, 1080, 3840, 2160, 3, 3, 2, 1, 64, 1)
C2_UNEVEN = (1920, 1077, 3840, 2154, 3, 3, 2, 1, 64, 1)
C3 = (2560, 1440, 3840, 2160, 4, 3, 3, 2, 256, 3)
C4 = (3840, 2160, 7680, 4320, 3, 3, 2, 1, 128, 1)
DYN = (1280, 720, 1920, 1080, 3, 3, 3, 2, 64, 6)


def cdiv(a, b):
    return -(-a // b)


# ---- near ties at the places long segments make special ---------------------------------------------

def relocate(i, targets, n, d, a):
    """The first row of `targets` with window i's phase where make_near_ties.classify gives the window its stored class,
    else None.  For 2/1 the weights of every row of a phase are identical, so that row keeps the class anyway (the CPU
    test below checks both)."""
    ph = (int(WIN["coord"][i]) * d) % n
    for yy in targets:
        if (yy * d) % n == ph and NT.classify(WIN["win"][i], yy, n, d, a)[0] == WIN["cls"][i]:
            return yy
    return None


def near_tie_rows(n, d, a, oh, boundary):
    """Output rows for the V windows of (n, d, a): {idx: row} for a frame with the segment boundary `boundary` (the
    first rows after it, and the last rows before it, which the segment's last chunk completes) and {idx: row} for the
    last frame (its last rows).  Windows that keep their class at none of those rows stay at their stored coordinate
    when it lies inside the frame."""
    span = 4 * n
    groups = [list(range(boundary, boundary + span)), list(range(boundary - span, boundary)),
              list(range(oh - span, oh - a * n // d))]
    mid, last = {}, {}
    for j, i in enumerate(config_rows(n, d, a)):
        g = j % 3
        yy = relocate(i, groups[g], n, d, a)
        if yy is None:
            yy = int(WIN["coord"][i])
            g = 0
            if not V_TOP <= yy < oh - 2 * a * n // d:
                continue
        (last if g == 2 else mid)[int(i)] = yy
    return mid, last


@pytest.mark.parametrize("shape", [C2, C3], ids=["c2", "c3"])
def test_relocated_windows_keep_their_class(oracle, shape):
    """Every window the batch tests plant, at the rows they plant it for any segment boundary the planner may choose
    (up to 8 segments), still has its stored class; and for 2/1 every row of a phase has the same weights."""
    iw, ih, ow, oh, c, a, n, d = shape[:8]
    vperiods = cdiv(oh, n)
    if (n, d) == (2, 1):
        w1 = NT.weights(1, n, d, a)[0]
        for yy in range(3, 2 * C4[3], 2):
            assert np.array_equal(NT.weights(yy, n, d, a)[0], w1), yy
    moved = 0
    for segs in range(2, 9):
        mid, last = near_tie_rows(n, d, a, oh, cdiv(vperiods, segs) * n)
        assert last, segs
        for rows in (mid, last):
            for i, yy in rows.items():
                moved += yy != int(WIN["coord"][i])
                assert NT.classify(WIN["win"][i], yy, n, d, a)[0] == WIN["cls"][i], (segs, i, yy)
    assert moved > 0


def test_oracle_bands_equal_the_whole_frame(oracle):
    """oracle.upscale(rows=) computes only what a band reads; it must give the rows of the whole-frame result,
    in place (VERBATIM, whose top rows read final output) and not."""
    for (iw, ih, n, d, a, c) in [(64, 40, 2, 1, 3, 3), (60, 41, 3, 2, 3, 4), (50, 30, 17, 10, 3, 1), (31, 23, 3, 1, 2, 2)]:
        img = noise_hwc(oracle, ih, iw, c, seed=iw)
        ow, oh = iw * n // d, ih * n // d
        for variant in (oracle.VERBATIM, oracle.CLEAN):
            full = oracle.upscale(img, ow, oh, a, n, d, variant=variant)
            for r0 in range(oh):
                for cnt in {1, min(3, oh - r0), oh - r0}:
                    band = oracle.upscale(img, ow, oh, a, n, d, variant=variant, rows=(r0, cnt))
                    assert np.array_equal(band, full[r0:r0 + cnt]), (iw, ih, n, d, variant, r0, cnt)


# ---- GPU helpers ------------------------------------------------------------------------------------

def need_memory(torch, nbytes):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes * 1.05:
        pytest.skip(f"needs {nbytes / 1e9:.1f} GB of device memory, {free / 1e9:.1f} GB free")


def fill_frames(torch, d_in, seed):
    """bench.py's content: even frames image-like, 128 + 90 sin(0.05x + c + 0.3f) cos(0.037y) + U[-8, 7], odd frames
    uniform noise, from a seeded generator on the device."""
    F, H, W, C = d_in.shape
    gen = torch.Generator(device=d_in.device)
    gen.manual_seed(seed)
    yy = torch.arange(H, device=d_in.device, dtype=torch.float32).view(H, 1, 1)
    xx = torch.arange(W, device=d_in.device, dtype=torch.float32).view(1, W, 1)
    cc = torch.arange(C, device=d_in.device, dtype=torch.float32).view(1, 1, C)
    for f in range(F):
        if f % 2 == 1:
            d_in[f] = torch.randint(0, 256, (H, W, C), dtype=torch.uint8, device=d_in.device, generator=gen)
        else:
            base = 128 + 90 * torch.sin(0.05 * xx + cc + 0.3 * f) * torch.cos(0.037 * yy)
            base += torch.randint(-8, 8, (H, W, C), device=d_in.device, generator=gen)
            d_in[f] = base.clamp_(0, 255).to(torch.uint8)


def canary_out(torch, shape):
    """An output batch inside a buffer filled with CANARY, TAIL bytes of it after the last frame."""
    n = int(np.prod(shape))
    buf = torch.full((n + TAIL,), CANARY, dtype=torch.uint8, device="cuda")
    return buf, buf[:n].view(shape)


def assert_tail(torch, buf, n_out):
    assert bool((buf[n_out:] == CANARY).all()), "canary bytes after the last frame were overwritten"


def checked_rows(oh, n, d, launch):
    """[(r0, r1)]: the top and bottom EDGE_ROWS and the rows within 3 chunks of every segment boundary."""
    rows = np.zeros(oh, bool)
    rows[:EDGE_ROWS] = rows[-EDGE_ROWS:] = True
    m = cdiv(3 * launch["chunk_rows"] * n, d)
    for b in range(launch["seg_periods"] * n, oh, launch["seg_periods"] * n):
        rows[max(0, b - m):b + m] = True
    edges = np.flatnonzero(np.diff(np.concatenate([[0], rows.astype(np.int8), [0]])))
    return list(zip(edges[0::2], edges[1::2]))


def compare_batch(torch, oracle, d_in, d_out, shape, launch, whole, variant):
    """Whole frames `whole`, the checked rows of every other frame; bit for bit against the oracle."""
    iw, ih, ow, oh, c, a, n, d = shape[:8]
    ranges = checked_rows(oh, n, d, launch)
    frames = range(d_out.shape[0])

    def one(f):
        img = d_in[f].cpu().numpy()
        bad = []
        for r0, r1 in ([(0, oh)] if f in whole else ranges):
            got = d_out[f, r0:r1].cpu().numpy()
            want = oracle.upscale(img, ow, oh, a, n, d, variant=variant, rows=(int(r0), int(r1 - r0)))
            ne = np.argwhere(got != want)
            if len(ne):
                bad.append((f, int(r0 + ne[0][0]), int(ne[0][1]), len(ne)))
        return bad

    with concurrent.futures.ThreadPoolExecutor(4) as ex:
        bad = [b for r in ex.map(one, frames) for b in r]
    assert not bad, f"{len(bad)} mismatching ranges; (frame, first row, column, bytes): {bad[:8]}"


def whole_frames(F):
    return {0, F - 1, 2 * (F // 4), 2 * (F // 4) + 1}    # first, last, an image-like and a noise frame from the middle


def run_batch(lz, d_in, d_out, shape, flags=0):
    a, n, d = shape[5:8]
    lz.upscale_batch_device(d_in, d_out, a=a, scale_n=n, scale_d=d, flags=flags)
    return lz.stats(), lz.launch()


def assert_regime(launch, shape, min_chunks=0):
    """Batch branch of the planner (cols * 4 > resident CTAs), more than one wave, at least min_chunks per segment."""
    a, n, d, F = shape[5:9]
    cols = launch["grid_x"] * launch["grid_z"]
    ctas = cols * launch["grid_y"]
    chunks = cdiv(launch["seg_periods"] * d + 2 * a - 1, launch["chunk_rows"])
    print("launch report", shape[:4], F, "frames:", launch, "chunks per segment", chunks)
    assert launch["main_launches"] == 1 and launch["grid_z"] == F, launch
    assert cols * 4 > launch["resident_ctas"], ("not the batch branch", launch)
    assert ctas > launch["resident_ctas"], ("one wave", launch)
    assert chunks >= min_chunks, (chunks, launch)
    return chunks


def batch_case(torch, lz, oracle, shape, seed, flags_list=(0,), min_chunks=0, plant=False):
    iw, ih, ow, oh, c, a, n, d, F, kid = shape
    n_in, n_out = F * ih * iw * c, F * oh * ow * c
    need_memory(torch, n_in + n_out + TAIL)
    d_in = torch.empty((F, ih, iw, c), dtype=torch.uint8, device="cuda")
    fill_frames(torch, d_in, seed)
    buf, d_out = canary_out(torch, (F, oh, ow, c))
    try:
        planted = []
        for flags in flags_list:
            st, launch = run_batch(lz, d_in, d_out, shape, flags)
            torch.cuda.synchronize()
            assert st["kernel_id"] == kid, st
            assert_regime(launch, shape, min_chunks)
            if plant and not planted:
                planted = plant_near_ties(torch, oracle, d_in, shape, launch)
                lz.enable_stats(True)
                try:
                    st, _ = run_batch(lz, d_in, d_out, shape, flags)
                    torch.cuda.synchronize()
                finally:
                    lz.enable_stats(False)
                assert st["strict_samples"] >= strict_floor(planted), (st, strict_floor(planted))
            variant = oracle.CLEAN if flags & lz.FLAG_NO_ALIAS else oracle.VERBATIM
            compare_batch(torch, oracle, d_in, d_out, shape, launch, whole_frames(F), variant)
            assert_tail(torch, buf, n_out)
        return launch
    finally:
        del d_in, d_out, buf
        torch.cuda.empty_cache()


def plant_near_ties(torch, oracle, d_in, shape, launch):
    """V windows just after the first segment boundary and in the last chunk before it (in a noise frame in the middle)
    and in the last rows of the last frame (noise too: F is even)."""
    iw, ih, ow, oh, c, a, n, d, F = shape[:9]
    mid, last = near_tie_rows(n, d, a, oh, launch["seg_periods"] * n)
    f_mid = 2 * (F // 4) + 1
    planted = []
    for f, rows in ((f_mid, mid), (F - 1, last)):
        img, p = v_image(oracle, n, d, a, c, base=d_in[f].cpu().numpy(), place=rows.get)
        for (_, _, _, i) in p:
            assert NT.classify(WIN["win"][i], rows[i], n, d, a)[0] == WIN["cls"][i]
        d_in[f].copy_(torch.from_numpy(img))
        planted += p
    counts = planted_counts(planted)
    assert counts[NEAR] + counts[WRONG] > 0, counts
    return planted


# ---- the batches bench.py times ---------------------------------------------------------------------

@pytest.mark.gpu
def test_c2_as_timed(torch_cuda, lz, oracle):
    """The headline batch, default flags (near ties planted in long segments) and FLAG_NO_ALIAS."""
    batch_case(torch_cuda, lz, oracle, C2, seed=2, flags_list=(0, lz.FLAG_NO_ALIAS), min_chunks=20, plant=True)


@pytest.mark.gpu
def test_c2_uneven_last_segment(torch_cuda, lz, oracle):
    launch = batch_case(torch_cuda, lz, oracle, C2_UNEVEN, seed=5)
    vperiods = cdiv(C2_UNEVEN[3], C2_UNEVEN[6])
    assert vperiods % launch["seg_periods"] != 0, ("the last segment is not shorter", launch)


@pytest.mark.gpu
def test_c3_as_timed(torch_cuda, lz, oracle):
    batch_case(torch_cuda, lz, oracle, C3, seed=3, min_chunks=50, plant=True)


@pytest.mark.gpu
def test_c4_as_timed(torch_cuda, lz, oracle):
    """128 8K frames (about 16 GB): the last output frame lies beyond 2^32 bytes."""
    iw, ih, ow, oh, c = C4[:5]
    assert (C4[8] - 1) * oh * ow * c > 1 << 32
    batch_case(torch_cuda, lz, oracle, C4, seed=4, min_chunks=150)


@pytest.mark.gpu
def test_dyn_batch(torch_cuda, lz, oracle):
    batch_case(torch_cuda, lz, oracle, DYN, seed=6)


@pytest.mark.gpu
def test_c2_tolerance_mode_batch(torch_cuda, lz):
    """FLAG_TOLERANCE_1LSB on the headline batch: every byte within 1 LSB of the exact batch, image-like frames
    nearly all identical."""
    torch = torch_cuda
    iw, ih, ow, oh, c, a, n, d, F, kid = C2
    need_memory(torch, F * (ih * iw + 2 * oh * ow) * c + TAIL)
    d_in = torch.empty((F, ih, iw, c), dtype=torch.uint8, device="cuda")
    fill_frames(torch, d_in, seed=7)
    exact = torch.empty((F, oh, ow, c), dtype=torch.uint8, device="cuda")
    run_batch(lz, d_in, exact, C2)
    buf, d_out = canary_out(torch, (F, oh, ow, c))
    st, launch = run_batch(lz, d_in, d_out, C2, lz.FLAG_TOLERANCE_1LSB)
    torch.cuda.synchronize()
    assert st["kernel_id"] == kid
    assert_regime(launch, C2)
    diff = (d_out.to(torch.int16) - exact.to(torch.int16)).abs_()
    assert int(diff.max()) <= 1
    same = int((diff[0::2] == 0).sum()) / diff[0::2].numel()
    print("tolerance mode: exact-match fraction on image-like frames", same, "on all", int((diff == 0).sum()) / diff.numel())
    assert same > 0.99999, same
    assert_tail(torch, buf, F * oh * ow * c)
    del d_in, exact, buf, d_out, diff
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_independent_single_frame_calls(torch_cuda, lz):
    """Eight c2 frames, one FLAG_INDEPENDENT call each into its own buffer on one stream, equal the exact batch."""
    torch = torch_cuda
    iw, ih, ow, oh, c, a, n, d, _, kid = C2
    F = 8
    d_in = torch.empty((F, ih, iw, c), dtype=torch.uint8, device="cuda")
    fill_frames(torch, d_in, seed=8)
    batch = torch.empty((F, oh, ow, c), dtype=torch.uint8, device="cuda")
    _, batch_launch = run_batch(lz, d_in, batch, C2)
    outs = [canary_out(torch, (oh, ow, c)) for _ in range(F)]
    for f in range(F):
        lz.upscale_device(d_in[f], outs[f][1], a=a, scale_n=n, scale_d=d, flags=lz.FLAG_INDEPENDENT)
        assert lz.stats()["kernel_id"] == kid
    single = lz.launch()
    torch.cuda.synchronize()
    print("batch launch", batch_launch, "single-frame launch", single)
    grid = lambda L: (L["grid_x"], L["grid_y"], L["grid_z"])   # noqa: E731
    assert grid(single) != grid(batch_launch) and single["grid_z"] == 1
    for f in range(F):
        assert torch.equal(outs[f][1], batch[f]), f
        assert_tail(torch, outs[f][0], oh * ow * c)


# ---- batches past the grid limit: frame groups ------------------------------------------------------

POOL = 7


def pool_images(oracle, c, h=16, w=16):
    return np.stack([smooth_hwc(oracle, h, w, c, seed=k) if k % 2 == 0 else noise_hwc(oracle, h, w, c, seed=k)
                     for k in range(POOL)])


def pooled_batch(torch, pool, F):
    """Frame f = pool[f % POOL] on the device."""
    idx = torch.arange(F, device="cuda") % POOL
    return torch.from_numpy(pool).cuda()[idx].contiguous(), idx


def assert_groups(torch, lz, d_out, buf, want_pool, idx, kid, launches_per_group=(1, 2)):
    """launches_per_group: the main kernel, and the alias-rows kernel unless the main kernel produced those rows."""
    torch.cuda.synchronize()
    st, launch = lz.stats(), lz.launch()
    print("frame groups:", launch, st)
    assert st["kernel_id"] == kid, st
    assert launch["main_launches"] >= 2 and launch["grid_z"] <= MAX_GRID_FRAMES, launch
    assert st["kernel_launches"] in [k * launch["main_launches"] for k in launches_per_group], (st, launch)
    want = torch.from_numpy(want_pool).cuda()
    F = d_out.shape[0]
    for f0 in range(0, F, 8192):               # in slices: the expected batch is built on the device
        f1 = min(F, f0 + 8192)
        ne = (d_out[f0:f1] != want[idx[f0:f1]]).reshape(f1 - f0, -1).any(1)
        bad = (torch.nonzero(ne).flatten() + f0).tolist()
        assert not bad, f"{len(bad)} frames differ from the oracle, first {bad[:8]}"
    assert_tail(torch, buf, d_out.numel())


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["v6", "dyn_3_2", "generic", "independent"])
def test_batch_past_the_grid_limit(torch_cuda, lz, oracle, case):
    """65,537 frames through lanczos_b200_upscale_batch: two frame groups."""
    torch = torch_cuda
    F, c, a = MAX_GRID_FRAMES + 2, 3, 3
    n, d, flags, kid, per_group = {"v6": (2, 1, 0, 1, (1, 2)), "dyn_3_2": (3, 2, 0, 6, (2,)),
                                   "generic": (2, 1, lz.FLAG_GENERIC_KERNEL, 0, (2,)),
                                   "independent": (2, 1, lz.FLAG_INDEPENDENT, 1, (1, 2))}[case]
    pool = pool_images(oracle, c)
    oh = ow = 16 * n // d
    want = np.stack([oracle.upscale(img, ow, oh, a, n, d) for img in pool])
    d_in, idx = pooled_batch(torch, pool, F)
    buf, d_out = canary_out(torch, (F, oh, ow, c))
    lz.upscale_batch_device(d_in, d_out, a=a, scale_n=n, scale_d=d, flags=flags)
    assert_groups(torch, lz, d_out, buf, want, idx, kid, per_group)
    if case == "generic":
        assert lz.stats()["alias_rows"] > 0          # the alias-rows kernel ran, once per group


@pytest.mark.gpu
def test_planar_past_the_grid_limit(torch_cuda, lz, oracle):
    """16,384 RGBA frames through lanczos_b200_upscale_planar: 65,536 one-channel planes."""
    torch = torch_cuda
    F, c = 16384, 4
    pool = np.stack([np.ascontiguousarray(p.transpose(2, 0, 1)) for p in pool_images(oracle, c)])
    want = np.stack([oracle.expected_planar(p, 32, 32, 3, 2, 1) for p in pool])
    d_in, idx = pooled_batch(torch, pool, F)
    buf, d_out = canary_out(torch, (F, c, 32, 32))
    lz.upscale_planar_device(d_in, d_out, a=3, scale_n=2, scale_d=1)
    assert_groups(torch, lz, d_out, buf, want, idx, 8)


@pytest.mark.gpu
def test_hls_mode_past_the_grid_limit(torch_cuda, lz, oracle):
    torch = torch_cuda
    F, c = MAX_GRID_FRAMES + 2, 3
    pool = pool_images(oracle, c)
    want = np.stack([oracle.hls_upscale(img, 2, a=3, bp=8) for img in pool])
    d_in, idx = pooled_batch(torch, pool, F)
    buf, d_out = canary_out(torch, (F, 32, 32, c))
    lz.upscale_hls_device(d_in, d_out, a=3)
    assert_groups(torch, lz, d_out, buf, want, idx, 101, (1,))


def test_planar_plane_count_overflow_is_rejected(lz):
    """n_frames * channels past INT32_MAX is a dimension error, not a wrapped count (checked before any device work)."""
    import ctypes as C
    desc = lz.make_desc(16, 16, 32, 32, 4, 3)
    rc = lz.lib().lanczos_b200_upscale_planar(C.byref(desc), C.c_void_p(16), C.c_void_p(16), 1 << 30, 0, 0, 0, None)
    assert rc == -2
