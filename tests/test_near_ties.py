"""Adversarial windows: reference sums that land on or next to an integer (tests/golden/near_ties.npz).

On noise and image-like content a sum is almost never close enough to an integer for the details of the exact path
to decide the output byte: which weights it uses (this coordinate's own or the phase table's), the tap order, whether
the multiply-add is fused, the global rather than band-local coordinate, and whether the guard really bounds the fp32
error.  tests/golden/make_near_ties.py found windows where each of these decides; here they are planted into images
(the rest is noise) and every kernel is compared bit for bit with the CPU oracle, which stays the truth.

  H windows: the 2a taps of output column xx in one row and channel.
  V windows: column blocks constant along each input row; inside them the horizontal result at an output column X is
  a known function q_X of the row value, so the rows of output row yy are set to values whose q_X is the window.
"""
import os

import numpy as np
import pytest

from harness import device_upscale, torch_cuda  # noqa: F401
from util import (EMPTY, NEAR, NT, SPECIALISED, TIE, V_TOP, WIN, WRONG, axis_tables, config_rows, h_image, noise_hwc,
                  planar, planted_counts, restate_planar, strict_floor, tap0, up_len, v_image)

HERE = os.path.dirname(os.path.abspath(__file__))


# ---- CPU tests ---------------------------------------------------------------------------------------

CONFIGS = [tuple(c) for c in NT.CONFIGS]


def test_windows_file_is_small_and_covers_every_config():
    assert os.path.getsize(os.path.join(HERE, "golden", "near_ties.npz")) < 1 << 20
    for (n, d, a) in CONFIGS:
        assert (len(config_rows(n, d, a)) == 0) == ((n, d, a) in EMPTY), (n, d, a)


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: "%d_%d_a%d" % c)
def test_stored_windows_keep_their_class(oracle, cfg):
    """Every window, re-evaluated from oracle_kernel, still has its recorded class, flags and nearest integer."""
    n, d, a = cfg
    for i in config_rows(n, d, a):
        cls, flags, k, dist = NT.classify(WIN["win"][i], int(WIN["coord"][i]), n, d, a)
        assert (cls, flags, k) == (WIN["cls"][i], WIN["flags"][i], WIN["k"][i]), (cfg, int(WIN["coord"][i]), WIN["win"][i])
        assert dist == WIN["dist"][i]
        if cls == TIE:
            assert dist <= NT.TIE_TOL
        elif cls == NEAR:
            assert dist <= NT.NEAR_TOL
        else:
            assert NT.WRONG_LO <= dist <= NT.WRONG_HI and flags & (NT.F_WRONG_OUTER | NT.F_WRONG_ASC)


def test_weights_are_the_oracles(oracle):
    for (n, d, a) in CONFIGS:
        xx = 1000 * n + 1
        w, first = NT.weights(xx, n, d, a)
        x = xx / (n / d)
        assert first == int(np.floor(x)) - a + 1
        for k in range(2 * a):
            assert w[k] == oracle.lib().oracle_kernel(x - (first + k), a)


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: "%d_%d_a%d" % c)
def test_builder_plants_every_class_in_both_passes(oracle, cfg):
    """The H and V pass of each configuration carry every non-empty class (V: at least half of its windows), and the
    planted taps hold the stored windows."""
    n, d, a = cfg
    taps = 2 * a
    stored = planted_counts([(int(i),) for i in config_rows(n, d, a)])
    img, hp = h_image(oracle, n, d, a, 3)
    assert planted_counts(hp) == stored
    for (r, ch, i) in hp:
        lo = tap0(int(WIN["coord"][i]), n, d, a)
        assert np.array_equal(img[r, lo:lo + taps, ch], WIN["win"][i][:taps])
    img, vp = v_image(oracle, n, d, a, 3)
    got = planted_counts(vp)
    below = planted_counts([(int(i),) for i in config_rows(n, d, a) if WIN["coord"][i] >= V_TOP])
    for cls in (TIE, WRONG, NEAR):
        assert got[cls] >= min(1, below[cls]) and 2 * got[cls] >= below[cls], (cls, got, below)


def restated_mid(img, n, d, a, out_w):
    c, h, w = img.shape
    wx, ix, vx = axis_tables(out_w, w, n, d, a)
    s = np.zeros((c, h, out_w))
    for k in range(2 * a):
        s = np.where(vx[:, k], s + img[:, :, ix[:, k]].astype(np.float64) * wx[:, k], s)
    return s


@pytest.mark.parametrize("cfg", [(3, 2, 3), (17, 10, 3), (3, 1, 2), (2, 1, 1)],
                         ids=lambda c: "%d_%d_a%d" % c)
def test_restatement_and_planted_sums(oracle, cfg):
    """The numpy restatement equals the oracle (upscale CLEAN and VERBATIM, expected_planar fast and literal) on the
    built images, and in it the planted H sums and the V windows' intermediate columns are the stored ones."""
    n, d, a = cfg
    taps = 2 * a
    himg, hp = h_image(oracle, n, d, a, 3)
    pl = planar(himg)
    ow, oh = up_len(pl.shape[2], n, d), up_len(pl.shape[1], n, d)
    mid = restated_mid(pl, n, d, a, ow)
    for (r, ch, i) in hp:
        xx = int(WIN["coord"][i])
        w, _ = NT.weights(xx, n, d, a)
        assert mid[ch, r, xx] == NT.seq_sum(WIN["win"][i][:taps], w)[0]
    for clean in (False, True):
        want = restate_planar(pl, ow, oh, a, n, d, clean)
        variant = oracle.CLEAN if clean else oracle.VERBATIM
        assert np.array_equal(oracle.expected_planar(pl, ow, oh, a, n, d, variant=variant, fast=True), want)
        assert np.array_equal(planar(oracle.upscale(himg, ow, oh, a, n, d, variant=variant)), want)
    img, vp = v_image(oracle, n, d, a, 3)
    pl = planar(img)
    ow, oh = up_len(pl.shape[2], n, d), up_len(pl.shape[1], n, d)
    mid = NT.quantise(restated_mid(pl, n, d, a, ow))
    for (b, ch, X, i) in vp:
        lo = tap0(int(WIN["coord"][i]), n, d, a)
        assert np.array_equal(mid[ch, lo:lo + taps, X], WIN["win"][i][:taps])
    for clean in (False, True):
        want = restate_planar(pl, ow, oh, a, n, d, clean)
        variant = oracle.CLEAN if clean else oracle.VERBATIM
        assert np.array_equal(planar(oracle.upscale(img, ow, oh, a, n, d, variant=variant)), want)
        if not clean:
            assert np.array_equal(oracle.expected_planar(pl, ow, oh, a, n, d, variant=variant, fast=False), want)


def test_compiled_reference_at_near_ties(oracle):
    """When oracle/_ref has been built, the reference's own lanczos_expected agrees with the oracle on planted images."""
    cfgs = [c for c in oracle.ref_configs() if (c[4], c[5], c[6]) in CONFIGS]
    if not cfgs:
        pytest.skip("oracle/_ref not built")
    for cfg in cfgs:
        iw, ih, ow, oh, n, d, a, c = cfg
        img = noise_hwc(oracle, ih, iw, c, seed=9)
        taps = 2 * a
        # the windows of this configuration whose taps fit the small image, one per row and channel
        slot = 0
        for i in config_rows(n, d, a):
            lo = tap0(int(WIN["coord"][i]), n, d, a)
            if lo + taps <= iw and slot < ih * c:
                img[slot // c, lo:lo + taps, slot % c] = WIN["win"][i][:taps]
                slot += 1
        pl = planar(img)
        assert np.array_equal(oracle.ref_expected_planar(pl, cfg), oracle.expected_planar(pl, ow, oh, a, n, d)), cfg


# ---- GPU tests ---------------------------------------------------------------------------------------

def check_image(torch, lz, oracle, img, planted, a, n, d, kid):
    ow, oh = up_len(img.shape[1], n, d), up_len(img.shape[0], n, d)
    want = oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM)
    got = device_upscale(torch, lz, img, ow, oh, a, n, d, stats=True)
    st = lz.stats()
    assert st["kernel_id"] == kid, st
    bad = np.argwhere(got != want)
    assert len(bad) == 0, ("kernel", kid, len(bad), bad[:8].tolist())
    assert st["strict_samples"] >= strict_floor(planted), (st, strict_floor(planted))
    got = device_upscale(torch, lz, img, ow, oh, a, n, d, flags=lz.FLAG_NO_ALIAS)
    assert lz.stats()["kernel_id"] == kid
    assert np.array_equal(got, oracle.upscale(img, ow, oh, a, n, d, variant=oracle.CLEAN)), ("no alias", kid)


@pytest.mark.gpu
@pytest.mark.parametrize("kid", sorted(SPECIALISED))
def test_every_kernel_instance_at_near_ties(torch_cuda, lz, oracle, kid):
    """H windows in a wide image, V windows in a tall one, coordinates up to ~27,650: bit-exact, on the exact path."""
    c, a, n, d = SPECIALISED[kid]
    img, hp = h_image(oracle, n, d, a, c, seed=kid)
    check_image(torch_cuda, lz, oracle, img, hp, a, n, d, kid)
    img, vp = v_image(oracle, n, d, a, c, seed=kid)
    check_image(torch_cuda, lz, oracle, img, vp, a, n, d, kid)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [(3, 3, 3, 2), (3, 3, 17, 10), (4, 3, 2, 1), (3, 1, 2, 1)], ids=lambda c: "c%d_a%d_%d_%d" % c)
def test_generic_kernel_at_near_ties(torch_cuda, lz, oracle, cfg):
    c, a, n, d = cfg
    for img, _ in (h_image(oracle, n, d, a, c, seed=3), v_image(oracle, n, d, a, c, seed=3)):
        ow, oh = up_len(img.shape[1], n, d), up_len(img.shape[0], n, d)
        got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d, flags=lz.FLAG_GENERIC_KERNEL)
        assert lz.stats()["kernel_id"] == 0
        assert np.array_equal(got, oracle.upscale(img, ow, oh, a, n, d))


@pytest.mark.gpu
@pytest.mark.parametrize("kid", [6, 3, 5, 11, 23], ids=str)
def test_bands_that_start_and_end_at_planted_rows(torch_cuda, lz, oracle, kid):
    """Bands whose first and last rows are planted V rows in the thousands: only a band can tell the global row index
    of the exact path from a band-local one of the same phase."""
    torch = torch_cuda
    c, a, n, d = SPECIALISED[kid]
    img, vp = v_image(oracle, n, d, a, c, seed=kid)
    ow, oh = up_len(img.shape[1], n, d), up_len(img.shape[0], n, d)
    want = oracle.upscale(img, ow, oh, a, n, d)
    rows = sorted({int(WIN["coord"][p[-1]]) for p in vp if WIN["coord"][p[-1]] >= 1000})
    assert len(rows) >= 2
    desc = lz.make_desc(img.shape[1], img.shape[0], ow, oh, c, a, n, d)
    for r0, r1 in [(rows[0], rows[1] + 1), (rows[1], rows[-1] + 1), (rows[-1], rows[-1] + 1)]:
        in0, inn = lz.band_input_rows(desc, r0, r1 - r0)
        d_in = torch.from_numpy(np.ascontiguousarray(img[in0:in0 + inn])).cuda()
        d_out = torch.zeros((r1 - r0, ow, c), dtype=torch.uint8, device="cuda")
        lz.upscale_band_device(desc, d_in, d_out, r0, r1 - r0, in0, inn)
        torch.cuda.synchronize()
        assert lz.stats()["kernel_id"] == kid
        assert np.array_equal(d_out.cpu().numpy(), want[r0:r1]), (r0, r1)


@pytest.mark.gpu
@pytest.mark.parametrize("kid", [1, 3, 5, 6], ids=str)
def test_batch_with_windows_in_a_later_frame(torch_cuda, lz, oracle, kid):
    torch = torch_cuda
    c, a, n, d = SPECIALISED[kid]
    for img, _ in (h_image(oracle, n, d, a, c, seed=11), v_image(oracle, n, d, a, c, seed=11)):
        h, w = img.shape[:2]
        ow, oh = up_len(w, n, d), up_len(h, n, d)
        frames = np.stack([noise_hwc(oracle, h, w, c, seed=12), noise_hwc(oracle, h, w, c, seed=13), img])
        d_in = torch.from_numpy(frames).cuda()
        d_out = torch.zeros((3, oh, ow, c), dtype=torch.uint8, device="cuda")
        lz.upscale_batch_device(d_in, d_out, a=a, scale_n=n, scale_d=d)
        torch.cuda.synchronize()
        assert lz.stats()["kernel_id"] == kid
        assert np.array_equal(d_out[2].cpu().numpy(), oracle.upscale(img, ow, oh, a, n, d))


@pytest.mark.gpu
@pytest.mark.parametrize("kid", [8, 9, 10, 11, 13, 15, 24], ids=str)
def test_planar_entry_point_at_near_ties(torch_cuda, lz, oracle, kid):
    torch = torch_cuda
    _, a, n, d = SPECIALISED[kid]
    for img, _ in (h_image(oracle, n, d, a, 3, seed=21), v_image(oracle, n, d, a, 3, seed=21)):
        pl = planar(img)
        ow, oh = up_len(pl.shape[2], n, d), up_len(pl.shape[1], n, d)
        d_out = torch.empty((3, oh, ow), dtype=torch.uint8, device="cuda")
        lz.upscale_planar_device(torch.from_numpy(pl).cuda(), d_out, a=a, scale_n=n, scale_d=d)
        torch.cuda.synchronize()
        assert lz.stats()["kernel_id"] == kid
        assert np.array_equal(d_out.cpu().numpy(), oracle.expected_planar(pl, ow, oh, a, n, d))


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [(3, 3, 2, 1), (3, 3, 3, 2), (3, 3, 17, 10)], ids=lambda c: "c%d_a%d_%d_%d" % c)
def test_host_pipeline_odd_width(lz, oracle, cfg):
    """The host driver widens odd rows to whole words in its own buffers and runs the image as row bands."""
    c, a, n, d = cfg
    img, _ = h_image(oracle, n, d, a, c, seed=31, odd=True)
    assert img.shape[1] % 2 == 1
    ow, oh = up_len(img.shape[1], n, d), up_len(img.shape[0], n, d)
    assert np.array_equal(lz.upscale(img, ow, oh, a=a, scale_n=n, scale_d=d), oracle.upscale(img, ow, oh, a, n, d))
    img, _ = v_image(oracle, n, d, a, c, seed=31)
    img = np.ascontiguousarray(img[:, :-1])
    ow, oh = up_len(img.shape[1], n, d), up_len(img.shape[0], n, d)
    assert np.array_equal(lz.upscale(img, ow, oh, a=a, scale_n=n, scale_d=d), oracle.upscale(img, ow, oh, a, n, d))


@pytest.mark.gpu
@pytest.mark.parametrize("kid", [1, 3, 5, 6, 9], ids=str)
def test_fast_aligned_and_tolerance_flags_at_near_ties(torch_cuda, lz, oracle, kid):
    """FLAG_FAST_ALIGNED: every interpolated row stays exact; FLAG_TOLERANCE_1LSB: every byte within 1 LSB."""
    c, a, n, d = SPECIALISED[kid]
    for img, _ in (h_image(oracle, n, d, a, c, seed=41), v_image(oracle, n, d, a, c, seed=41)):
        ow, oh = up_len(img.shape[1], n, d), up_len(img.shape[0], n, d)
        want = oracle.upscale(img, ow, oh, a, n, d)
        got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d, flags=lz.FLAG_FAST_ALIGNED)
        interp = (np.arange(oh) * d) % n != 0
        assert np.array_equal(got[interp], want[interp])
        got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d, flags=lz.FLAG_TOLERANCE_1LSB)
        assert lz.stats()["kernel_id"] == kid
        assert np.abs(got.astype(np.int16) - want.astype(np.int16)).max() <= 1
