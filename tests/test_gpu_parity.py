"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle.
Bar (BASELINE.json north_star): the software path is floating point, so <= 1 LSB is required;
this implementation is expected to be BIT-EXACT (exact-match fraction 1.0), which is what is asserted.
"""
import ctypes as C
import os

import numpy as np
import pytest

from harness import device_upscale, torch_cuda  # noqa: F401
from util import dark_hwc, diff_stats, golden_files, interleaved, noise_hwc, patchwork_hwc, planar, smooth_hwc

pytestmark = pytest.mark.gpu


SMALL = [  # in_w, in_h, n, d, a, c
    (96, 54, 2, 1, 3, 3), (96, 54, 2, 1, 2, 3), (96, 54, 3, 2, 3, 3), (100, 60, 17, 10, 3, 3),
    (64, 48, 3, 2, 3, 4), (54, 30, 3, 1, 2, 3), (37, 23, 2, 1, 3, 4), (50, 40, 17, 10, 2, 3),
    (33, 17, 4, 1, 3, 1), (131, 77, 2, 1, 3, 3), (129, 65, 3, 2, 3, 4), (70, 90, 5, 3, 3, 2),
    (40, 40, 1, 1, 3, 3), (200, 37, 2, 1, 4, 3), (45, 200, 2, 1, 1, 4), (97, 101, 7, 4, 3, 3),
]


@pytest.mark.parametrize("cfg", SMALL, ids=lambda c: "x".join(map(str, c)))
@pytest.mark.parametrize("kind", ["noise", "smooth", "dark"])
def test_small_images_bit_exact(torch_cuda, lz, oracle, cfg, kind):
    iw, ih, n, d, a, c = cfg
    ow, oh = oracle.out_dims(iw, ih, n, d)
    img = {"noise": noise_hwc, "smooth": smooth_hwc, "dark": dark_hwc}[kind](oracle, ih, iw, c, seed=iw)
    want = oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM)
    got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d)
    st = diff_stats(got, want)
    assert st["n_diff"] == 0, st
    want_clean = oracle.upscale(img, ow, oh, a, n, d, variant=oracle.CLEAN)
    got_clean = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d, flags=lz.FLAG_NO_ALIAS)
    assert np.array_equal(got_clean, want_clean)


@pytest.mark.parametrize("path", golden_files(), ids=os.path.basename)
def test_golden_fixtures_planar_api(torch_cuda, lz, path):
    """Outputs of the reference's own lanczos_expected, through the same-shaped planar entry point."""
    z = np.load(path)
    iw, ih, ow, oh, n, d, a, c = (int(v) for v in z["cfg"])
    got = lz.lanczos_expected(z["img_in"], ow, oh, a=a, scale_n=n, scale_d=d)
    assert np.array_equal(got, z["img_out"])


def test_structured_known_answers(torch_cuda, lz, oracle):
    # all-0, all-255 (non-unit DC gain), impulse (reads back the weight table), step edges, checkerboard
    h, w = 48, 64
    imgs = {
        "zero": np.zeros((h, w, 3), np.uint8),
        "full": np.full((h, w, 3), 255, np.uint8),
        "impulse": np.zeros((h, w, 3), np.uint8),
        "vstep": np.zeros((h, w, 3), np.uint8),
        "checker": np.zeros((h, w, 3), np.uint8),
    }
    imgs["impulse"][h // 2, w // 2] = 255
    imgs["vstep"][:, w // 2:] = 255
    yy, xx = np.mgrid[0:h, 0:w]
    imgs["checker"][((yy + xx) & 1) == 1] = 255
    for name, img in imgs.items():
        for (n, d) in [(2, 1), (3, 2), (17, 10)]:
            ow, oh = oracle.out_dims(w, h, n, d)
            want = oracle.upscale(img, ow, oh, 3, n, d)
            got = device_upscale(torch_cuda, lz, img, ow, oh, 3, n, d)
            assert np.array_equal(got, want), (name, n, d)
    assert not device_upscale(torch_cuda, lz, imgs["zero"], 128, 96, 3, 2, 1).any()


def test_batch_equals_single_frames(torch_cuda, lz, oracle):
    torch = torch_cuda
    f, ih, iw, c, n, d = 5, 40, 56, 4, 3, 2
    ow, oh = oracle.out_dims(iw, ih, n, d)
    frames = np.stack([noise_hwc(oracle, ih, iw, c, seed=s) for s in range(f)])
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.zeros((f, oh, ow, c), dtype=torch.uint8, device="cuda")
    lz.upscale_batch_device(d_in, d_out, a=3, scale_n=n, scale_d=d)
    torch.cuda.synchronize()
    got = d_out.cpu().numpy()
    for i in range(f):
        assert np.array_equal(got[i], oracle.upscale(frames[i], ow, oh, 3, n, d)), i


def test_pitched_input_keeps_the_tma_kernel(torch_cuda, lz, oracle):
    """Padded rows whose pitch is a multiple of 16 bytes (but not the row size) stay on the specialised kernels:
    the tensor map takes the pitch as its row stride (VERDICT r1 weak #10)."""
    torch = torch_cuda
    for (iw, ih, c, n, d, a, kid) in [(320, 45, 3, 2, 1, 3, 1), (256, 40, 4, 3, 2, 3, 3), (320, 33, 3, 17, 10, 3, 5)]:
        ow, oh = oracle.out_dims(iw, ih, n, d)
        img = noise_hwc(oracle, ih, iw, c, seed=iw + c)
        in_pitch, out_pitch = iw * c + 48, ow * c + 20
        buf_in = torch.full((3, ih, in_pitch), 0x77, dtype=torch.uint8, device="cuda")      # a batch of 3 padded frames
        for f in range(3):
            buf_in[f, :, : iw * c] = torch.from_numpy(np.roll(img, f, axis=0).reshape(ih, iw * c)).cuda()
        buf_out = torch.full((3, oh, out_pitch), 0xAB, dtype=torch.uint8, device="cuda")
        desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, in_pitch, out_pitch)
        rc = lz.lib().lanczos_b200_upscale_batch(C.byref(desc), C.c_void_p(buf_in.data_ptr()), C.c_void_p(buf_out.data_ptr()),
                                                 3, ih * in_pitch, oh * out_pitch, 0, None)
        assert rc == 0
        torch.cuda.synchronize()
        assert lz.stats()["kernel_id"] == kid, (iw, c, lz.stats())
        out = buf_out.cpu().numpy()
        for f in range(3):
            assert np.array_equal(out[f, :, : ow * c].reshape(oh, ow, c), oracle.upscale(np.roll(img, f, axis=0), ow, oh, a, n, d)), (iw, f)
        assert (out[:, :, ow * c:] == 0xAB).all()


def test_tolerance_mode_full_size(torch_cuda, lz, oracle):
    """LANCZOS_FLAG_TOLERANCE_1LSB at the headline size (1080p -> 2160p, several strips and segments per frame, a batch)
    against the bit-exact GPU output, which test_headline_config_full_size pins to the oracle: every byte within 1 LSB,
    > 99.999 % identical on image-like content, > 98 % on uniform noise."""
    torch = torch_cuda
    frames = np.stack([smooth_hwc(oracle, 1080, 1920, 3, seed=1), noise_hwc(oracle, 1080, 1920, 3, seed=2)])
    d_in = torch.from_numpy(frames).cuda()
    exact = torch.empty((2, 2160, 3840, 3), dtype=torch.uint8, device="cuda")
    tol = torch.empty_like(exact)
    lz.upscale_batch_device(d_in, exact, a=3, flags=lz.FLAG_NO_ALIAS)
    lz.upscale_batch_device(d_in, tol, a=3, flags=lz.FLAG_NO_ALIAS | lz.FLAG_TOLERANCE_1LSB)
    torch.cuda.synchronize()
    assert lz.stats()["kernel_id"] == 1
    diff = (exact.to(torch.int16) - tol.to(torch.int16)).abs()
    assert int(diff.max()) <= 1
    assert float((diff[0] == 0).float().mean()) > 0.99999
    assert float((diff[1] == 0).float().mean()) > 0.98
    # spot-check the exact batch against the oracle on a band of rows of the noise frame
    want = oracle.upscale(frames[1], 3840, 2160, 3, 2, 1, variant=oracle.CLEAN, rows=(1000, 64))
    assert np.array_equal(exact[1, 1000:1064].cpu().numpy(), want)


def test_independent_flag_single_frame_calls(torch_cuda, lz, oracle):
    """LANCZOS_FLAG_INDEPENDENT: one call per frame on ONE stream, launched with programmatic dependent launch and
    without waiting for the previous call; distinct buffers per frame, results identical to the batch launch, and
    work queued afterwards on the stream (the copy back) still sees every frame complete."""
    torch = torch_cuda
    f, ih, iw, c = 12, 270, 480, 3
    frames = np.stack([noise_hwc(oracle, ih, iw, c, seed=50 + s) for s in range(f)])
    d_in = torch.from_numpy(frames).cuda()
    d_batch = torch.zeros((f, 2 * ih, 2 * iw, c), dtype=torch.uint8, device="cuda")
    lz.upscale_batch_device(d_in, d_batch, a=3)
    for rep in range(3):
        d_out = torch.zeros_like(d_batch)
        for i in range(f):
            lz.upscale_device(d_in[i], d_out[i], a=3, flags=lz.FLAG_INDEPENDENT)
        got = d_out.cpu()                       # stream-ordered after the last launch
        assert torch.equal(got, d_batch.cpu()), rep
    assert np.array_equal(d_batch[0].cpu().numpy(), oracle.upscale(frames[0], 2 * iw, 2 * ih, 3, 2, 1))


def test_pitched_buffers(torch_cuda, lz, oracle):
    torch = torch_cuda
    ih, iw, c, n, d = 33, 50, 3, 2, 1
    ow, oh = 100, 66
    img = noise_hwc(oracle, ih, iw, c, seed=21)
    in_pitch, out_pitch = iw * c + 13, ow * c + 29
    buf_in = torch.zeros((ih, in_pitch), dtype=torch.uint8, device="cuda")
    buf_in[:, : iw * c] = torch.from_numpy(img.reshape(ih, iw * c)).cuda()
    buf_out = torch.full((oh, out_pitch), 0xAB, dtype=torch.uint8, device="cuda")
    desc = lz.make_desc(iw, ih, ow, oh, c, 3, n, d, in_pitch, out_pitch)
    rc = lz.lib().lanczos_b200_upscale(C.byref(desc), C.c_void_p(buf_in.data_ptr()), C.c_void_p(buf_out.data_ptr()), 0, None)
    assert rc == 0
    torch.cuda.synchronize()
    out = buf_out.cpu().numpy()
    assert np.array_equal(out[:, : ow * c].reshape(oh, ow, c), oracle.upscale(img, ow, oh, 3, n, d))
    assert (out[:, ow * c:] == 0xAB).all()   # padding untouched


def test_stream_shim_after_a_pitched_call_on_the_same_geometry(torch_cuda, lz, oracle):
    """Plans are cached per geometry and shared by callers with different row pitches: the packed-word shim
    must run on its own dense buffers even when a padded call created the plan first."""
    torch = torch_cuda
    lz.lib().lanczos_b200_clear_plans()
    ih, iw, ow, oh = 26, 40, 80, 52
    img = noise_hwc(oracle, ih, iw, 3, seed=31)
    want = oracle.upscale(img, ow, oh, 3, 2, 1)
    in_pitch, out_pitch = iw * 3 + 40, ow * 3 + 16
    buf_in = torch.zeros((ih, in_pitch), dtype=torch.uint8, device="cuda")
    buf_in[:, : iw * 3] = torch.from_numpy(img.reshape(ih, iw * 3)).cuda()
    buf_out = torch.zeros((oh, out_pitch), dtype=torch.uint8, device="cuda")
    desc = lz.make_desc(iw, ih, ow, oh, 3, 3, 2, 1, in_pitch, out_pitch)
    assert lz.lib().lanczos_b200_upscale(C.byref(desc), C.c_void_p(buf_in.data_ptr()), C.c_void_p(buf_out.data_ptr()), 0, None) == 0
    torch.cuda.synchronize()
    assert np.array_equal(buf_out.cpu().numpy()[:, : ow * 3].reshape(oh, ow, 3), want)
    words = img[..., 0].astype(np.uint32) | (img[..., 1].astype(np.uint32) << 8) | (img[..., 2].astype(np.uint32) << 16)
    out = lz.lanczos_stream(words, iw, ih, ow, oh).reshape(oh, ow)
    got = np.stack([(out >> (8 * i)) & 0xFF for i in range(3)], axis=-1).astype(np.uint8)
    assert np.array_equal(got, want)
    # and the dense device entry point after the padded one
    assert np.array_equal(device_upscale(torch, lz, img, ow, oh, 3, 2, 1), want)


@pytest.mark.parametrize("cfg", [(50, 33, 2, 1, 3), (64, 40, 2, 1, 3), (44, 30, 3, 2, 4)])
def test_host_api_pitched_buffers_keep_their_padding(torch_cuda, lz, oracle, cfg):
    """lanczos_b200_upscale_host with padded host rows: pixels only are read and written (ADVICE r1)."""
    iw, ih, n, d, c = cfg
    ow, oh = oracle.out_dims(iw, ih, n, d)
    frames = 7
    in_pitch, out_pitch = iw * c + 5, ow * c + 11
    h_in = np.full((frames, ih, in_pitch), 0x5A, np.uint8)
    imgs = [noise_hwc(oracle, ih, iw, c, seed=40 + f) for f in range(frames)]
    for f in range(frames):
        h_in[f, :, : iw * c] = imgs[f].reshape(ih, iw * c)
    h_in = np.ascontiguousarray(h_in.reshape(-1)[: frames * ih * in_pitch - 5])      # last row ends with its pixels
    h_out = np.full(frames * oh * out_pitch, 0xC3, np.uint8)
    desc = lz.make_desc(iw, ih, ow, oh, c, 3, n, d, in_pitch, out_pitch)
    for n_frames, streams in [(frames, 2), (1, 3)]:
        h_out[:] = 0xC3
        rc = lz.lib().lanczos_b200_upscale_host(C.byref(desc), h_in.ctypes.data_as(C.c_void_p), h_out.ctypes.data_as(C.c_void_p),
                                                n_frames, 0, 0, 0, streams)
        assert rc == 0
        out = h_out.reshape(frames, oh, out_pitch)
        for f in range(n_frames):
            assert np.array_equal(out[f, :, : ow * c].reshape(oh, ow, c), oracle.upscale(imgs[f], ow, oh, 3, n, d)), f
        assert (out[:, :, ow * c:] == 0xC3).all()
        assert (out[n_frames:] == 0xC3).all()


def test_reference_sample_size_takes_a_specialised_kernel(torch_cuda, lz, oracle):
    """The reference author's own configuration (lanczos.h:13-28): 162x89 -> 486x267, 3x, LANCZOS_A 2, planar like
    lanczos_expected.  162 pixels are not a whole number of words: the host drivers widen the image with zero columns
    (= dropped taps) inside their own device buffers, so the literal size still runs on lanczos_dyn (VERDICT r1 #2)."""
    for kind, maker in (("noise", noise_hwc), ("dark", dark_hwc)):
        img = maker(oracle, 89, 162, 3, seed=11)
        want = oracle.upscale(img, 486, 267, 2, 3, 1)
        got = lz.lanczos_expected(planar(img), 486, 267, a=2, scale_n=3, scale_d=1)
        assert lz.stats()["kernel_id"] == 13, lz.stats()
        assert np.array_equal(interleaved(got), want), kind
        got_i = lz.upscale(img, 486, 267, a=2, scale_n=3, scale_d=1)       # interleaved host path: 162*3 bytes -> 164*3
        assert lz.stats()["kernel_id"] == 12, lz.stats()
        assert np.array_equal(got_i, want), kind
    # odd widths of the headline ratio, host paths: widened to whole words, specialised kernel, same bytes
    for (iw, ih, c, kid) in [(131, 77, 3, 1), (37, 23, 3, 1), (50, 33, 1, 0)]:
        img = noise_hwc(oracle, ih, iw, c, seed=iw)
        want = oracle.upscale(img, 2 * iw, 2 * ih, 3, 2, 1)
        assert np.array_equal(lz.upscale(img, 2 * iw, 2 * ih), want), (iw, ih, c)
        if kid:
            assert lz.stats()["kernel_id"] == kid, (iw, lz.stats())
        many = lz.upscale_bands_multi_gpu(img, 2 * iw, 2 * ih, [0, 0])
        assert np.array_equal(many, want), (iw, ih, c)


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("cfg", [(120, 90, 17, 10, 3, 3), (64, 64, 2, 1, 3, 3), (90, 64, 3, 2, 3, 4)])
def test_row_bands_concatenate_to_full(torch_cuda, lz, oracle, cfg, world):
    """Each band sees only its own input rows (halo included) and uses global phases (SURVEY.md 8e)."""
    torch = torch_cuda
    from lanczos_hls_b200.sharding import band_range
    iw, ih, n, d, a, c = cfg
    ow, oh = oracle.out_dims(iw, ih, n, d)
    img = noise_hwc(oracle, ih, iw, c, seed=world)
    want = oracle.upscale(img, ow, oh, a, n, d)
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d)
    out = np.zeros_like(want)
    for rank in range(world):
        r0, r1 = band_range(oh, rank, world)
        in0, inn = lz.band_input_rows(desc, r0, r1 - r0)
        d_in = torch.from_numpy(np.ascontiguousarray(img[in0:in0 + inn])).cuda()
        d_out = torch.zeros((r1 - r0, ow, c), dtype=torch.uint8, device="cuda")
        lz.upscale_band_device(desc, d_in, d_out, r0, r1 - r0, in0, inn)
        torch.cuda.synchronize()
        out[r0:r1] = d_out.cpu().numpy()
    assert np.array_equal(out, want)


def test_band_argument_errors(torch_cuda, lz):
    torch = torch_cuda
    desc = lz.make_desc(64, 64, 128, 128, 3, 3)
    d_in = torch.zeros((10, 64, 3), dtype=torch.uint8, device="cuda")
    d_out = torch.zeros((16, 128, 3), dtype=torch.uint8, device="cuda")
    with pytest.raises(lz.LanczosError) as e:   # rows 32..47 need input rows 14..26, only 20..29 supplied
        lz.upscale_band_device(desc, d_in, d_out, 32, 16, 20, 10)
    assert e.value.code == -7
    with pytest.raises(lz.LanczosError) as e:
        lz.upscale_band_device(desc, d_in, d_out, 120, 16, 0, 10)
    assert e.value.code == -7
    assert lz.lib().lanczos_b200_upscale(C.byref(desc), None, None, 0, None) == -1
    # supplied rows must be rows of the image (ADVICE r1): negative start, negative count, past the last row
    for (r0, nr) in [(-2, 12), (0, -1), (60, 10)]:
        with pytest.raises(lz.LanczosError) as e:
            lz.upscale_band_device(desc, d_in, d_out, 0, 4, r0, nr)
        assert e.value.code == -7


def test_host_api_single_and_batch(torch_cuda, lz, oracle):
    img = noise_hwc(oracle, 300, 200, 3, seed=4)           # single frame: pipelined as row bands
    want = oracle.upscale(img, 400, 600, 3, 2, 1)
    assert np.array_equal(lz.upscale(img, 400, 600), want)
    frames = np.stack([noise_hwc(oracle, 40, 60, 4, seed=s) for s in range(9)])
    got = lz.upscale(frames, 90, 60, n_streams=2)         # 3/2 derived from 90/60
    for i in range(9):
        assert np.array_equal(got[i], oracle.upscale(frames[i], 90, 60, 3, 3, 2)), i
    many = lz.upscale_bands_multi_gpu(img, 400, 600, [0] * min(3, max(1, lz.device_count()) * 3))
    assert np.array_equal(many, want)


def test_packed_word_stream_shim(torch_cuda, lz, oracle):
    """24-bit words, channel 0 in bits 7:0 (worker.cpp:35-43), raster order in and out."""
    ih, iw = 30, 44
    img = noise_hwc(oracle, ih, iw, 3, seed=8)
    words = img[..., 0].astype(np.uint32) | (img[..., 1].astype(np.uint32) << 8) | (img[..., 2].astype(np.uint32) << 16)
    out = lz.lanczos_stream(words, iw, ih, 88, 60).reshape(60, 88)
    want = oracle.upscale(img, 88, 60, 3, 2, 1)
    got = np.stack([(out >> (8 * i)) & 0xFF for i in range(3)], axis=-1).astype(np.uint8)
    assert np.array_equal(got, want)
    assert (out >> 24 == 0).all()


def test_headline_config_full_size(torch_cuda, lz, oracle):
    """BASELINE config 2: 1920x1080 -> 3840x2160 RGB8, 2x, Lanczos-3, uniform noise, full frame."""
    img = noise_hwc(oracle, 1080, 1920, 3, seed=0)
    want = oracle.upscale(img, 3840, 2160, 3, 2, 1)
    got = device_upscale(torch_cuda, lz, img, 3840, 2160, 3, 2, 1)
    st = diff_stats(got, want)
    assert st["n_diff"] == 0, st


def test_config3_rgba_three_halves_full_size(torch_cuda, lz, oracle):
    """BASELINE config 3 (one frame of the batch): 2560x1440 -> 3840x2160 RGBA8, 3/2 via gcd."""
    img = smooth_hwc(oracle, 1440, 2560, 4, seed=1)
    want = oracle.upscale(img, 3840, 2160, 3, 3, 2)
    got = device_upscale(torch_cuda, lz, img, 3840, 2160, 3, 0, 0)
    assert np.array_equal(got, want)


def test_config5_shape_reduced_and_properties(torch_cuda, lz, oracle):
    """BASELINE config 5 geometry (x1.7 = 17/10, out = floor(in*17/10), unaligned output pitch) at
    2048^2 against the oracle, and band == full at 4096^2 on the GPU alone (size-independent)."""
    torch = torch_cuda
    from lanczos_hls_b200.sharding import band_range
    img = noise_hwc(oracle, 2048, 2048, 3, seed=2)
    ow = oh = 2048 * 17 // 10
    assert (ow * 3) % 16 != 0
    want = oracle.upscale(img, ow, oh, 3, 17, 10)
    assert np.array_equal(device_upscale(torch, lz, img, ow, oh, 3, 17, 10), want)
    big = np.tile(img, (2, 2, 1))
    bw = bh = 4096 * 17 // 10
    full = device_upscale(torch, lz, big, bw, bh, 3, 17, 10)
    desc = lz.make_desc(4096, 4096, bw, bh, 3, 3, 17, 10)
    for rank in range(8):
        r0, r1 = band_range(bh, rank, 8)
        in0, inn = lz.band_input_rows(desc, r0, r1 - r0)
        d_in = torch.from_numpy(np.ascontiguousarray(big[in0:in0 + inn])).cuda()
        d_out = torch.zeros((r1 - r0, bw, 3), dtype=torch.uint8, device="cuda")
        lz.upscale_band_device(desc, d_in, d_out, r0, r1 - r0, in0, inn)
        torch.cuda.synchronize()
        assert np.array_equal(d_out.cpu().numpy(), full[r0:r1]), rank


def c5_hashes():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c5_hash.txt")
    out = []
    if os.path.exists(path):
        for ln in open(path):
            if ln.strip() and not ln.startswith("#"):
                f = ln.split()
                out.append((int(f[0]), int(f[2]), f[8]))
    return out


@pytest.mark.parametrize("cfg", c5_hashes(), ids=lambda c: "%dsq" % c[0])
def test_config5_full_size_hash(torch_cuda, lz, oracle, cfg):
    """BASELINE configs[4] at its LITERAL size (16384^2 -> 27852^2, 17/10) against the oracle: the oracle's output
    was hashed once in the build container (tests/golden/make_c5_hash.py -> tests/golden/c5_hash.txt); here the same
    xorshift input is regenerated, upscaled as 8 row bands (each with its own halo rows) and the FNV-1a-64 of the
    interleaved result compared."""
    torch = torch_cuda
    from lanczos_hls_b200.sharding import band_range
    size, osize, want = cfg
    img = oracle.xorshift_bytes(size * size * 3, oracle.SEED + 5).reshape(size, size, 3)
    desc = lz.make_desc(size, size, osize, osize, 3, 3, 17, 10)
    out = np.empty((osize, osize, 3), np.uint8)
    for rank in range(8):
        r0, r1 = band_range(osize, rank, 8)
        in0, inn = lz.band_input_rows(desc, r0, r1 - r0)
        d_in = torch.from_numpy(img[in0:in0 + inn]).cuda()
        d_out = torch.empty((r1 - r0, osize, 3), dtype=torch.uint8, device="cuda")
        lz.upscale_band_device(desc, d_in, d_out, r0, r1 - r0, in0, inn)
        torch.cuda.synchronize()
        if (osize * 3) % 4 == 0:                 # 27852 * 3 bytes: whole words, the any-ratio kernel; 3481 * 3 is not
            assert lz.stats()["kernel_id"] == 5
        out[r0:r1] = d_out.cpu().numpy()
        del d_in, d_out
    assert "%016x" % oracle.fnv1a64(out) == want


def test_determinism_and_strict_counter(torch_cuda, lz, oracle):
    img = noise_hwc(oracle, 270, 480, 3, seed=6)
    a = device_upscale(torch_cuda, lz, img, 960, 540, 3, 2, 1)
    b = device_upscale(torch_cuda, lz, img, 960, 540, 3, 2, 1, stats=True)
    st = lz.stats()
    assert np.array_equal(a, b)
    assert st["kernel_launches"] >= 1 and st["alias_rows"] == 5
    assert st["strict_samples"] > 0      # noise always has sums near an integer


def test_fast_aligned_flag_is_within_one_lsb(torch_cuda, lz, oracle):
    """LANCZOS_FLAG_FAST_ALIGNED skips the exact re-evaluation of phase-0 ROWS: <= 1 LSB, and every
    mismatch sits on a phase-0 row where the reference returned v-1 (sin(k*pi) residues, SURVEY.md 7)."""
    for maker, seed in ((dark_hwc, 3), (noise_hwc, 4)):
        img = maker(oracle, 270, 480, 3, seed=seed)
        want = oracle.upscale(img, 960, 540, 3, 2, 1)
        got = device_upscale(torch_cuda, lz, img, 960, 540, 3, 2, 1, flags=lz.FLAG_FAST_ALIGNED)
        d = got.astype(np.int16) - want.astype(np.int16)
        assert np.abs(d).max() <= 1
        ys = np.nonzero(d)[0]
        assert (ys % 2 == 0).all()            # 2x: phase-0 rows are the even output rows
        assert (d[d != 0] == 1).all()         # we return v, the reference v-1
        exact = float((d == 0).mean())
        assert exact > 0.98, exact            # exact-match fraction stays above 98 % even on noise


SPECIALISED = [  # shapes that take the specialised (TMA + systolic) kernels: in_w, in_h, n, d, a, c, kernel_id
    (960, 540, 2, 1, 3, 3, 1), (240, 97, 2, 1, 3, 3, 1), (80, 41, 2, 1, 3, 3, 1), (400, 33, 2, 1, 3, 4, 2),
    (640, 360, 3, 2, 3, 4, 3), (124, 70, 3, 2, 3, 4, 3), (496, 301, 2, 1, 2, 3, 4),
    # any-ratio kernel (lanczos_dyn): the reference author's own sample configuration (lanczos.h:13-28: 162x89 ->
    # 486x267, 3x, LANCZOS_A 2; 160 wide here: the TMA kernels want input rows of a multiple of 16 bytes), then the other ratios,
    # tap counts and channel counts that used to fall to the generic kernel (VERDICT r1 missing #2)
    (160, 89, 3, 1, 2, 3, 12), (368, 121, 4, 1, 3, 3, 14), (240, 77, 5, 3, 3, 3, 16), (400, 90, 7, 4, 3, 3, 17),
    (248, 66, 2, 1, 3, 2, 18), (320, 75, 2, 1, 4, 3, 19), (320, 75, 2, 1, 1, 3, 20), (200, 61, 3, 1, 3, 4, 21),
    (160, 50, 4, 1, 3, 4, 22), (320, 90, 3, 2, 2, 3, 23), (1040, 140, 17, 10, 3, 3, 5), (512, 120, 3, 1, 3, 3, 7),
]


@pytest.mark.parametrize("cfg", SPECIALISED, ids=lambda c: "x".join(map(str, c)))
@pytest.mark.parametrize("kind", ["noise", "smooth", "dark"])
def test_specialised_kernels_bit_exact(torch_cuda, lz, oracle, cfg, kind):
    """Odd widths/heights on the specialised kernels: partial strips, partial chunks, several vertical segments."""
    iw, ih, n, d, a, c, kid = cfg
    if (iw * c) % 4 or (iw * n // d * c) % 4:
        pytest.skip("row bytes not a multiple of 4: generic kernel")
    ow, oh = oracle.out_dims(iw, ih, n, d)
    img = {"noise": noise_hwc, "smooth": smooth_hwc, "dark": dark_hwc}[kind](oracle, ih, iw, c, seed=iw + ih)
    want = oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM)
    got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d)
    assert lz.stats()["kernel_id"] == kid
    st = diff_stats(got, want)
    assert st["n_diff"] == 0, st


@pytest.mark.parametrize("cfg", [  # in_w, in_h, n, d, a, c, kernel id, patch rows, patch pixels
    (704, 420, 2, 1, 3, 3, 1, 37, 150), (704, 420, 2, 1, 3, 3, 1, 9, 40), (704, 300, 2, 1, 3, 3, 1, 150, 704),
    (512, 300, 3, 2, 3, 4, 3, 31, 100), (512, 300, 2, 1, 3, 4, 2, 23, 512),
], ids=lambda c: "x".join(map(str, c)))
def test_patchwork_content_switches_phase0_modes(torch_cuda, lz, oracle, cfg):
    """The phase-0 second look has three regimes inside one vertical segment of one strip -- filter clean, chunk flagged
    (exact chunk pass after the hot loop), warp in noisy mode (no filter, every phase-0 row from the exact chunk pass) --
    and switches between them at chunk boundaries: patches of image-like content, uniform noise and dark noise of
    several sizes (smaller than a chunk, a few chunks, wider than a strip) exercise every transition, whole image and as
    row bands."""
    iw, ih, n, d, a, c, kid, band, col = cfg
    ow, oh = oracle.out_dims(iw, ih, n, d)
    img = patchwork_hwc(oracle, ih, iw, c, seed=iw + band, band=band, col=col)
    want = oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM)
    got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d)
    assert lz.stats()["kernel_id"] == kid
    st = diff_stats(got, want)
    assert st["n_diff"] == 0, st
    # the same as three row bands (other segment boundaries, the flag state starts afresh in every band)
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d)
    out = np.zeros_like(want)
    edges = [0, oh // 3 + 1, 2 * oh // 3 - 1, oh]
    for r0, r1 in zip(edges[:-1], edges[1:]):
        in0, inn = lz.band_input_rows(desc, r0, r1 - r0)
        d_in = torch_cuda.from_numpy(np.ascontiguousarray(img[in0:in0 + inn])).cuda()
        d_out = torch_cuda.zeros((r1 - r0, ow, c), dtype=torch_cuda.uint8, device="cuda")
        lz.upscale_band_device(desc, d_in, d_out, r0, r1 - r0, in0, inn)
        torch_cuda.cuda.synchronize()
        out[r0:r1] = d_out.cpu().numpy()
    assert np.array_equal(out, want)


@pytest.mark.parametrize("cfg", [(960, 540, 2, 1, 3, 3), (640, 360, 3, 2, 3, 4), (240, 97, 2, 1, 3, 3)],
                         ids=lambda c: "x".join(map(str, c)))
def test_tolerance_mode_is_within_one_lsb(torch_cuda, lz, oracle, cfg):
    """LANCZOS_FLAG_TOLERANCE_1LSB (north star: "at most 1 LSB per channel with the exact-match fraction
    stated"): tolerance = 1 LSB on every byte; exact-match fraction > 0.9999 on image-like content and
    > 0.98 on uniform noise (where the reference itself returns v-1 for ~2 % of the phase-0 samples)."""
    iw, ih, n, d, a, c = cfg
    ow, oh = oracle.out_dims(iw, ih, n, d)
    for maker, floor in ((smooth_hwc, 0.9999), (noise_hwc, 0.98), (dark_hwc, 0.98)):
        img = maker(oracle, ih, iw, c, seed=5)
        want = oracle.upscale(img, ow, oh, a, n, d, variant=oracle.CLEAN)
        got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d, flags=lz.FLAG_TOLERANCE_1LSB | lz.FLAG_NO_ALIAS)
        dlt = np.abs(got.astype(np.int16) - want.astype(np.int16))
        assert dlt.max() <= 1                                  # the tolerance: 1 LSB
        exact = float((dlt == 0).mean())
        assert exact > floor, (maker.__name__, exact)
    # with the in-place top rows (default flags) the top rows are still produced exactly by the alias kernel
    img = smooth_hwc(oracle, ih, iw, c, seed=6)
    want = oracle.upscale(img, ow, oh, a, n, d, variant=oracle.VERBATIM)
    got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d, flags=lz.FLAG_TOLERANCE_1LSB)
    assert np.abs(got.astype(np.int16) - want.astype(np.int16)).max() <= 1


def test_generic_and_specialised_kernels_agree(torch_cuda, lz, oracle):
    """Both code paths must give the reference's bits (kernel_id tells which one ran)."""
    img = noise_hwc(oracle, 200, 320, 3, seed=12)
    want = oracle.upscale(img, 640, 400, 3, 2, 1)
    a = device_upscale(torch_cuda, lz, img, 640, 400, 3, 2, 1)
    ka = lz.stats()["kernel_id"]
    b = device_upscale(torch_cuda, lz, img, 640, 400, 3, 2, 1, flags=lz.FLAG_GENERIC_KERNEL)
    kb = lz.stats()["kernel_id"]
    assert ka == 1 and kb == 0
    assert np.array_equal(a, want) and np.array_equal(b, want)


def test_config4_shape_4k_to_8k_one_frame(torch_cuda, lz, oracle):
    """BASELINE config 4 (one frame of the batch): 3840x2160 -> 7680x4320 RGB8, 2x."""
    img = smooth_hwc(oracle, 2160, 3840, 3, seed=5)
    img[:300, :400] = noise_hwc(oracle, 300, 400, 3, seed=6)      # a noisy corner keeps the exact path busy
    want = oracle.upscale(img, 7680, 4320, 3, 2, 1)
    got = device_upscale(torch_cuda, lz, img, 7680, 4320, 3, 2, 1)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("cfg", [  # in_w, in_h, out_w, out_h, n, d, a, c: output sizes that are NOT in * N / D
    (64, 48, 120, 100, 2, 1, 3, 3), (64, 48, 140, 90, 2, 1, 3, 3), (240, 60, 484, 118, 2, 1, 3, 3),
    (90, 64, 132, 100, 3, 2, 3, 4), (50, 40, 80, 70, 17, 10, 3, 3), (33, 29, 70, 40, 2, 1, 2, 1),
])
@pytest.mark.parametrize("kind", ["noise", "smooth"])
def test_output_size_independent_of_ratio(torch_cuda, lz, oracle, cfg, kind):
    """OUT_WIDTH / OUT_HEIGHT are loop bounds only in the reference (full_TB.h:56,69): the ratio comes from
    SCALE_N / SCALE_D, and coordinates past the last input sample just lose taps (full_TB.h:59,72)."""
    iw, ih, ow, oh, n, d, a, c = cfg
    img = {"noise": noise_hwc, "smooth": smooth_hwc}[kind](oracle, ih, iw, c, seed=iw + oh)
    want = oracle.upscale(img, ow, oh, a, n, d)
    got = device_upscale(torch_cuda, lz, img, ow, oh, a, n, d)
    st = diff_stats(got, want)
    assert st["max"] == 0, st


PLANAR = [  # in_w, in_h, n, d, a, planes, expected kernel_id (0 = generic)
    (960, 540, 2, 1, 3, 3, 8), (240, 97, 2, 1, 3, 3, 8), (96, 54, 2, 1, 3, 1, 8), (640, 360, 3, 2, 3, 4, 9),
    (496, 301, 2, 1, 2, 3, 10), (240, 120, 17, 10, 3, 3, 11), (131, 77, 2, 1, 3, 3, 0), (90, 50, 5, 3, 3, 2, 0),
    # the reference's own sample configuration in the reference's own (planar) layout, and 3x / 4x planes with a = 3
    (160, 89, 3, 1, 2, 3, 13), (160, 89, 3, 1, 3, 3, 15), (160, 60, 4, 1, 3, 3, 24),
]


@pytest.mark.parametrize("cfg", PLANAR, ids=lambda c: "x".join(map(str, c)))
@pytest.mark.parametrize("kind", ["noise", "smooth", "dark"])
def test_planar_device_api_bit_exact(torch_cuda, lz, oracle, cfg, kind):
    """lanczos_b200_upscale_planar takes the arrays of lanczos_expected (full_TB.h:20-21, 79-96) as they are."""
    iw, ih, n, d, a, c, kid = cfg
    ow, oh = oracle.out_dims(iw, ih, n, d)
    img = planar({"noise": noise_hwc, "smooth": smooth_hwc, "dark": dark_hwc}[kind](oracle, ih, iw, c, seed=iw))
    want = oracle.expected_planar(img, ow, oh, a, n, d, fast=True)
    d_in = torch_cuda.from_numpy(img).cuda()
    d_out = torch_cuda.empty((c, oh, ow), dtype=torch_cuda.uint8, device="cuda")
    lz.upscale_planar_device(d_in, d_out, a=a, scale_n=n, scale_d=d)
    torch_cuda.cuda.synchronize()
    assert lz.stats()["kernel_id"] == kid
    st = diff_stats(d_out.cpu().numpy(), want)
    assert st["max"] == 0, st


def test_planar_batch_of_frames(torch_cuda, lz, oracle):
    f, c, ih, iw = 3, 3, 54, 96
    imgs = np.stack([planar(noise_hwc(oracle, ih, iw, c, seed=40 + i)) for i in range(f)])
    d_in = torch_cuda.from_numpy(imgs).cuda()
    d_out = torch_cuda.empty((f, c, 108, 192), dtype=torch_cuda.uint8, device="cuda")
    lz.upscale_planar_device(d_in, d_out, a=3)
    torch_cuda.cuda.synchronize()
    got = d_out.cpu().numpy()
    for i in range(f):
        assert np.array_equal(got[i], oracle.expected_planar(imgs[i], 192, 108, 3, 2, 1, fast=True))


def test_concurrent_host_threads(torch_cuda, lz, oracle):
    """The library is re-entrant (the reference is single-shot: globals lanczos.cpp:17-18, static pos :54): four host
    threads, each with its own stream and its own descriptors, get the reference's pixels."""
    import threading
    jobs = [(96, 54, 2, 1, 3, 3), (64, 48, 3, 2, 3, 4), (100, 60, 17, 10, 3, 3), (240, 97, 2, 1, 3, 3)]
    results, errors = {}, []

    def worker(idx):
        try:
            iw, ih, n, d, a, c = jobs[idx]
            ow, oh = oracle.out_dims(iw, ih, n, d)
            st = torch_cuda.cuda.Stream()
            for rep in range(6):
                img = noise_hwc(oracle, ih, iw, c, seed=100 * idx + rep)
                with torch_cuda.cuda.stream(st):
                    d_in = torch_cuda.from_numpy(img).cuda()
                    d_out = torch_cuda.empty((oh, ow, c), dtype=torch_cuda.uint8, device="cuda")
                    lz.upscale_device(d_in, d_out, a=a, scale_n=n, scale_d=d)
                st.synchronize()
                results[(idx, rep)] = (d_out.cpu().numpy(), img, (ow, oh, a, n, d))
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for (idx, rep), (got, img, (ow, oh, a, n, d)) in results.items():
        assert np.array_equal(got, oracle.upscale(img, ow, oh, a, n, d)), (idx, rep)


def test_planar_pitched_planes(torch_cuda, lz, oracle):
    """Planes with a row pitch larger than the width and planes that are not adjacent in memory."""
    c, ih, iw = 3, 54, 96
    img = planar(noise_hwc(oracle, ih, iw, c, seed=9))
    want = oracle.expected_planar(img, 192, 108, 3, 2, 1, fast=True)
    big_in = torch_cuda.zeros((c, ih + 3, iw + 32), dtype=torch_cuda.uint8, device="cuda")
    big_out = torch_cuda.full((c, 108 + 5, 192 + 64), 7, dtype=torch_cuda.uint8, device="cuda")
    big_in[:, :ih, :iw] = torch_cuda.from_numpy(img).cuda()
    lz.upscale_planar_device(big_in[:, :ih, :iw], big_out[:, :108, :192], a=3)
    torch_cuda.cuda.synchronize()
    got = big_out.cpu().numpy()
    assert np.array_equal(got[:, :108, :192], want)
    assert (got[:, 108:, :] == 7).all() and (got[:, :, 192:] == 7).all()      # nothing outside the planes is touched


@pytest.mark.parametrize("cfg", [  # in_w, in_h, n, d, a, c: one shape per specialised kernel family
    (240, 97, 2, 1, 3, 3), (124, 70, 3, 2, 3, 4), (240, 120, 17, 10, 3, 3), (96, 54, 3, 1, 3, 3), (37, 23, 2, 1, 3, 4),
])
def test_nothing_is_written_outside_the_output_rectangle(torch_cuda, lz, oracle, cfg):
    """Canary bytes around a pitched output (and below its last row) survive every kernel family."""
    iw, ih, n, d, a, c = cfg
    ow, oh = oracle.out_dims(iw, ih, n, d)
    img = noise_hwc(oracle, ih, iw, c, seed=3)
    pad = 64                                             # keeps pitch and base aligned for the specialised kernels
    big = torch_cuda.full((oh + 4, ow * c + pad), 0xA5, dtype=torch_cuda.uint8, device="cuda")
    d_out = big[:oh].as_strided((oh, ow, c), (ow * c + pad, c, 1))
    d_in = torch_cuda.from_numpy(img).cuda()
    lz.upscale_device(d_in, d_out, a=a, scale_n=n, scale_d=d)
    torch_cuda.cuda.synchronize()
    got = big.cpu().numpy()
    assert np.array_equal(got[:oh, :ow * c].reshape(oh, ow, c), oracle.upscale(img, ow, oh, a, n, d))
    assert (got[:oh, ow * c:] == 0xA5).all() and (got[oh:] == 0xA5).all()


def test_hls_mode_writes_only_its_output(lz, oracle):
    import torch
    img = noise_hwc(oracle, 50, 167, 3, seed=5)
    big = torch.full((100 + 3, 334 * 3 + 32), 0x5A, dtype=torch.uint8, device="cuda")
    d_out = big[:100].as_strided((100, 334, 3), (334 * 3 + 32, 3, 1))
    lz.upscale_hls_device(torch.from_numpy(img).cuda(), d_out)
    torch.cuda.synchronize()
    got = big.cpu().numpy()
    assert np.array_equal(got[:100, :334 * 3].reshape(100, 334, 3), oracle.hls_upscale(img, 2))
    assert (got[:100, 334 * 3:] == 0x5A).all() and (got[100:] == 0x5A).all()
