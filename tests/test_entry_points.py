"""The C-ABI entry points: the order in which they check their arguments, and the counters of the host drivers.

Every entry point validates in its own order: some try the device before the descriptor, some after.  A caller sees
that order as the error code of a call that is wrong in two ways, so the CPU tests pin it, with a device ordinal that
exists nowhere (the answers are the same with and without a GPU).

The host drivers (lanczos_b200_upscale_host, _upscale_host_bands, _expected) run the device entry points' launch path
on their own scratch buffers.  The GPU tests pin what their counters report against the device calls that do the
same work.
"""
import ctypes as C

import numpy as np
import pytest

from harness import (ERR_ALIGN, ERR_CUDA, ERR_DIMS, ERR_NULL, ERR_TAPS, NO_DEVICE, device_upscale, in_thread,  # noqa: F401
                     torch_cuda)
from util import noise_hwc, planar


def entry_calls(lz, desc, null=False):
    """name -> a call of that entry point on `desc` and the device NO_DEVICE; `null` passes a null buffer instead."""
    L = lz.lib()
    img = np.zeros(1 << 16, np.uint8)
    buf = None if null else C.c_void_p(img.ctypes.data)
    host = C.c_void_p(img.ctypes.data)
    d = C.byref(desc)
    devs = (C.c_int32 * 1)(NO_DEVICE)
    return {
        "upscale_batch": lambda: L.lanczos_b200_upscale_batch(d, host, buf, 1, 0, 0, NO_DEVICE, None),
        "upscale_batch_negative": lambda: L.lanczos_b200_upscale_batch(d, host, buf, -1, 0, 0, NO_DEVICE, None),
        "upscale_planar": lambda: L.lanczos_b200_upscale_planar(d, host, buf, 1, 0, 0, NO_DEVICE, None),
        "upscale_band": lambda: L.lanczos_b200_upscale_band(d, host, buf, 0, 4, 0, 4, NO_DEVICE, None),
        "upscale_hls": lambda: L.lanczos_b200_upscale_hls(d, host, buf, 8, 1, 0, 0, NO_DEVICE, None),
        "upscale_host": lambda: L.lanczos_b200_upscale_host(d, host, buf, 1, 0, 0, NO_DEVICE, 3),
        "upscale_host_bands": lambda: L.lanczos_b200_upscale_host_bands(d, host, buf, devs, 1),
        "upscale_host_bands_none": lambda: L.lanczos_b200_upscale_host_bands(d, host, buf, devs, 0),
        "expected": lambda: L.lanczos_b200_expected(d, host, buf, NO_DEVICE),
        "stream": lambda: L.lanczos_b200_stream(d, host, buf, NO_DEVICE),
    }


# name: (code with a valid descriptor, code with a = 9)
CODES = {
    "upscale_batch": (ERR_CUDA, ERR_CUDA),
    "upscale_batch_negative": (ERR_DIMS, ERR_DIMS),
    "upscale_planar": (ERR_CUDA, ERR_CUDA),
    "upscale_band": (ERR_CUDA, ERR_CUDA),
    "upscale_hls": (ERR_CUDA, ERR_TAPS),
    "upscale_host": (ERR_CUDA, ERR_CUDA),
    "upscale_host_bands": (ERR_CUDA, ERR_TAPS),
    "upscale_host_bands_none": (ERR_DIMS, ERR_DIMS),
    "expected": (ERR_CUDA, ERR_TAPS),
    "stream": (ERR_CUDA, ERR_CUDA),
}


@pytest.mark.parametrize("name", sorted(CODES))
def test_error_order(lz, name):
    valid = lz.make_desc(16, 16, 32, 32, 3, 3, 2, 1)
    bad_a = lz.make_desc(16, 16, 32, 32, 3, 9, 2, 1)
    got = (in_thread(entry_calls(lz, valid)[name]), in_thread(entry_calls(lz, bad_a)[name]))
    assert got == CODES[name]
    assert in_thread(entry_calls(lz, bad_a, null=True)[name]) == ERR_NULL


def test_error_order_of_layout_checks(lz):
    L = lz.lib()
    img = np.zeros(1 << 16, np.uint8)
    p = C.c_void_p(img.ctypes.data)
    # the word stream takes three channels only, and says so before it looks for the device
    four = lz.make_desc(16, 16, 32, 32, 4, 3, 2, 1)
    assert in_thread(lambda: L.lanczos_b200_stream(C.byref(four), p, p, NO_DEVICE)) == ERR_ALIGN
    # n_frames * channels planes must fit a 32-bit count
    three = lz.make_desc(16, 16, 32, 32, 3, 3, 2, 1)
    big = (1 << 31) // 3 + 1
    assert in_thread(lambda: L.lanczos_b200_upscale_planar(C.byref(three), p, p, big, 0, 0, NO_DEVICE, None)) == ERR_DIMS
    assert in_thread(lambda: L.lanczos_b200_upscale_planar(C.byref(three), p, p, big - 1, 0, 0, NO_DEVICE, None)) == ERR_CUDA


# ---- GPU: counters of the host drivers ------------------------------------------------------------------------

# (in_w, in_h, out_w, out_h, channels, a, N, D, flags).  Rows of whole 16-byte words and widths the host drivers do not
# widen: their scratch images have the caller's dense pitches, so the device calls below see the same descriptor.
HOST_CASES = {
    "2_1_c3": (64, 160, 128, 320, 3, 3, 2, 1, 0),
    "3_2_c4": (64, 128, 96, 192, 4, 3, 3, 2, 0),
    "17_10_c3": (160, 100, 272, 170, 3, 3, 17, 10, 0),
    "2_1_c3_generic": (64, 160, 128, 320, 3, 3, 2, 1, 1 << 2),
    "2_1_c1_a2_no_alias": (64, 160, 128, 320, 1, 2, 2, 1, 1 << 0),
}


def band_call(torch, lz, desc, img, r0, rows):
    """Output rows [r0, r0 + rows) of img through lanczos_b200_upscale_band: (rows, stats, launch)."""
    in0, inn = lz.band_input_rows(desc, r0, rows)
    d_in = torch.from_numpy(np.ascontiguousarray(img[in0:in0 + inn])).cuda()
    d_out = torch.empty((rows, desc.out_w, desc.channels), dtype=torch.uint8, device="cuda")
    lz.upscale_band_device(desc, d_in, d_out, r0, rows, in0, inn)
    torch.cuda.synchronize()
    return d_out.cpu().numpy(), lz.stats(), lz.launch()


def frame_call(torch, lz, case, img):
    iw, ih, ow, oh, c, a, n, d, flags = case
    return device_upscale(torch, lz, img, ow, oh, a, n, d, flags), lz.stats(), lz.launch()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(HOST_CASES))
@pytest.mark.parametrize("n_streams", [2, 3])
def test_upscale_host_counts_its_device_calls(torch_cuda, lz, oracle, name, n_streams):
    torch = torch_cuda
    iw, ih, ow, oh, c, a, n, d, flags = case = HOST_CASES[name]
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, flags=flags)

    # whole frames: one device call per frame
    frames = np.stack([noise_hwc(oracle, ih, iw, c, seed=f) for f in range(2 * n_streams)])
    want, launches = [], 0
    for img in frames:
        out, st, last_launch = frame_call(torch, lz, case, img)
        want.append(out)
        launches += st["kernel_launches"]
    kid = st["kernel_id"]
    got = lz.upscale(frames, ow, oh, a, n, d, flags, n_streams=n_streams)
    st = lz.stats()
    assert np.array_equal(got, np.stack(want))
    assert (st["kernel_id"], st["kernel_launches"]) == (kid, launches), st
    assert lz.launch() == last_launch

    # one frame: row bands at out_h * b / bands
    img = frames[0]
    bands = max(1, min(oh // 64, 2 * n_streams))
    edges = [oh * b // bands for b in range(bands + 1)]
    launches = 0
    for r0, r1 in zip(edges, edges[1:]):
        out, st, last_launch = band_call(torch, lz, desc, img, r0, r1 - r0)
        assert np.array_equal(out, want[0][r0:r1])
        launches += st["kernel_launches"]
    kid = st["kernel_id"]
    got = lz.upscale(img, ow, oh, a, n, d, flags, n_streams=n_streams)
    st = lz.stats()
    assert np.array_equal(got, want[0])
    assert (st["kernel_id"], st["kernel_launches"]) == (kid, launches), st
    assert lz.launch() == last_launch


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(HOST_CASES))
def test_upscale_host_bands_counts_launches_only(torch_cuda, lz, oracle, name):
    """Two bands on device 0.  The driver sums the bands' launches into otherwise cleared stats (kernel_id reads 0)
    and leaves the calling thread's launch shape as it was."""
    torch = torch_cuda
    iw, ih, ow, oh, c, a, n, d, flags = case = HOST_CASES[name]
    desc = lz.make_desc(iw, ih, ow, oh, c, a, n, d, flags=flags)
    img = noise_hwc(oracle, ih, iw, c, seed=3)
    want, _, _ = frame_call(torch, lz, case, img)
    launches = 0
    for r0, r1 in ((0, oh // 2), (oh // 2, oh)):
        launches += band_call(torch, lz, desc, img, r0, r1 - r0)[1]["kernel_launches"]
    before = lz.launch()
    got = lz.upscale_bands_multi_gpu(img, ow, oh, [0, 0], a, n, d, flags)
    st = lz.stats()
    assert np.array_equal(got, want)
    assert (st["kernel_id"], st["kernel_launches"], st["alias_rows"]) == (0, launches, 0), st
    assert lz.launch() == before


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(HOST_CASES))
def test_expected_counts_one_planar_call(torch_cuda, lz, oracle, name):
    torch = torch_cuda
    iw, ih, ow, oh, c, a, n, d, flags = HOST_CASES[name]
    img = planar(noise_hwc(oracle, ih, iw, c, seed=5))
    d_out = torch.empty((c, oh, ow), dtype=torch.uint8, device="cuda")
    lz.upscale_planar_device(torch.from_numpy(img).cuda(), d_out, a, n, d, flags)
    torch.cuda.synchronize()
    want, want_stats, want_launch = d_out.cpu().numpy(), lz.stats(), lz.launch()
    got = lz.lanczos_expected(img, ow, oh, a, n, d, flags)
    assert np.array_equal(got, want)
    assert lz.stats() == want_stats
    assert lz.launch() == want_launch
