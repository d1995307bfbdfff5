"""Shared plumbing for the tests that call the library: the torch_cuda fixture, the error codes of the C ABI, and the
two ways the GPU tests run an upscale -- a plain device call into a pre-filled output, and a raw C-ABI call on laid-out
buffers whose every byte outside the output must survive."""
import ctypes as C
import threading

import numpy as np
import pytest

NO_DEVICE = 1 << 20           # a device ordinal that exists nowhere
ERR_NULL, ERR_DIMS, ERR_TAPS, ERR_BAND, ERR_CUDA, ERR_ALIGN = -1, -2, -4, -7, -8, -10

CANARY = 0xA7                 # fills every output before a call
LEAD = 64                     # canary bytes before the output base of canary_call (plus out_off)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def in_thread(fn):
    """fn() on a thread of its own: the failed cudaSetDevice stays in that thread's CUDA error state."""
    out = []
    t = threading.Thread(target=lambda: out.append(fn()))
    t.start()
    t.join()
    return out[0]


def device_upscale(torch, lz, img, ow, oh, a, n, d, flags=0, stats=False):
    """[H][W][C] host image -> [oh][ow][C] host result through lz.upscale_device.  The output starts out as CANARY
    bytes, so a pixel the kernel leaves unwritten cannot pass by holding what an earlier call left in the same memory.
    stats: count strict samples during the call; lz.stats() reads the counters afterwards."""
    d_in = torch.from_numpy(img).cuda()
    d_out = torch.full((oh, ow, img.shape[2]), CANARY, dtype=torch.uint8, device="cuda")
    lz.enable_stats(stats)
    try:
        lz.upscale_device(d_in, d_out, a=a, scale_n=n, scale_d=d, flags=flags)
        torch.cuda.synchronize()
    finally:
        lz.enable_stats(False)
    return d_out.cpu().numpy()


def canary_layout(row_bytes, rows, frames, off, pad, gap):
    """(base, pitch, frame stride, buffer bytes) of `frames` frames of `rows` rows of `row_bytes` in a canary buffer:
    LEAD + off bytes before the base, `pad` bytes after every row, `gap` after every frame, two rows and 64 bytes after
    the last frame's gap."""
    pitch = row_bytes + pad
    fstride = pitch * rows + gap
    base = LEAD + off
    return base, pitch, fstride, base + fstride * frames + 2 * pitch + 64


def overwritten(host, base, frames, rows, row_bytes, pitch, fstride):
    """Offsets from `base` of the bytes of `host` outside the output rows that no longer hold CANARY: in the lead, the
    row padding, the frame gaps and the tail."""
    outside = np.ones(len(host), bool)
    np.lib.stride_tricks.as_strided(outside[base:], shape=(frames, rows, row_bytes), strides=(fstride, pitch, 1))[...] = False
    return np.nonzero(outside & (host != CANARY))[0] - base


def canary_call(torch, lz, desc, frames, entry, win=None, rect=None, in_off=0, in_pad=0, in_gap=0, out_off=0,
                out_pad=0, out_gap=0, seed=0, stats=False, bit_precision=8):
    """One call of lanczos_b200_<entry> (upscale, upscale_batch, upscale_region or upscale_hls, the last with
    `bit_precision`) on `frames` (list of [H][W][C] host images) with `desc` (its pitches are replaced), on device
    buffers laid out as asked.

    Input: the rect (ix, iy, w, h) of every frame (default the whole frame) at `in_off` bytes past a 256-byte
    boundary, rows padded by `in_pad` bytes, frames `in_gap` bytes apart; every other byte of the buffer is random
    (from `seed`).  Output: the window (x0, y0, w, h) (default the whole output), laid out by canary_layout in a buffer
    of CANARY bytes.  stats: count strict samples during the call.  Returns (outputs, lz.stats(), lz.launch()) after
    checking that the call succeeded and that every byte outside the output rows still holds CANARY."""
    ih, iw, c = frames[0].shape
    nf = len(frames)
    x0, y0, w, h = win or (0, 0, desc.out_w, desc.out_h)
    ix, iy, riw, rih = rect or (0, 0, iw, ih)
    in_pitch = riw * c + in_pad
    in_fs = in_pitch * rih + in_gap
    src = np.random.default_rng(seed).integers(0, 256, in_off + in_fs * nf + 256, dtype=np.uint8)
    for f, img in enumerate(frames):
        view = np.lib.stride_tricks.as_strided(src[in_off + f * in_fs:], shape=(rih, riw * c), strides=(in_pitch, 1))
        view[...] = img[iy:iy + rih, ix:ix + riw].reshape(rih, riw * c)
    rb = w * c
    base, out_pitch, out_fs, total = canary_layout(rb, h, nf, out_off, out_pad, out_gap)
    d_in = torch.from_numpy(src).cuda()
    buf = torch.full((total,), CANARY, dtype=torch.uint8, device="cuda")
    assert d_in.data_ptr() % 256 == 0 and buf.data_ptr() % 256 == 0
    d = lz.Desc.from_buffer_copy(desc)
    d.in_pitch, d.out_pitch = in_pitch, out_pitch
    p_in, p_out = C.c_void_p(d_in.data_ptr() + in_off), C.c_void_p(buf.data_ptr() + base)
    L = lz.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lz.enable_stats(stats)
    try:
        if entry == "upscale":
            assert nf == 1
            rc = L.lanczos_b200_upscale(C.byref(d), p_in, p_out, 0, stream)
        elif entry == "upscale_batch":
            rc = L.lanczos_b200_upscale_batch(C.byref(d), p_in, p_out, nf, in_fs, out_fs, 0, stream)
        elif entry == "upscale_hls":
            rc = L.lanczos_b200_upscale_hls(C.byref(d), p_in, p_out, bit_precision, nf, in_fs, out_fs, 0, stream)
        else:
            assert entry == "upscale_region", entry
            rc = L.lanczos_b200_upscale_region(C.byref(d), p_in, p_out, x0, y0, w, h, ix, iy, riw, rih, nf, in_fs,
                                               out_fs, 0, stream)
        torch.cuda.synchronize()
        st, ln = lz.stats(), lz.launch()
    finally:
        lz.enable_stats(False)
    assert rc == 0, (rc, L.lanczos_b200_strerror(rc), entry, win, rect)
    host = buf.cpu().numpy()
    view = np.lib.stride_tricks.as_strided(host[base:], shape=(nf, h, rb), strides=(out_fs, out_pitch, 1))
    outs = [np.array(view[f]).reshape(h, w, c) for f in range(nf)]
    hit = overwritten(host, base, nf, h, rb, out_pitch, out_fs)
    assert len(hit) == 0, ("canary bytes overwritten", entry, win, len(hit), hit[:8].tolist())
    return outs, st, ln
