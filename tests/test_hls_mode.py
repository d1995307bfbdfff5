"""Fixed-point "HLS mode" (SURVEY.md 8f-1): the integer arithmetic of the reference's lanczos()
(worker.cpp:45-130, kernel.cpp:40-67).  Parity with the reference itself is UNPINNED (its LUT needs
Xilinx hls::sinpi, absent here); the CUDA path is checked bit for bit against oracle/hls_oracle.c."""
import numpy as np
import pytest

from harness import CANARY
from util import noise_hwc, smooth_hwc


def test_lut_restatement(oracle, lz):
    # SURVEY.md 8c: 2x, BP=8: a=2 -> [256,146,0,-17,0], a=3 -> [256,155,0,-35,-1,6,0]
    assert oracle.hls_lut(2, 2).tolist() == [256, 146, 0, -17, 0]
    assert oracle.hls_lut(3, 2).tolist() == [256, 155, 0, -35, -1, 6, 0]
    for (a, n, bp) in [(2, 2, 8), (3, 2, 8), (3, 4, 8), (2, 3, 10), (3, 2, 6)]:
        assert np.array_equal(lz.hls_lut(a, n, bp), oracle.hls_lut(a, n, bp))
    with pytest.raises(lz.LanczosError):
        lz.hls_lut(3, 64)        # kernel_t(i) wraps for i >= 128 (kernel.cpp:42)


def test_oracle_dering_and_borders(oracle):
    img = noise_hwc(oracle, 24, 32, 3, seed=1)
    out = oracle.hls_upscale(img, 2)
    # phase-0 samples nearly reproduce the input: LUT[0] = 1.0, LUT[2N] = floor(-1.6e-17 * 256) = -1/256 (the
    # unpinned sin(2*pi) residue) pulls the sum below v, and both passes floor -> a few LSB low at most
    d0 = img.astype(int) - out[::2, ::2].astype(int)
    assert d0.min() >= 0 and d0.max() <= 4
    # de-ring clamp (worker.cpp:66-74): every output lies between its two central taps along x
    mid = out[:, 1:-1:2].astype(int)
    lo = np.minimum(out[:, 0:-2:2], out[:, 2::2]).astype(int)
    hi = np.maximum(out[:, 0:-2:2], out[:, 2::2]).astype(int)
    assert ((mid >= lo - 3) & (mid <= hi + 3)).all()   # neighbours are themselves up to 4 LSB low (see above)
    flat = oracle.hls_upscale(np.full((12, 12, 3), 200, np.uint8), 2)
    assert (flat[6:-2, 6:-2] == 200).all()           # the clamp pins flat regions (unlike the software path)
    assert (flat[-6:, -6:] == 200).all()             # bottom/right: last row/column replicated
    assert flat[0, 6, 0] == 200                      # top: zero rows enter the window, but the clamp to the central taps pins it


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [(96, 54, 2, 3, 3, 8), (50, 40, 2, 2, 4, 8), (33, 47, 3, 2, 1, 8),
                                 (64, 64, 4, 3, 3, 8), (70, 30, 2, 3, 3, 10), (131, 77, 2, 3, 3, 6),
                                 # the tiled kernel: several tiles, ragged right / bottom edges, every instance
                                 (400, 130, 2, 3, 3, 8), (167, 29, 2, 3, 4, 8), (517, 40, 2, 3, 1, 8), (90, 77, 2, 2, 3, 8),
                                 (83, 50, 4, 2, 3, 8), (161, 13, 2, 3, 3, 8), (7, 5, 2, 3, 3, 8)],
                         ids=lambda c: "x".join(map(str, c)))
def test_gpu_matches_integer_restatement(lz, oracle, cfg):
    import torch
    w, h, n, a, c, bp = cfg
    for maker in (noise_hwc, smooth_hwc):
        img = maker(oracle, h, w, c, seed=w)
        want = oracle.hls_upscale(img, n, a, bp)
        d_in = torch.from_numpy(img).cuda()
        d_out = torch.full((h * n, w * n, c), CANARY, dtype=torch.uint8, device="cuda")
        lz.upscale_hls_device(d_in, d_out, a=a, bit_precision=bp)
        torch.cuda.synchronize()
        assert np.array_equal(d_out.cpu().numpy(), want)
    tiled = bp == 8 and (c, a, n) in {(3, 3, 2), (4, 3, 2), (1, 3, 2), (3, 2, 2), (3, 3, 4), (3, 2, 4)}
    assert lz.stats()["kernel_id"] == (101 if tiled else 100)


@pytest.mark.gpu
def test_gpu_hls_batch_and_errors(lz, oracle):
    import torch
    frames = np.stack([noise_hwc(oracle, 20, 28, 3, seed=s) for s in range(3)])
    d_in = torch.from_numpy(frames).cuda()
    d_out = torch.full((3, 40, 56, 3), CANARY, dtype=torch.uint8, device="cuda")
    lz.upscale_hls_device(d_in, d_out)
    torch.cuda.synchronize()
    for i in range(3):
        assert np.array_equal(d_out[i].cpu().numpy(), oracle.hls_upscale(frames[i], 2))
    bad = torch.zeros((30, 42, 3), dtype=torch.uint8, device="cuda")     # 3/2 is not an integer scale
    with pytest.raises(lz.LanczosError) as e:
        lz.upscale_hls_device(d_in[0], bad)
    assert e.value.code == -5


@pytest.mark.parametrize("cfg", [(3, 8), (2, 8), (3, 6), (3, 10)], ids=lambda c: "a%d_bp%d" % c)
def test_sample_arithmetic_against_compiled_reference(oracle, cfg):
    """The pin of the fixed-point path: oracle/hls_oracle.c's per-sample arithmetic against the reference's OWN
    compute / compute_ / clamp_to_byte (worker.cpp:45-130), compiled as they are against the integer-backed
    ap_fixed / ap_uint stand-ins of oracle/ap_shim.h (oracle/Makefile target refhls).  Windows: random bytes, flat
    runs, extremes; kernels: every phase of the LUT for 2x..5x, and random kernel_t values small enough that the
    10 integer bits of num_el_t cannot wrap, plus a few that do (AP_WRAP is part of the restatement)."""
    import ctypes as C
    import os
    a, bp = cfg
    if not os.path.exists(oracle.ref_hls_path(a, bp)):
        pytest.skip("oracle/_ref/libref_hls_* not built (no reference tree)")
    R = oracle.ref_hls_lib(a, bp)
    L = oracle.lib()
    got = (C.c_int32 * 3)()
    R.ref_hls_config(got)
    assert list(got) == [3, a, bp]
    rng = np.random.default_rng(a * 100 + bp)
    taps = 2 * a
    kernels = []
    for n in (2, 3, 4, 5):
        lut = oracle.hls_lut(a, n, bp)
        for ph in range(n):                      # output x = base*n + ph: weights LUT[|ph - (j - a + 1) * n|]
            kernels.append(np.array([lut[abs(ph - (j - a + 1) * n)] for j in range(taps)], np.int32))
    for _ in range(40):
        kernels.append(rng.integers(-(1 << bp) // 3, (1 << bp) // 3, size=taps).astype(np.int32))
    for _ in range(10):
        kernels.append(rng.integers(-(1 << (bp + 2)), 1 << (bp + 2), size=taps).astype(np.int32))   # wraps
    i32p, u8p = C.POINTER(C.c_int32), C.POINTER(C.c_uint8)
    n_cases = 0
    for k in kernels:
        kp = k.ctypes.data_as(i32p)
        for trial in range(60):
            win = rng.integers(0, 256, size=(taps, 3)).astype(np.uint8)
            if trial % 6 == 1:
                win[:] = rng.integers(0, 256)
            elif trial % 6 == 2:
                win[:] = rng.choice([0, 255], size=(taps, 3))
            out = np.zeros(3, np.int32)
            R.ref_hls_compute(win.ctypes.data_as(u8p), kp, out.ctypes.data_as(i32p))
            mine = [L.oracle_hls_mac1(np.ascontiguousarray(win[:, c]).ctypes.data_as(u8p), kp, a, bp) for c in range(3)]
            assert out.tolist() == mine, (k.tolist(), win.tolist())
            # second pass: fixed-point intermediates as the first pass produces them (>= 0, < 256), and raw extremes
            mid = rng.integers(0, 256 << bp, size=(taps, 3)).astype(np.int32)
            if trial % 6 == 3:
                mid[:] = rng.integers(0, 256 << bp)
            out2 = np.zeros(3, np.int32)
            R.ref_hls_compute2(mid.ctypes.data_as(i32p), kp, out2.ctypes.data_as(i32p))
            mine2 = [L.oracle_hls_mac2(np.ascontiguousarray(mid[:, c]).ctypes.data_as(i32p), kp, a, bp) for c in range(3)]
            assert out2.tolist() == mine2, (k.tolist(), mid.tolist())
            b = np.zeros(3, np.uint8)
            R.ref_hls_clamp_to_byte(out2.ctypes.data_as(i32p), b.ctypes.data_as(u8p))
            assert b.tolist() == [L.oracle_hls_to_byte(int(v), bp) for v in out2]
            n_cases += 3
    # clamp_to_byte on its whole domain, negative values included
    for raw in list(range(-(512 << bp), 512 << bp, 37)) + [-1, 0, 1, (256 << bp) - 1, 256 << bp]:
        v = np.array([raw, raw, raw], np.int32)
        b = np.zeros(3, np.uint8)
        R.ref_hls_clamp_to_byte(v.ctypes.data_as(i32p), b.ctypes.data_as(u8p))
        assert b[0] == L.oracle_hls_to_byte(raw, bp), raw
    assert n_cases > 10000
