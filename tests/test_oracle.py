"""CPU tests of the oracle: pinned against the reference's compiled software path, the golden
fixtures generated from it, and the known-answer hashes of SURVEY.md Appendix A."""
import os

import numpy as np
import pytest

from util import golden_files, noise_hwc, planar

KATS = [  # (in_w, in_h, n, d, a) -> FNV-1a of the verbatim reference output (SURVEY.md Appendix A)
    ((96, 54, 2, 1, 3), 0xF8BAF542D95C747D),
    ((96, 54, 2, 1, 2), 0x1D39E6E9FEE0221C),
    ((96, 54, 3, 2, 3), 0x2C5585279E7698D9),
    ((100, 60, 17, 10, 3), 0xE8AFE818592C0EB3),
    ((960, 540, 2, 1, 3), 0x14F498CC6C5C39F3),
    ((960, 540, 2, 1, 2), 0x8D5F557661F63065),
]


@pytest.mark.parametrize("cfg,want", KATS)
def test_known_answer_hashes(oracle, cfg, want):
    w, h, n, d, a = cfg
    ow, oh = oracle.out_dims(w, h, n, d)
    img = oracle.xorshift_bytes(3 * w * h).reshape(3, h, w)
    out = oracle.expected_planar(img, ow, oh, a, n, d, fast=True)
    assert oracle.fnv1a64(out) == want
    if w < 200:  # the literal per-tap-sin restatement is slow: small cases only
        lit = oracle.expected_planar(img, ow, oh, a, n, d, fast=False)
        assert np.array_equal(lit, out)


@pytest.mark.parametrize("path", golden_files(), ids=os.path.basename)
def test_golden_fixtures(oracle, path):
    """Fixtures hold outputs of the reference's own lanczos_expected (tests/golden/make_golden.py)."""
    z = np.load(path)
    iw, ih, ow, oh, n, d, a, c = (int(v) for v in z["cfg"])
    out = oracle.expected_planar(z["img_in"], ow, oh, a, n, d, fast=True)
    assert np.array_equal(out, z["img_out"])
    lit = oracle.expected_planar(z["img_in"], ow, oh, a, n, d, fast=False)
    assert np.array_equal(lit, z["img_out"])


def test_against_compiled_reference(oracle):
    """Bit-equality with the compiled reference: with the hashes of its outputs that tests/golden/make_golden.py stored
    in tests/golden/ref_hashes.txt (input: xorshift seed SEED, planar), and with oracle/_ref itself on fresh seeds
    where those objects have been built from a reference tree (oracle/Makefile targets ref, refhls)."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_hashes.txt")) as fh:
        stored = [[int(v) for v in ln.split()[:8]] + [int(ln.split()[8], 16)] for ln in fh if not ln.startswith("#")]
    assert len(stored) == 3
    for iw, ih, ow, oh, n, d, a, c, want in stored:
        img = oracle.xorshift_bytes(c * ih * iw).reshape(c, ih, iw)
        assert oracle.fnv1a64(oracle.expected_planar(img, ow, oh, a, n, d)) == want, (iw, ih, ow, oh, n, d, a, c)
    for cfg in [c for c in oracle.ref_configs() if c[0] * c[1] <= 100 * 60]:
        iw, ih, ow, oh, n, d, a, c = cfg
        for seed in (11, 12):
            img = oracle.xorshift_bytes(c * ih * iw, oracle.SEED + seed).reshape(c, ih, iw)
            ref = oracle.ref_expected_planar(img, cfg)
            assert np.array_equal(oracle.expected_planar(img, ow, oh, a, n, d), ref), cfg


def test_kernel_values(oracle):
    L = oracle.lib().oracle_kernel
    assert L(0.0, 3) == 1.0
    # no |x|<a window and no exact zeros at integers (full_TB.h:51-53): sin(k*pi) residues survive
    assert 0 < abs(L(1.0, 3)) < 1e-16 and 0 < abs(L(2.0, 3)) < 1e-16
    assert abs(L(0.5, 3) - 0.6079271018540267) < 1e-15
    assert abs(L(1.5, 3) + 0.13509491152311703) < 1e-15
    assert abs(L(0.5, 2) - 0.5731591682507563) < 1e-15


def test_dc_gain_and_borders(oracle):
    """No renormalisation, zero borders (full_TB.h:59): a flat 255 field does not stay flat."""
    img = np.full((1, 20, 20), 255, np.uint8)
    out = oracle.expected_planar(img, 40, 40, 3, 2, 1, variant=oracle.CLEAN)
    assert out[0, 20, 20] == 255          # phase 0 both ways (clean: no aliasing)
    assert out[0, 20, 21] == 253          # phase 1/2 horizontally: floor(255*0.994299)
    assert out[0, 21, 21] == 251          # both: floor(253*0.994299)
    assert out[0, 0, 39] < 200            # right border: 3 of 6 taps dropped
    zero = oracle.expected_planar(np.zeros((2, 9, 7), np.uint8), 14, 18, 3, 2, 1)
    assert not zero.any()


def test_alias_only_touches_top_rows(oracle):
    """In-place column pass (full_TB.h:67-77) differs from ping-pong only in the first rows."""
    for (w, h, n, d, a, rows) in [(40, 30, 2, 1, 3, 5), (40, 30, 3, 2, 3, 7), (40, 30, 17, 10, 3, 5), (40, 30, 2, 1, 2, 3)]:
        ow, oh = oracle.out_dims(w, h, n, d)
        img = planar(noise_hwc(oracle, h, w, 3, seed=5))
        v = oracle.expected_planar(img, ow, oh, a, n, d, variant=oracle.VERBATIM)
        c = oracle.expected_planar(img, ow, oh, a, n, d, variant=oracle.CLEAN)
        assert np.array_equal(v[:, rows:], c[:, rows:])
        assert not np.array_equal(v[:, :rows], c[:, :rows])


def test_interleaved_front_end_and_bands(oracle):
    img = noise_hwc(oracle, 31, 45, 4, seed=3)
    ow, oh = oracle.out_dims(45, 31, 3, 2)
    full = oracle.upscale(img, ow, oh, 3, 3, 2)
    pl = oracle.expected_planar(planar(img), ow, oh, 3, 3, 2)
    assert np.array_equal(np.transpose(full, (2, 0, 1)), pl)
    band = oracle.upscale(img, ow, oh, 3, 3, 2, rows=(10, 17))
    assert np.array_equal(band, full[10:27])


def test_threads_do_not_change_results(oracle):
    img = planar(noise_hwc(oracle, 64, 80, 3, seed=9))
    a = oracle.expected_planar(img, 160, 128, 3, 2, 1, threads=1)
    b = oracle.expected_planar(img, 160, 128, 3, 2, 1, threads=0)
    assert np.array_equal(a, b)


def test_rejects_bad_arguments(oracle):
    img = np.zeros((3, 8, 8), np.uint8)
    with pytest.raises(ValueError):
        oracle.expected_planar(img, 16, 4, 3, 2, 1)   # out_h < in_h: H result would not fit (full_TB.h:85)
    with pytest.raises(ValueError):
        oracle.expected_planar(img, 16, 16, 0, 2, 1)
