"""CPU tests of the host logic and the C-ABI surface (no compute calls: there is no GPU here)."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(lz):
    hdr = open(os.path.join(ROOT, "include", "lanczos_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = sorted(set(re.findall(r"\b(lanczos_b200_\w+)\s*\(", hdr)))
    assert len(names) >= 25
    L = ctypes.CDLL(lz.lib_path())
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert lz.abi_version() == 1


def test_ratio_reduction_matches_reference_gcd(lz):
    # gcd.h via the preprocessor gives 3840/2560 -> 3/2, 3840/1920 -> 2/1, 486/162 -> 3/1, 1700/1000 -> 17/10
    assert lz.reduce_ratio(3840, 2560) == (3, 2)
    assert lz.reduce_ratio(3840, 1920) == (2, 1)
    assert lz.reduce_ratio(486, 162) == (3, 1)
    assert lz.reduce_ratio(1700, 1000) == (17, 10)
    r = lz.resolve(lz.make_desc(2560, 1440, 3840, 2160, 4, 3))
    assert (r.scale_n, r.scale_d, r.in_pitch, r.out_pitch) == (3, 2, 2560 * 4, 3840 * 4)
    r = lz.resolve(lz.make_desc(100, 60, 170, 102, 3, 3, 34, 20))
    assert (r.scale_n, r.scale_d) == (17, 10)


@pytest.mark.parametrize("kw,code", [
    (dict(in_w=0), -2), (dict(out_h=10, in_h=20), -2), (dict(channels=5), -3), (dict(channels=0), -3),
    (dict(a=0), -4), (dict(a=5), -4), (dict(scale_n=1, scale_d=2), -5), (dict(scale_n=-2, scale_d=1), -5),
    (dict(in_pitch=10), -2), (dict(out_pitch=3), -2),
])
def test_descriptor_validation(lz, kw, code):
    base = dict(in_w=16, in_h=16, out_w=32, out_h=32, channels=3, a=3)
    base.update(kw)
    with pytest.raises(lz.LanczosError) as e:
        lz.resolve(lz.make_desc(**base))
    assert e.value.code == code


def test_phase_table_matches_oracle_kernel(lz, oracle):
    sweep = [(n, d, a) for n in range(2, 17) for d in range(1, n) if math.gcd(n, d) == 1 for a in range(1, 5)]
    for (n, d, a) in [(2, 1, 3), (3, 2, 3), (17, 10, 3), (3, 1, 2), (4, 1, 3), (1, 1, 3), (65, 64, 4)] + sweep:
        t = lz.phase_table(lz.make_desc(d * 8, d * 8, n * 8, n * 8, 3, a, n, d))
        assert t.shape == (n, 2 * a)
        for xx in range(n):
            ph = (xx * d) % n
            x = xx / (n / d)
            first = xx * d // n - a + 1
            want = [oracle.lib().oracle_kernel(x - (first + k), a) for k in range(2 * a)]
            assert np.array_equal(t[ph], np.array(want, np.float64).astype(np.float32))
    t = lz.phase_table(lz.make_desc(8, 8, 16, 16, 3, 3))
    assert t[0, 2] == 1.0 and abs(t[0, 1]) < 1e-16          # phase 0: identity plus sin(k*pi) residues
    assert abs(t[1].sum() - 0.994299) < 1e-5                # no renormalisation (SURVEY.md 7)
    assert lz.lib().lanczos_b200_kernel(0.5, 3) == oracle.lib().oracle_kernel(0.5, 3)


def test_alias_rows(lz):
    # rows xx with floor(xx*D/N)+a > xx (SURVEY.md 7): 0-4 for 2x/a=3, 0-6 for 3/2, 0-4 for 17/10, 0-2 for 2x/a=2
    assert lz.alias_rows(lz.make_desc(1920, 1080, 3840, 2160, 3, 3)) == 5
    assert lz.alias_rows(lz.make_desc(2560, 1440, 3840, 2160, 4, 3)) == 7
    assert lz.alias_rows(lz.make_desc(1000, 1000, 1700, 1700, 3, 3)) == 5
    assert lz.alias_rows(lz.make_desc(960, 540, 1920, 1080, 3, 2)) == 3
    assert lz.alias_rows(lz.make_desc(960, 540, 1920, 1080, 3, 3, flags=lz.FLAG_NO_ALIAS)) == 0


def test_band_input_rows(lz):
    from lanczos_hls_b200.sharding import band_input_rows_py, band_range
    d = lz.make_desc(16384, 16384, 27852, 27852, 3, 3, 17, 10)
    k0 = lz.alias_rows(d)
    covered = 0
    for world in (1, 2, 4, 8):
        for rank in range(world):
            r0, r1 = band_range(27852, rank, world)
            lo, cnt = lz.band_input_rows(d, r0, r1 - r0)
            # SURVEY.md 8d: floor(r0*10/17)-2 .. floor((r1-1)*10/17)+3, clipped
            want_lo = max(0, r0 * 10 // 17 - 2) if r0 >= k0 else 0
            want_hi = min(16383, (r1 - 1) * 10 // 17 + 3)
            assert (lo, lo + cnt - 1) == (want_lo, want_hi)
            assert band_input_rows_py(r0, r1 - r0, 16384, 3, 17, 10, k0, 12)[0] == lo
            covered += (r1 - r0) if world == 8 else 0
    assert covered == 27852
    with pytest.raises(lz.LanczosError):
        lz.band_input_rows(d, 27000, 1000)


def test_inexact_ratio_is_detected_not_mishandled(lz):
    # any ratio for which floor((double)xx/SCALE) == floor(xx*D/N) everywhere must resolve fine
    for (n, d) in [(2, 1), (3, 2), (17, 10), (3, 1), (5, 3), (7, 4), (1, 1), (16, 9)]:
        assert lz.alias_rows(lz.make_desc(d * 50, d * 50, n * 50, n * 50, 3, 3, n, d)) >= 0


def test_compute_without_gpu_fails_loudly(lz):
    if lz.device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(lz.LanczosError) as e:
        lz.upscale(np.zeros((8, 8, 3), np.uint8), 16, 16)
    assert e.value.code == -8  # LANCZOS_ERR_CUDA: no CPU fallback
