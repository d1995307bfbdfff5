"""ctypes loader for the CPU oracle and the compiled reference (TEST INFRASTRUCTURE ONLY).

Only tests/, bench.py's cpu_baseline / --impl reference legs and
__graft_entry__.smoke() may import this module; the product package
(lanczos_hls_b200) never does.
"""
import ctypes as C
import glob
import os
import re
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
VERBATIM, CLEAN = 0, 1
SEED = 0x9E3779B97F4A7C15

_lib = None


def build():
    """Compile the oracle (and oracle/_ref when /root/reference is present)."""
    subprocess.run(["make", "-s", "-C", HERE], check=True)


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(HERE, "liblanczos_oracle.so")
        if not os.path.exists(path):
            build()
        L = C.CDLL(path)
        u8p = C.POINTER(C.c_uint8)
        L.oracle_expected_planar.argtypes = [u8p, u8p] + [C.c_int] * 9
        L.oracle_expected_planar_fast.argtypes = [u8p, u8p] + [C.c_int] * 10
        L.oracle_upscale_interleaved.argtypes = [u8p, C.c_int64, u8p, C.c_int64] + [C.c_int] * 10
        L.oracle_upscale_interleaved_rows.argtypes = [u8p, C.c_int64, u8p, C.c_int64] + [C.c_int] * 12
        L.oracle_kernel.argtypes = [C.c_double, C.c_int]
        L.oracle_kernel.restype = C.c_double
        L.oracle_fill_xorshift.argtypes = [u8p, C.c_int64, C.c_uint64]
        L.oracle_fill_xorshift.restype = None
        L.oracle_fnv1a64.argtypes = [u8p, C.c_int64]
        L.oracle_fnv1a64.restype = C.c_uint64
        L.oracle_hls_lut.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32)]
        L.oracle_hls_upscale.argtypes = [u8p, u8p] + [C.c_int] * 8
        i32p = C.POINTER(C.c_int32)
        L.oracle_hls_mac1.argtypes = [u8p, i32p, C.c_int, C.c_int]
        L.oracle_hls_mac1.restype = C.c_int32
        L.oracle_hls_mac2.argtypes = [i32p, i32p, C.c_int, C.c_int]
        L.oracle_hls_mac2.restype = C.c_int32
        L.oracle_hls_to_byte.argtypes = [C.c_int32, C.c_int]
        L.oracle_hls_to_byte.restype = C.c_uint8
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def xorshift_bytes(n, seed=SEED):
    out = np.empty(n, dtype=np.uint8)
    lib().oracle_fill_xorshift(_p(out), n, C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF))
    return out


def fnv1a64(a):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return int(lib().oracle_fnv1a64(_p(a), a.size))


def out_dims(in_w, in_h, n, d):
    """OUT = IN*N/D with integer division (SURVEY.md Appendix A)."""
    return in_w * n // d, in_h * n // d


def expected_planar(img, out_w, out_h, a, n, d, variant=VERBATIM, fast=True, threads=0):
    """img: uint8 [C][H][W] -> uint8 [C][out_h][out_w] (reference lanczos_expected layout)."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    c, h, w = img.shape
    out = np.empty((c, out_h, out_w), dtype=np.uint8)
    if fast:
        rc = lib().oracle_expected_planar_fast(_p(img), _p(out), c, w, h, out_w, out_h, a, n, d, variant, threads)
    else:
        rc = lib().oracle_expected_planar(_p(img), _p(out), c, w, h, out_w, out_h, a, n, d, variant)
    if rc != 0:
        raise ValueError(f"oracle rejected the arguments (rc={rc})")
    return out


def upscale(img, out_w, out_h, a, n, d, variant=VERBATIM, threads=0, rows=None):
    """img: uint8 [H][W][C] interleaved -> uint8 [out_h][out_w][C]; rows=(row0,count) returns a band."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w, c = img.shape
    row0, cnt = (0, out_h) if rows is None else rows
    out = np.empty((cnt, out_w, c), dtype=np.uint8)
    rc = lib().oracle_upscale_interleaved_rows(_p(img), w * c, _p(out), out_w * c, c, w, h, out_w, out_h,
                                               a, n, d, variant, threads, row0, cnt)
    if rc != 0:
        raise ValueError(f"oracle rejected the arguments (rc={rc})")
    return out


# ---- the compiled reference (oracle/_ref, one .so per compile-time config) ----

_REF_RE = re.compile(r"libref_(\d+)x(\d+)_(\d+)x(\d+)_(\d+)_(\d+)_a(\d+)_c(\d+)\.so$")


def ref_configs():
    """[(in_w,in_h,out_w,out_h,n,d,a,c)] for every prebuilt reference object."""
    out = []
    for p in sorted(glob.glob(os.path.join(HERE, "_ref", "libref_*.so"))):
        m = _REF_RE.search(p)
        if m:
            out.append(tuple(int(g) for g in m.groups()))
    return out


def ref_path(cfg):
    iw, ih, ow, oh, n, d, a, c = cfg
    return os.path.join(HERE, "_ref", f"libref_{iw}x{ih}_{ow}x{oh}_{n}_{d}_a{a}_c{c}.so")


_ref_libs = {}


def ref_lib(cfg):
    if cfg not in _ref_libs:
        L = C.CDLL(ref_path(cfg))
        L.ref_lanczos_expected.argtypes = [C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]
        got = (C.c_int * 8)()
        L.ref_config(got)
        assert tuple(got) == (cfg[0], cfg[1], cfg[2], cfg[3], cfg[4], cfg[5], cfg[6], cfg[7]), (tuple(got), cfg)
        _ref_libs[cfg] = L
    return _ref_libs[cfg]


def ref_expected_planar(img, cfg):
    """Run the reference's own lanczos_expected (full_TB.h:79-96) compiled for `cfg`."""
    iw, ih, ow, oh, n, d, a, c = cfg
    img = np.ascontiguousarray(img, dtype=np.uint8)
    assert img.shape == (c, ih, iw)
    out = np.empty((c, oh, ow), dtype=np.uint8)
    ref_lib(cfg).ref_lanczos_expected(_p(img), _p(out))
    return out


# ---- fixed-point HLS path (parity UNPINNED, see oracle/hls_oracle.c) ----

def hls_lut(a, n, bp=8):
    buf = (C.c_int32 * (a * n + 1))()
    if lib().oracle_hls_lut(a, n, bp, buf) != 0:
        raise ValueError("bad HLS LUT arguments")
    return np.array(buf[:], dtype=np.int32)


def hls_upscale(img, n, a=3, bp=8, out_w=None, out_h=None):
    """Fixed-point HLS path on an interleaved [H][W][C] image, integer scale n; the output is
    out_w x out_h (default w*n x h*n), also when that is not the input's size times n."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w, c = img.shape
    out_w = w * n if out_w is None else out_w
    out_h = h * n if out_h is None else out_h
    out = np.empty((out_h, out_w, c), dtype=np.uint8)
    if lib().oracle_hls_upscale(_p(img), _p(out), c, w, h, out_w, out_h, a, n, bp) != 0:
        raise ValueError("oracle rejected the HLS arguments")
    return out


def ref_hls_path(a, bp):
    return os.path.join(HERE, "_ref", "libref_hls_a%d_c3_bp%d.so" % (a, bp))


def ref_hls_lib(a, bp):
    """The reference's own compute / compute_ / clamp_to_byte (worker.cpp:10-130) compiled against oracle/ap_shim.h."""
    L = C.CDLL(ref_hls_path(a, bp))
    u8p, i32p = C.POINTER(C.c_uint8), C.POINTER(C.c_int32)
    L.ref_hls_compute.argtypes = [u8p, i32p, i32p]
    L.ref_hls_compute2.argtypes = [i32p, i32p, i32p]
    L.ref_hls_clamp_to_byte.argtypes = [i32p, u8p]
    L.ref_hls_config.argtypes = [i32p]
    return L
