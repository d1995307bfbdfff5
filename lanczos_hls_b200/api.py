"""ctypes binding of include/lanczos_b200.h and the reference-shaped host API.

Reference interface mirrored here (file:line in the reference tree):
  lanczos_expected(byte in[C][IN_H][IN_W], byte out[C][OUT_H][OUT_W])  full_TB.h:79-82
  lanczos(stream_t in, stream_t out) on packed 24-bit words               lanczos.h:121-126
  params.h macros IN_WIDTH.. LANCZOS_A, SCALE_N, SCALE_D                  lanczos.h:9-31,47-48
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

FLAG_NO_ALIAS = 1 << 0
FLAG_FAST_ALIGNED = 1 << 1
FLAG_TOLERANCE_1LSB = 1 << 3
FLAG_INDEPENDENT = 1 << 4
FLAG_GENERIC_KERNEL = 1 << 2


class LanczosError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"lanczos_b200 error {code}: {msg}")
        self.code = code


class Desc(C.Structure):
    """lanczos_desc (include/lanczos_b200.h): runtime form of the reference's params.h macros."""
    _fields_ = [
        ("in_w", C.c_int32), ("in_h", C.c_int32), ("out_w", C.c_int32), ("out_h", C.c_int32),
        ("channels", C.c_int32), ("a", C.c_int32), ("scale_n", C.c_int32), ("scale_d", C.c_int32),
        ("in_pitch", C.c_int64), ("out_pitch", C.c_int64), ("flags", C.c_uint32), ("reserved", C.c_uint32),
    ]

    def key(self):
        return tuple(getattr(self, f) for f, _ in self._fields_)


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("strict_samples", C.c_int64),
                ("kernel_id", C.c_int32), ("alias_rows", C.c_int32)]


class Launch(C.Structure):
    """lanczos_launch (include/lanczos_b200.h)."""
    _fields_ = [("grid_x", C.c_int32), ("grid_y", C.c_int32), ("grid_z", C.c_int32), ("seg_periods", C.c_int32),
                ("chunk_rows", C.c_int32), ("main_launches", C.c_int32), ("resident_ctas", C.c_int64)]


_lib = None


def lib_path():
    return os.path.join(HERE, "liblanczos_b200.so")


def lib():
    """Load liblanczos_b200.so. Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise LanczosError(-100, f"{path} is missing: build it with `python -m lanczos_hls_b200.build` "
                                 "(there is no CPU fallback)")
    L = C.CDLL(path)
    u8p, vp, dp = C.c_void_p, C.c_void_p, C.POINTER(Desc)
    i32, i64 = C.c_int32, C.c_int64
    L.lanczos_b200_upscale.argtypes = [dp, u8p, u8p, C.c_int, vp]
    L.lanczos_b200_upscale_batch.argtypes = [dp, u8p, u8p, i32, i64, i64, C.c_int, vp]
    L.lanczos_b200_upscale_planar.argtypes = [dp, u8p, u8p, i32, i64, i64, C.c_int, vp]
    L.lanczos_b200_upscale_band.argtypes = [dp, u8p, u8p, i32, i32, i32, i32, C.c_int, vp]
    L.lanczos_b200_band_input_rows.argtypes = [dp, i32, i32, C.POINTER(i32), C.POINTER(i32)]
    L.lanczos_b200_region_input_rect.argtypes = [dp, i32, i32, i32, i32] + [C.POINTER(i32)] * 4
    L.lanczos_b200_upscale_region.argtypes = [dp, u8p, u8p] + [i32] * 9 + [i64, i64, C.c_int, vp]
    L.lanczos_b200_upscale_host_region.argtypes = [dp, u8p, u8p, i32, i32, i32, i32, i64, C.c_int]
    L.lanczos_b200_upscale_host.argtypes = [dp, u8p, u8p, i32, i64, i64, C.c_int, i32]
    L.lanczos_b200_upscale_host_bands.argtypes = [dp, u8p, u8p, C.POINTER(i32), i32]
    L.lanczos_b200_expected.argtypes = [dp, u8p, u8p, C.c_int]
    L.lanczos_b200_stream.argtypes = [dp, vp, vp, C.c_int]
    L.lanczos_b200_upscale_hls.argtypes = [dp, u8p, u8p, i32, i32, i64, i64, C.c_int, vp]
    L.lanczos_b200_hls_lut.argtypes = [i32, i32, i32, C.POINTER(i32), i32]
    L.lanczos_b200_reduce_ratio.argtypes = [i32, i32, C.POINTER(i32), C.POINTER(i32)]
    L.lanczos_b200_resolve.argtypes = [dp, dp]
    L.lanczos_b200_kernel.argtypes = [C.c_double, i32]
    L.lanczos_b200_kernel.restype = C.c_double
    L.lanczos_b200_phase_table.argtypes = [dp, C.POINTER(C.c_float), i32]
    L.lanczos_b200_phase0_chain.argtypes = [dp, C.POINTER(C.c_float)]
    L.lanczos_b200_alias_rows.argtypes = [dp]
    L.lanczos_b200_host_alloc.argtypes = [C.c_size_t]
    L.lanczos_b200_host_alloc.restype = C.c_void_p
    L.lanczos_b200_host_free.argtypes = [C.c_void_p]
    L.lanczos_b200_host_free.restype = None
    L.lanczos_b200_device_alloc.argtypes = [C.c_int, C.c_size_t]
    L.lanczos_b200_device_alloc.restype = C.c_void_p
    L.lanczos_b200_device_free.argtypes = [C.c_int, C.c_void_p]
    L.lanczos_b200_device_free.restype = None
    L.lanczos_b200_memcpy_h2d.argtypes = [C.c_int, vp, vp, C.c_size_t]
    L.lanczos_b200_memcpy_d2h.argtypes = [C.c_int, vp, vp, C.c_size_t]
    L.lanczos_b200_synchronize.argtypes = [C.c_int]
    L.lanczos_b200_enable_stats.argtypes = [C.c_int]
    L.lanczos_b200_enable_stats.restype = None
    L.lanczos_b200_get_stats.argtypes = [C.POINTER(Stats)]
    L.lanczos_b200_get_launch.argtypes = [C.POINTER(Launch)]
    L.lanczos_b200_strerror.argtypes = [C.c_int]
    L.lanczos_b200_strerror.restype = C.c_char_p
    L.lanczos_b200_last_cuda_error.restype = C.c_char_p
    L.lanczos_b200_clear_plans.restype = None
    _lib = L
    return L


def _check(rc):
    if rc < 0:
        L = lib()
        msg = L.lanczos_b200_strerror(rc).decode()
        if rc == -8:
            msg += " (" + L.lanczos_b200_last_cuda_error().decode() + ")"
        raise LanczosError(rc, msg)
    return rc


def abi_version():
    return lib().lanczos_b200_abi_version()


def device_count():
    return lib().lanczos_b200_device_count()


def make_desc(in_w, in_h, out_w, out_h, channels=3, a=3, scale_n=0, scale_d=0, in_pitch=0, out_pitch=0, flags=0):
    return Desc(in_w, in_h, out_w, out_h, channels, a, scale_n, scale_d, in_pitch, out_pitch, flags, 0)


def resolve(desc):
    out = Desc()
    _check(lib().lanczos_b200_resolve(C.byref(desc), C.byref(out)))
    return out


def reduce_ratio(out_len, in_len):
    n, d = C.c_int32(), C.c_int32()
    _check(lib().lanczos_b200_reduce_ratio(out_len, in_len, C.byref(n), C.byref(d)))
    return n.value, d.value


def phase_table(desc):
    """float32 [N][2a] polyphase weights (row p = phase p)."""
    r = resolve(desc)
    buf = np.zeros((r.scale_n, 2 * r.a), dtype=np.float32)
    _check(lib().lanczos_b200_phase_table(C.byref(desc), buf.ctypes.data_as(C.POINTER(C.c_float)), buf.size))
    return buf


def alias_rows(desc):
    return _check(lib().lanczos_b200_alias_rows(C.byref(desc)))


def band_input_rows(desc, out_row0, out_rows):
    a, b = C.c_int32(), C.c_int32()
    _check(lib().lanczos_b200_band_input_rows(C.byref(desc), out_row0, out_rows, C.byref(a), C.byref(b)))
    return a.value, b.value


def region_input_rect(desc, x0, y0, w, h):
    """(in_x0, in_y0, in_w, in_h): the input pixels the output window [x0, x0+w) x [y0, y0+h) reads."""
    r = [C.c_int32() for _ in range(4)]
    _check(lib().lanczos_b200_region_input_rect(C.byref(desc), x0, y0, w, h, *[C.byref(v) for v in r]))
    return tuple(v.value for v in r)


def enable_stats(on=True):
    lib().lanczos_b200_enable_stats(1 if on else 0)


def stats():
    s = Stats()
    lib().lanczos_b200_get_stats(C.byref(s))
    return {"kernel_launches": s.kernel_launches, "strict_samples": s.strict_samples,
            "kernel_id": s.kernel_id, "alias_rows": s.alias_rows}


def launch():
    """Shape of the first main-kernel launch of the last call on this thread, and the number of main launches."""
    s = Launch()
    _check(lib().lanczos_b200_get_launch(C.byref(s)))
    return {f: getattr(s, f) for f, _ in Launch._fields_}


class PinnedBuffer:
    """Page-locked host memory exposed as a numpy uint8 array (for full-speed PCIe copies)."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        self.ptr = lib().lanczos_b200_host_alloc(self.nbytes)
        if not self.ptr:
            raise LanczosError(-9, "cudaMallocHost failed")
        self.array = np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self.ptr))

    def free(self):
        if self.ptr:
            self.array = None
            lib().lanczos_b200_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _np_ptr(a):
    return C.c_void_p(a.ctypes.data)


# ---- host arrays in, host arrays out ---------------------------------------------------------

def lanczos_expected(img_in, out_w, out_h, a=3, scale_n=0, scale_d=0, flags=0, device=0):
    """Same layout as the reference's lanczos_expected: uint8 [C][IN_H][IN_W] -> [C][OUT_H][OUT_W]."""
    img_in = np.ascontiguousarray(img_in, dtype=np.uint8)
    c, h, w = img_in.shape
    desc = make_desc(w, h, out_w, out_h, c, a, scale_n, scale_d, flags=flags)
    out = np.empty((c, out_h, out_w), dtype=np.uint8)
    _check(lib().lanczos_b200_expected(C.byref(desc), _np_ptr(img_in), _np_ptr(out), device))
    return out


def upscale(img, out_w, out_h, a=3, scale_n=0, scale_d=0, flags=0, device=0, n_streams=3, out=None):
    """uint8 [H][W][C] or [F][H][W][C] interleaved host array(s) -> upscaled host array(s)."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    batched = img.ndim == 4
    f = img.shape[0] if batched else 1
    h, w, c = img.shape[-3:]
    desc = make_desc(w, h, out_w, out_h, c, a, scale_n, scale_d, flags=flags)
    if out is None:
        out = np.empty(((f,) if batched else ()) + (out_h, out_w, c), dtype=np.uint8)
    _check(lib().lanczos_b200_upscale_host(C.byref(desc), _np_ptr(img), _np_ptr(out), f, 0, 0, device, n_streams))
    return out


def phase0_chain(desc):
    """(verified, [W0, W1, 1, W3, W4]) of the plan's exact fp32 phase-0 chain (a = 3), see include/lanczos_b200.h."""
    buf = (C.c_float * 5)()
    rc = lib().lanczos_b200_phase0_chain(C.byref(desc), buf)
    if rc < 0:
        _check(rc)
    return bool(rc), [float(v) for v in buf]


def bind_host_to_device(device=0):
    """Pin the calling process to the CPUs next to GPU `device` (NVML CPU affinity), so that pinned host
    buffers allocated afterwards are NUMA-local to the GPU's PCIe root.  With one process per GPU this keeps
    the host-buffer path (lanczos_b200_upscale_host) from crossing the socket interconnect.  Returns the CPU
    list, or None when NVML or the affinity call is unavailable (nothing is changed then)."""
    import os
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(device)
        bus = "%08x:%02x:%02x.0" % (getattr(props, "pci_domain_id", 0), props.pci_bus_id, props.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode() if hasattr(bus, "encode") else bus)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return allowed
    except Exception:
        return None


def upscale_bands_multi_gpu(img, out_w, out_h, devices, a=3, scale_n=0, scale_d=0, flags=0):
    """One large [H][W][C] host image split into row bands over `devices` (single process)."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    h, w, c = img.shape
    desc = make_desc(w, h, out_w, out_h, c, a, scale_n, scale_d, flags=flags)
    out = np.empty((out_h, out_w, c), dtype=np.uint8)
    devs = (C.c_int32 * len(devices))(*devices)
    _check(lib().lanczos_b200_upscale_host_bands(C.byref(desc), _np_ptr(img), _np_ptr(out), devs, len(devices)))
    return out


def lanczos_stream(words_in, in_w, in_h, out_w, out_h, a=3, scale_n=0, scale_d=0, flags=0, device=0):
    """Packed 24-bit RGB words in raster order, like the HLS top function's AXI streams."""
    words_in = np.ascontiguousarray(words_in, dtype=np.uint32).reshape(-1)
    assert words_in.size == in_w * in_h
    desc = make_desc(in_w, in_h, out_w, out_h, 3, a, scale_n, scale_d, flags=flags)
    out = np.empty(out_w * out_h, dtype=np.uint32)
    _check(lib().lanczos_b200_stream(C.byref(desc), _np_ptr(words_in), _np_ptr(out), device))
    return out


# ---- device tensors (torch is plumbing only: memory + streams) ------------------------------

def _stream_ptr(t):
    import torch
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def upscale_device(d_in, d_out, a=3, scale_n=0, scale_d=0, flags=0):
    """torch uint8 CUDA tensors [H][W][C] -> [OH][OW][C], asynchronous on the current stream."""
    h, w, c = d_in.shape
    oh, ow, _ = d_out.shape
    desc = make_desc(w, h, ow, oh, c, a, scale_n, scale_d, d_in.stride(0), d_out.stride(0), flags)
    _check(lib().lanczos_b200_upscale(C.byref(desc), C.c_void_p(d_in.data_ptr()), C.c_void_p(d_out.data_ptr()),
                                      d_in.device.index or 0, _stream_ptr(d_in)))
    return d_out


def upscale_batch_device(d_in, d_out, a=3, scale_n=0, scale_d=0, flags=0):
    """torch uint8 CUDA tensors [F][H][W][C] -> [F][OH][OW][C], one launch for the batch."""
    f, h, w, c = d_in.shape
    _, oh, ow, _ = d_out.shape
    desc = make_desc(w, h, ow, oh, c, a, scale_n, scale_d, d_in.stride(1), d_out.stride(1), flags)
    _check(lib().lanczos_b200_upscale_batch(C.byref(desc), C.c_void_p(d_in.data_ptr()), C.c_void_p(d_out.data_ptr()),
                                            f, d_in.stride(0), d_out.stride(0), d_in.device.index or 0,
                                            _stream_ptr(d_in)))
    return d_out


def upscale_planar_device(d_in, d_out, a=3, scale_n=0, scale_d=0, flags=0):
    """torch uint8 CUDA tensors [C][H][W] -> [C][OH][OW] or [F][C][H][W] -> [F][C][OH][OW]: the layout of the
    reference's lanczos_expected arguments (full_TB.h:20-21), every plane resampled on its own."""
    if d_in.dim() == 3:
        d_in, d_out = d_in.unsqueeze(0), d_out.unsqueeze(0)
    f, c, h, w = d_in.shape
    _, _, oh, ow = d_out.shape
    assert d_in.stride(0) == c * d_in.stride(1) and d_out.stride(0) == c * d_out.stride(1), "planes must be equally spaced"
    desc = make_desc(w, h, ow, oh, c, a, scale_n, scale_d, d_in.stride(2), d_out.stride(2), flags)
    _check(lib().lanczos_b200_upscale_planar(C.byref(desc), C.c_void_p(d_in.data_ptr()), C.c_void_p(d_out.data_ptr()),
                                             f, d_in.stride(1), d_out.stride(1), d_in.device.index or 0,
                                             _stream_ptr(d_in)))
    return d_out


def upscale_band_device(desc, d_in_band, d_out_band, out_row0, out_rows, in_row0, in_rows):
    """Row band of the image described by `desc`; tensors hold only the band's rows."""
    _check(lib().lanczos_b200_upscale_band(C.byref(desc), C.c_void_p(d_in_band.data_ptr()),
                                           C.c_void_p(d_out_band.data_ptr()), out_row0, out_rows, in_row0, in_rows,
                                           d_in_band.device.index or 0, _stream_ptr(d_in_band)))
    return d_out_band


def upscale_region_device(desc, d_in_rect, d_out, x0, y0, in_x0, in_y0, flags=None):
    """Output window of the image described by `desc` (its sizes, ratio, a and flags; its pitches are not used):
    torch uint8 CUDA tensors [h][w][C] or [F][h][w][C].  d_in_rect holds the input pixels from (in_x0, in_y0) and
    d_out receives the window whose first pixel is (x0, y0); sizes come from the shapes, row pitches from stride(-3)
    and frame strides from stride(0), so a slice of a full image works without a copy.  `flags` replaces desc.flags."""
    batched = d_in_rect.dim() == 4
    f = d_in_rect.shape[0] if batched else 1
    in_h, in_w = d_in_rect.shape[-3:-1]
    h, w = d_out.shape[-3:-1]
    d = Desc.from_buffer_copy(desc)
    d.in_pitch, d.out_pitch = d_in_rect.stride(-3), d_out.stride(-3)
    if flags is not None:
        d.flags = flags
    _check(lib().lanczos_b200_upscale_region(C.byref(d), C.c_void_p(d_in_rect.data_ptr()), C.c_void_p(d_out.data_ptr()),
                                             x0, y0, w, h, in_x0, in_y0, in_w, in_h, f,
                                             d_in_rect.stride(0) if batched else 0, d_out.stride(0) if batched else 0,
                                             d_in_rect.device.index or 0, _stream_ptr(d_in_rect)))
    return d_out


def upscale_region(img, out_w, out_h, x0, y0, w, h, a=3, scale_n=0, scale_d=0, flags=0, device=0):
    """Window [x0, x0+w) x [y0, y0+h) of the upscaled uint8 [H][W][C] host image: only the input pixels it reads go to
    the device, only the window comes back."""
    img = np.ascontiguousarray(img, dtype=np.uint8)
    ih, iw, c = img.shape
    desc = make_desc(iw, ih, out_w, out_h, c, a, scale_n, scale_d, flags=flags)
    out = np.empty((h, w, c), dtype=np.uint8)
    _check(lib().lanczos_b200_upscale_host_region(C.byref(desc), _np_ptr(img), _np_ptr(out), x0, y0, w, h, 0, device))
    return out


# ---- fixed-point "HLS mode" (the reference's lanczos() arithmetic, parity unpinned) ------------

def hls_lut(a, scale_n, bit_precision=8):
    """LUT of init_lanczos_kernel (kernel.cpp:40-45), a*scale_n+1 entries in units of 2^-BP."""
    buf = (C.c_int32 * (a * scale_n + 1))()
    _check(lib().lanczos_b200_hls_lut(a, scale_n, bit_precision, buf, len(buf)))
    return np.array(buf[:], dtype=np.int32)


def upscale_hls_device(d_in, d_out, a=3, bit_precision=8):
    """torch uint8 CUDA tensors [H][W][C] or [F][H][W][C]; integer scale = out/in."""
    batched = d_in.dim() == 4
    f = d_in.shape[0] if batched else 1
    h, w, c = d_in.shape[-3:]
    oh, ow = d_out.shape[-3:-1]
    desc = make_desc(w, h, ow, oh, c, a, 0, 0, d_in.stride(-3), d_out.stride(-3), 0)
    _check(lib().lanczos_b200_upscale_hls(C.byref(desc), C.c_void_p(d_in.data_ptr()), C.c_void_p(d_out.data_ptr()),
                                          bit_precision, f, d_in.stride(0) if batched else 0,
                                          d_out.stride(0) if batched else 0, d_in.device.index or 0, _stream_ptr(d_in)))
    return d_out
