"""lanczos_hls_b200 -- B200-native Lanczos upscaler (software path of PKBeam/Lanczos-HLS).

The product is the CUDA library `liblanczos_b200.so` behind the C ABI in
include/lanczos_b200.h.  This package is the thin host-side mirror of the
reference's interface for that path (`lanczos_expected`, the packed-word
`lanczos` stream, the params.h macros as a descriptor).  There is no CPU
fallback: every compute call goes through the CUDA library and raises if it is
missing or no GPU is usable.
"""
from .api import (  # noqa: F401
    Desc,
    LanczosError,
    FLAG_NO_ALIAS,
    FLAG_FAST_ALIGNED,
    FLAG_TOLERANCE_1LSB,
    FLAG_INDEPENDENT,
    FLAG_GENERIC_KERNEL,
    abi_version,
    alias_rows,
    band_input_rows,
    bind_host_to_device,
    device_count,
    lanczos_expected,
    lanczos_stream,
    lib,
    lib_path,
    make_desc,
    phase_table,
    phase0_chain,
    reduce_ratio,
    region_input_rect,
    resolve,
    stats,
    launch,
    enable_stats,
    upscale,
    upscale_bands_multi_gpu,
    upscale_device,
    upscale_batch_device,
    upscale_band_device,
    upscale_region,
    upscale_region_device,
    upscale_planar_device,
    PinnedBuffer,
    hls_lut,
    upscale_hls_device,
)
