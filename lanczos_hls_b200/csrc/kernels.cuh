// kernels.cuh -- launch interface between the C ABI (api.cu) and the CUDA kernels.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace lzb {

// Everything a kernel needs about one launch. Device pointers unless noted.
struct KParams {
    const uint8_t *in;   // points at input row `in_row0` of frame 0
    uint8_t *out;        // points at output row `out_row0` of frame 0
    long long in_pitch, out_pitch;               // bytes
    long long in_frame_stride, out_frame_stride; // bytes
    int n_frames;
    int in_w, in_h, out_w, out_h;  // full image (global coordinates)
    int channels, a, taps;         // taps = 2a
    int scale_n, scale_d;
    int out_row0, out_rows;        // band of output rows to produce
    int in_row0, in_rows;          // input rows present in `in`
    // per-coordinate tables (plan.h AxisTables)
    const int32_t *i0x; const float *wfx; const double *wdx;
    const int32_t *i0y; const float *wfy; const double *wdy;
    const float *phase_w;          // [scale_n][taps]
    float guard;                   // ascending taps, |.|-sum bound (generic + first-generation kernels)
    float guard_asc, guard_outer;  // sign-aware bounds: ascending order / outermost taps first (lanczos_v6.cu)
    int alias_rows, alias_top_row, alias_in_rows;
    unsigned flags;
    unsigned long long *strict_counter;  // may be null
};

// Shape of one main-kernel launch, handed back by the launchers (lanczos_b200_get_launch reports it).  The segment
// fields stay 0 for the kernels without vertical segments (generic, HLS).
struct LaunchShape {
    int grid_x = 0, grid_y = 0, grid_z = 0;
    int seg_periods = 0, chunk_rows = 0;
    long long resident_ctas = 0;
};
// Generic kernel: any ratio, any a<=4, channels 1..4. Returns cudaError_t as int.
int launch_generic(const KParams &p, LaunchShape *shape, cudaStream_t s);
// Specialised TMA + register-window kernels (lanczos_v6.cu, lanczos_dyn.cu). Their launchers return 0 when
// launched, a positive cudaError_t on failure, -1 when no specialisation applies (the caller then falls back).
struct FastHostTables {            // host-side views of the plan the specialised kernels need
    const float *phase_w;          // [N][2a]
    const double *phase_wd;        // [N][2a]
    const float *align_k;          // [2a]
    int exact_x, exact_y;          // AxisTables.aligned_exact
    int uniform_x, uniform_y;      // AxisTables.uniform_phase
    const int32_t *i0x_host;       // [out_w] host copy of AxisTables.i0 (x axis)
    const float *p0_chain;         // [5] Plan.p0_chain, or null when the plan could not verify it
};
// Static-phase kernels (lanczos_v6.cu): 8-byte V columns, PRMT-spliced copies, scalar constant-bank FFMA.
// *alias_in_kernel = 1 when the kernel also produced the in-place top rows (no launch_alias_rows needed).
int launch_v6(const KParams &p, const FastHostTables &t, int *kernel_id, int *alias_in_kernel, LaunchShape *shape,
              cudaStream_t s);
// Any-ratio member of the second generation (lanczos_dyn.cu): dynamic-phase H pass, static systolic V pass.
int launch_dyn(const KParams &p, const FastHostTables &t, int *kernel_id, LaunchShape *shape, cudaStream_t s);
// In-place top rows (full_TB.h:67-77 aliasing), exact double arithmetic.
int launch_alias_rows(const KParams &p, cudaStream_t s);
// Fixed-point HLS arithmetic (lanczos_hls.cu), integer scales; lut has a*n+1 entries in units of 2^-bp.
// *kernel_id: 101 = tiled kernel (a, n compile-time, bp = 8), 100 = generic tile kernel.
int launch_hls(const uint8_t *in, uint8_t *out, long long in_pitch, long long out_pitch, long long in_fs,
               long long out_fs, int n_frames, int in_w, int in_h, int out_w, int out_h, int channels, int a, int n,
               int bp, const int *lut, int *kernel_id, LaunchShape *shape, cudaStream_t s);
// Packed 24-bit words <-> interleaved RGB for lanczos_b200_stream.
int launch_words_to_rgb(const uint32_t *words, uint8_t *rgb, long long n_px, cudaStream_t s);
int launch_rgb_to_words(const uint8_t *rgb, uint32_t *words, long long n_px, cudaStream_t s);

// The reference quantiser double_to_uint8 (full_TB.h:29-37): clamp, then truncate toward zero.
__device__ __forceinline__ uint8_t quantise_f64(double x) {
    if (x > 255.0) return 255;
    if (x < 0.0) return 0;
    return (uint8_t)(int)x;
}

// Exact restatement of the reference inner loop (full_TB.h:58-63): plain double multiply then add,
// ascending tap order, no FMA contraction. Taps outside the image hold 0 (0*w adds +-0: same bits).
template <typename LoadTap>
__device__ __forceinline__ uint8_t strict_sample(const double *w, int taps, LoadTap tap) {
    double sum = 0.0;
    for (int k = 0; k < taps; k++) sum = __dadd_rn(sum, __dmul_rn((double)tap(k), w[k]));
    return quantise_f64(sum);
}

}  // namespace lzb
