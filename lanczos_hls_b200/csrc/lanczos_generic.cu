// lanczos_generic.cu -- generic fused H->V Lanczos kernel (any ratio N/D >= 1, a <= 4,
// channels 1..4) and the in-place top-rows kernel. sm_100a.
//
// Replaces, for the software path, lanczos_interpolate_row + lanczos_interpolate_col
// (reference full_TB.h:55-77) and, structurally, the HLS streaming loop
// fillColBuffer/fillRowBuffer (lanczos.cpp:21-51) with its cyclic line buffer
// (cyclic_buffer/cyclic_buffer.h:4-69): one CTA stages an input tile plus its Lanczos halo in
// shared memory, runs the horizontal pass into a shared uint8 intermediate (the reference
// truncates between the passes, full_TB.h:63), then the vertical pass straight to global.
//
// Arithmetic: fp32 FMA with per-coordinate float weights.  Whenever the fp32 sum lies within
// `guard` (a rigorous bound on the fp32-vs-double error, plan.cpp) of an integer 1..255, the
// sample is re-evaluated exactly like the reference does (double multiply, double add, ascending
// taps, kernels.cuh exact_add) so the truncated result is bit-identical.
#include "kernels.cuh"

namespace lzb {

namespace {

constexpr int GT_W = 64;        // output pixels per tile row
constexpr int GT_H = 32;        // output rows per tile
constexpr int GT_THREADS = 256;
constexpr int GT_IN_ROWS = GT_H + 8;   // upscale: input span <= outputs + 2a
constexpr int GT_IN_COLS = GT_W + 8;

__device__ __forceinline__ bool near_integer(float s, float guard) {
    const float r = rintf(s);
    return fabsf(s - r) < guard && r >= 1.f && r <= 255.f;
}

template <int C>
__global__ void __launch_bounds__(GT_THREADS) lanczos_generic_kernel(const KParams p) {
    __shared__ int s_i0x[GT_W], s_i0y[GT_H];
    __shared__ float s_wx[GT_W][8], s_wy[GT_H][8];
    __shared__ __align__(16) uint8_t s_in[GT_IN_ROWS][GT_IN_COLS * C];
    __shared__ __align__(16) uint8_t s_mid[GT_IN_ROWS][GT_W * C];

    const int tid = threadIdx.x;
    const int taps = p.taps;
    const int x0 = p.out_col0 + blockIdx.x * GT_W;    // first output pixel of the tile (global index)
    const int y0 = p.out_row0 + blockIdx.y * GT_H;    // first output row (global index)
    const int frame = blockIdx.z;
    const int tw = min(GT_W, p.out_col0 + p.out_cols - x0);
    const int th = min(GT_H, p.out_row0 + p.out_rows - y0);
    const uint8_t *in = p.in + (long long)frame * p.in_frame_stride;
    uint8_t *out = p.out + (long long)frame * p.out_frame_stride;

    if (tid < tw) {
        s_i0x[tid] = p.i0x[x0 + tid];
        for (int k = 0; k < taps; k++) s_wx[tid][k] = p.wfx[(long long)(x0 + tid) * taps + k];
    }
    if (tid >= 64 && tid < 64 + th) {
        const int t = tid - 64;
        s_i0y[t] = p.i0y[y0 + t];
        for (int k = 0; k < taps; k++) s_wy[t][k] = p.wfy[(long long)(y0 + t) * taps + k];
    }
    __syncthreads();

    const int cx0 = s_i0x[0];
    const int ncols = s_i0x[tw - 1] + taps - cx0;    // input pixels spanned (<= GT_IN_COLS)
    const int ry0 = s_i0y[0];
    const int nrows = s_i0y[th - 1] + taps - ry0;    // input rows spanned (<= GT_IN_ROWS)

    // stage the input tile + halo; everything outside the image is 0 (full_TB.h:59,72 drop those taps).  Inside the
    // image every staged byte is a tap of a window pixel, so it lies in the supplied input rect.
    const int row_bytes = ncols * C;
    for (int idx = tid; idx < nrows * row_bytes; idx += GT_THREADS) {
        const int r = idx / row_bytes, b = idx - r * row_bytes;
        const int gy = ry0 + r;
        const int gb = cx0 * C + b;
        uint8_t v = 0;
        if (gy >= 0 && gy < p.in_h && gb >= 0 && gb < p.in_w * C)
            v = in[(long long)(gy - p.in_row0) * p.in_pitch + gb - p.in_col0 * C];
        s_in[r][b] = v;
    }
    __syncthreads();

    // horizontal pass (full_TB.h:55-65) on every staged row
    const int out_bytes = tw * C;
    for (int idx = tid; idx < nrows * out_bytes; idx += GT_THREADS) {
        const int r = idx / out_bytes, j = idx - r * out_bytes;
        const int lx = j / C, c = j - lx * C;
        const uint8_t *src = &s_in[r][(s_i0x[lx] - cx0) * C + c];
        float s = 0.f;
        for (int k = 0; k < taps; k++) s = fmaf((float)src[k * C], s_wx[lx][k], s);
        uint8_t q = quantise_f32(s);
        if (near_integer(s, p.guard)) {
            const double *w = p.wdx + (long long)(x0 + lx) * taps;
            q = strict_sample(w, taps, [&](int k) { return src[k * C]; });
            if (p.strict_counter) atomicAdd(p.strict_counter, 1ULL);
        }
        s_mid[r][j] = q;
    }
    __syncthreads();

    // vertical pass (full_TB.h:67-77, ping-pong semantics; the in-place top rows are redone by
    // lanczos_alias_rows_kernel)
    for (int idx = tid; idx < th * out_bytes; idx += GT_THREADS) {
        const int ly = idx / out_bytes, j = idx - ly * out_bytes;
        const int rb = s_i0y[ly] - ry0;
        float s = 0.f;
        for (int k = 0; k < taps; k++) s = fmaf((float)s_mid[rb + k][j], s_wy[ly][k], s);
        uint8_t q = quantise_f32(s);
        if (near_integer(s, p.guard)) {
            const double *w = p.wdy + (long long)(y0 + ly) * taps;
            q = strict_sample(w, taps, [&](int k) { return s_mid[rb + k][j]; });
            if (p.strict_counter) atomicAdd(p.strict_counter, 1ULL);
        }
        out[(long long)(y0 + ly - p.out_row0) * p.out_pitch + (long long)(x0 - p.out_col0) * C + j] = q;
    }
}

// ---- in-place top rows ----------------------------------------------------------------------
// The reference's column pass works in place from the bottom row up (full_TB.h:67-77).  Row xx
// reads rows first..last of the same plane; every row i > xx in that window has already been
// overwritten with its FINAL value, rows i <= xx still hold the horizontal result.  That only
// happens for the first `alias_rows` rows.  One thread per output byte column of the window walks rows
// alias_top_row..0 with the reference's exact double arithmetic and writes rows < alias_rows.
__global__ void __launch_bounds__(128) lanczos_alias_rows_kernel(const KParams p) {
    const int C = p.channels, taps = p.taps;
    const long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // output byte column of the window
    if (col >= (long long)p.out_cols * C) return;
    const int frame = blockIdx.y;
    const uint8_t *in = p.in + (long long)frame * p.in_frame_stride;
    uint8_t *out = p.out + (long long)frame * p.out_frame_stride;
    const long long gcol = (long long)p.out_col0 * C + col;                  // ... and of the image
    const int xx = (int)(gcol / C), c = (int)(gcol - (long long)xx * C);
    const int i0x = p.i0x[xx];
    double wx[8];
    for (int k = 0; k < taps; k++) wx[k] = p.wdx[(long long)xx * taps + k];

    // horizontal result of input row i at this column, exact (full_TB.h:55-65)
    auto mid = [&](int i) -> uint8_t {
        const uint8_t *row = in + (long long)(i - p.in_row0) * p.in_pitch;
        return strict_sample(wx, taps, [&](int k) -> uint8_t {
            const int px = i0x + k;
            return (px >= 0 && px < p.in_w) ? row[(long long)(px - p.in_col0) * C + c] : (uint8_t)0;
        });
    };

    // horizontal results of the input rows the recurrence touches, computed once per row
    constexpr int kMaxT = 32;
    uint8_t T[kMaxT];
    const bool cached = p.alias_in_rows <= kMaxT;
    if (cached)
        for (int i = 0; i < p.alias_in_rows; i++) T[i] = mid(i);

    uint8_t fin[8];  // final values of rows (xx, xx+taps): index row & 7
    for (int k = 0; k < 8; k++) fin[k] = 0;
    for (int yy = p.alias_top_row; yy >= 0; yy--) {
        const int first = p.i0y[yy];
        const double *wy = p.wdy + (long long)yy * taps;
        double sum = 0.0;
        for (int k = 0; k < taps; k++) {
            const int i = first + k;
            if (i < 0 || i >= p.in_h) continue;  // full_TB.h:72 clips the window
            const uint8_t v = (i > yy) ? fin[i & 7] : (cached ? T[i] : mid(i));
            sum = exact_add(sum, v, wy[k]);
        }
        const uint8_t q = quantise_f64(sum);
        fin[yy & 7] = q;
        if (yy < p.alias_rows && yy >= p.out_row0 && yy < p.out_row0 + p.out_rows)
            out[(long long)(yy - p.out_row0) * p.out_pitch + col] = q;
    }
}

// ---- layout helpers --------------------------------------------------------------------------
// worker.cpp:35-43 packing: channel i in bits [8i+7:8i] of the stream word
__global__ void words_to_rgb_kernel(const uint32_t *words, uint8_t *rgb, long long n_px) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_px) return;
    const uint32_t w = words[i];
    rgb[3 * i + 0] = (uint8_t)(w & 0xff);
    rgb[3 * i + 1] = (uint8_t)((w >> 8) & 0xff);
    rgb[3 * i + 2] = (uint8_t)((w >> 16) & 0xff);
}
__global__ void rgb_to_words_kernel(const uint8_t *rgb, uint32_t *words, long long n_px) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_px) return;
    words[i] = (uint32_t)rgb[3 * i] | ((uint32_t)rgb[3 * i + 1] << 8) | ((uint32_t)rgb[3 * i + 2] << 16);
}

}  // namespace

int launch_generic(const KParams &p, LaunchShape *shape, cudaStream_t s) {
    dim3 grid((p.out_cols + GT_W - 1) / GT_W, (p.out_rows + GT_H - 1) / GT_H, p.n_frames);
    *shape = LaunchShape{(int)grid.x, (int)grid.y, (int)grid.z};
    dim3 block(GT_THREADS);
    switch (p.channels) {
        case 1: lanczos_generic_kernel<1><<<grid, block, 0, s>>>(p); break;
        case 2: lanczos_generic_kernel<2><<<grid, block, 0, s>>>(p); break;
        case 3: lanczos_generic_kernel<3><<<grid, block, 0, s>>>(p); break;
        default: lanczos_generic_kernel<4><<<grid, block, 0, s>>>(p); break;
    }
    return (int)cudaGetLastError();
}

int launch_alias_rows(const KParams &p, cudaStream_t s) {
    const long long cols = (long long)p.out_cols * p.channels;
    dim3 grid((unsigned)((cols + 127) / 128), p.n_frames);
    lanczos_alias_rows_kernel<<<grid, 128, 0, s>>>(p);
    return (int)cudaGetLastError();
}

int launch_words_to_rgb(const uint32_t *words, uint8_t *rgb, long long n_px, cudaStream_t s) {
    words_to_rgb_kernel<<<(unsigned)((n_px + 255) / 256), 256, 0, s>>>(words, rgb, n_px);
    return (int)cudaGetLastError();
}
int launch_rgb_to_words(const uint8_t *rgb, uint32_t *words, long long n_px, cudaStream_t s) {
    rgb_to_words_kernel<<<(unsigned)((n_px + 255) / 256), 256, 0, s>>>(rgb, words, n_px);
    return (int)cudaGetLastError();
}

}  // namespace lzb
