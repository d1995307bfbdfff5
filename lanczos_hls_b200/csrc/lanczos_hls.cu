// lanczos_hls.cu -- the reference's fixed-point HLS arithmetic ("HLS mode", SURVEY.md 8f-1) on sm_100a.
//
// PARITY UNPINNED against the reference itself (its LUT comes from Xilinx hls::sinpi, which is not
// available; see oracle/hls_oracle.c).  Bit-exact against the integer restatement in oracle/.
//
// Replaces (reference LanczosUpscaler/): kernel.cpp:40-67 (LUT indexed by |out*D - in*N|),
// worker.cpp:45-115 compute/compute_ (integer MAC, per-tap floor in the second pass, de-ring clamp
// to the two central taps), worker.cpp:118-130 clamp_to_byte, the zero / replicate borders of
// worker.cpp:170-198, :239-275 and cyclic_buffer.h:30-42, and the vertical-then-horizontal order
// of lanczos.cpp:68-98.  Integer scales only (SCALE_D = 1).
#include "kernels.cuh"

namespace lzb {
namespace {

constexpr int HT_W = 64, HT_H = 32, HT_THREADS = 256;
constexpr int HT_COLS = HT_W + 10;  // input columns a tile can touch (n >= 1, a <= 4)

struct HlsParams {
    const uint8_t *in; uint8_t *out;
    long long in_pitch, out_pitch, in_frame_stride, out_frame_stride;
    int in_w, in_h, out_w, out_h, a, n, bp;
    int lut[128];
};

template <int C>
__global__ void __launch_bounds__(HT_THREADS) lanczos_hls_kernel(const __grid_constant__ HlsParams p) {
    __shared__ int s_mid[HT_H][HT_COLS * C];   // vertical results, bp fraction bits
    const int tid = threadIdx.x, taps = 2 * p.a, n = p.n, a = p.a, bp = p.bp;
    const int x0 = blockIdx.x * HT_W, y0 = blockIdx.y * HT_H;
    const int tw = min(HT_W, p.out_w - x0), th = min(HT_H, p.out_h - y0);
    const uint8_t *in = p.in + (long long)blockIdx.z * p.in_frame_stride;
    uint8_t *out = p.out + (long long)blockIdx.z * p.out_frame_stride;
    const int cb0 = x0 / n - a + 1;                         // first (nominal) input column of the tile
    const int ncols = (x0 + tw - 1) / n + a - cb0 + 1;

    // vertical pass (ColWorkers, worker.cpp:138-155): zero rows above, last row replicated below
    for (int idx = tid; idx < th * ncols * C; idx += HT_THREADS) {
        const int ly = idx / (ncols * C), r = idx - ly * (ncols * C);
        const int lc = r / C, c = r - lc * C;
        const int col = cb0 + lc;
        int res = 0;
        if (col >= 0) {                                     // left of the image: zeros (worker.cpp:256-265)
            const int cc = min(col, p.in_w - 1);            // right of it: replicate (worker.cpp:244)
            const int y = y0 + ly, base = y / n;
            int acc = 0, c0 = 0, c1 = 0;
            for (int j = 0; j < taps; j++) {
                const int row = base - a + 1 + j;
                int v = 0;
                if (row >= 0) v = in[(long long)min(row, p.in_h - 1) * p.in_pitch + (long long)cc * C + c];
                acc += p.lut[abs(y - row * n)] * v;         // exact: bp fraction bits (worker.cpp:58)
                if (j == a - 1) c0 = v << bp;
                if (j == a) c1 = v << bp;
            }
            res = max(min(c0, c1), min(acc, max(c0, c1)));  // de-ring clamp (worker.cpp:66-74)
        }
        s_mid[ly][lc * C + c] = res;
    }
    __syncthreads();

    // horizontal pass (RowWorkers, worker.cpp:225-236) + clamp_to_byte (worker.cpp:118-130)
    for (int idx = tid; idx < th * tw * C; idx += HT_THREADS) {
        const int ly = idx / (tw * C), r = idx - ly * (tw * C);
        const int lx = r / C, c = r - lx * C;
        const int x = x0 + lx, base = x / n;
        int acc = 0, c0 = 0, c1 = 0;
        for (int j = 0; j < taps; j++) {
            const int col = base - a + 1 + j;
            const int v = s_mid[ly][(col - cb0) * C + c];
            acc += (int)(((long long)p.lut[abs(x - col * n)] * v) >> bp);   // per-tap floor (worker.cpp:95)
            if (j == a - 1) c0 = v;
            if (j == a) c1 = v;
        }
        acc = max(min(c0, c1), min(acc, max(c0, c1)));
        out[(long long)(y0 + ly) * p.out_pitch + (long long)x * C + c] = (uint8_t)(acc >> bp);
    }
}

// ---------------------------------------------------------------------------------------------
// Tiled kernel for the common cases (a, n compile-time, BP <= 8 so that an intermediate fits 16 bits):
// the input tile is staged once in shared memory with the reference's borders already applied, every
// thread of the vertical pass walks one byte column with its 2a taps in registers (the line buffer of
// cyclic_buffer.h:4-69 as a register window), the horizontal pass computes runs of 8 pixels per thread
// from the 16-bit intermediates and stores whole words.  LUT indices are compile-time, so the weights are
// constant-bank operands.  Same integer arithmetic as lanczos_hls_kernel above, bit for bit.
// ---------------------------------------------------------------------------------------------
template <int C, int A, int N>
struct HlsGeo {
    static constexpr int TAPS = 2 * A;
    static constexpr int TIX = ((256 / C - (TAPS - 1)) / 4) * 4;   // input pixels per tile row
    static constexpr int TIY = 12;                                 // input rows per tile
    static constexpr int TW = TIX * N, TH = TIY * N;               // output tile
    static constexpr int MC = TIX + TAPS - 1, MR = TIY + TAPS - 1; // columns / rows of input the tile touches
    static constexpr int MB = MC * C;                              // bytes per staged row
    static constexpr int RUN = 8;                                  // output pixels per horizontal work item
    static constexpr int RUN_IN = RUN / N + TAPS;                  // intermediate pixels one item reads (one spare)
    static_assert(MB <= 256, "one thread per byte column in the vertical pass");
    static_assert(RUN % N == 0 && TW % RUN == 0 && (RUN * C) % 4 == 0, "runs tile the row and are whole words");
};

// de-ring clamp of worker.cpp:66-74 / :103-111
__device__ __forceinline__ int dering(int acc, int c0, int c1) { return max(min(c0, c1), min(acc, max(c0, c1))); }

// The LUT is known to hold 2^BP at distance 0 and, at the other whole-pixel distances N*k, -1 where bit k of MASK is
// set and 0 elsewhere (floor of the +-1e-17 residues of L(k), kernel.cpp:40-45; launch_hls_tile checks it): samples
// that sit on an input sample then need a shift and a subtraction or two instead of 2a multiplications.
template <int C, int A, int N, int MASK>
__global__ void __launch_bounds__(256) lanczos_hls_tile_kernel(const __grid_constant__ HlsParams p) {
    using G = HlsGeo<C, A, N>;
    constexpr int TAPS = G::TAPS, BP = 8;
    __shared__ __align__(16) uint8_t s_in[G::MR][G::MB + 1];
    __shared__ __align__(16) uint16_t s_mid[G::TH][G::MB + 1];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * G::TW, y0 = blockIdx.y * G::TH;
    const uint8_t *in = p.in + (long long)blockIdx.z * p.in_frame_stride;
    uint8_t *out = p.out + (long long)blockIdx.z * p.out_frame_stride;
    const int cb0 = x0 / N - A + 1, rb0 = y0 / N - A + 1;          // first nominal input column / row of the tile

    // stage the input tile: zeros above / left of the image, last row / column replicated below / right
    // (worker.cpp:170-198, :239-275, cyclic_buffer.h:30-42)
    for (int idx = tid; idx < G::MR * G::MB; idx += 256) {
        const int lr = idx / G::MB, b = idx - lr * G::MB;
        const int col = cb0 + b / C, c = b % C, row = rb0 + lr;
        uint8_t v = 0;
        if (row >= 0 && col >= 0)
            v = in[(long long)min(row, p.in_h - 1) * p.in_pitch + (long long)min(col, p.in_w - 1) * C + c];
        s_in[lr][b] = v;
    }
    __syncthreads();

    // vertical pass (ColWorkers::exec, worker.cpp:138-155; compute, :45-78): thread = byte column
    if (tid < G::MB) {
        int win[TAPS];
#pragma unroll
        for (int j = 0; j < TAPS - 1; j++) win[j + 1] = s_in[j][tid];
#pragma unroll
        for (int m = 0; m < G::TIY; m++) {          // input row rb0 + A - 1 + m is the "base" row of N output rows
#pragma unroll
            for (int j = 0; j < TAPS - 1; j++) win[j] = win[j + 1];
            win[TAPS - 1] = s_in[m + TAPS - 1][tid];
#pragma unroll
            for (int r = 0; r < N; r++) {           // output row y = N * base + r, tap j is row base - A + 1 + j
                int acc = 0;
#pragma unroll
                for (int j = 0; j < TAPS; j++) {
                    const int dist = r - (j - A + 1) * N;           // y - row * N
                    const int k = (j - A + 1) < 0 ? -(j - A + 1) : (j - A + 1);
                    if (r == 0) {
                        if (k == 0) acc += win[j] << BP;
                        else if ((MASK >> k) & 1) acc -= win[j];
                    } else {
                        acc += p.lut[dist < 0 ? -dist : dist] * win[j];
                    }
                }
                s_mid[m * N + r][tid] = (uint16_t)dering(acc, win[A - 1] << BP, win[A] << BP);
            }
        }
    }
    __syncthreads();

    // horizontal pass (RowWorkers::exec, worker.cpp:225-236; compute_, :81-115) + clamp_to_byte (:118-130)
    constexpr int RUNS = G::TW / G::RUN;
    const bool words_ok = (p.out_pitch % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 3) == 0);
    for (int item = tid; item < G::TH * RUNS; item += 256) {
        const int ly = item / RUNS, run = item - ly * RUNS;
        const int y = y0 + ly, xr = x0 + run * G::RUN;              // first output pixel of the run
        if (y >= p.out_h || xr >= p.out_w) continue;
        const uint16_t *mrow = &s_mid[ly][(run * G::RUN / N) * C];  // intermediate pixel (xr / N - A + 1), channel 0
        int mid[G::RUN_IN * C];
#pragma unroll
        for (int i = 0; i < G::RUN_IN * C; i++) mid[i] = (i < (G::RUN / N + TAPS - 1) * C) ? (int)mrow[i] : 0;
        uint32_t ow[G::RUN * C / 4];
#pragma unroll
        for (int i = 0; i < G::RUN * C / 4; i++) ow[i] = 0u;
#pragma unroll
        for (int ob = 0; ob < G::RUN * C; ob++) {
            const int lx = ob / C, c = ob % C;
            const int base = lx / N, r = lx % N;                    // x = N * (xr / N + base) + r
            int acc = 0;
#pragma unroll
            for (int j = 0; j < TAPS; j++) {
                const int dist = r - (j - A + 1) * N;               // x - col * N
                const int k = (j - A + 1) < 0 ? -(j - A + 1) : (j - A + 1);
                const int v = mid[(base + j) * C + c];
                if (r == 0) {
                    if (k == 0) acc += v;                           // (2^BP * v) >> BP
                    else if ((MASK >> k) & 1) acc += (-v) >> BP;    // (-1 * v) >> BP, arithmetic shift = floor
                } else {
                    acc += (p.lut[dist < 0 ? -dist : dist] * v) >> BP;   // per-tap floor (worker.cpp:95)
                }
            }
            acc = dering(acc, mid[(base + A - 1) * C + c], mid[(base + A) * C + c]);
            ow[ob / 4] |= (uint32_t)(acc >> BP) << (8 * (ob % 4));
        }
        uint8_t *o = out + (long long)y * p.out_pitch + (long long)xr * C;
        if (words_ok && xr + G::RUN <= p.out_w) {
#pragma unroll
            for (int i = 0; i < G::RUN * C / 4; i++) reinterpret_cast<uint32_t *>(o)[i] = ow[i];
        } else {
            const int nb = (min(xr + G::RUN, p.out_w) - xr) * C;
            for (int i = 0; i < nb; i++) o[i] = (uint8_t)(ow[i / 4] >> (8 * (i % 4)));
        }
    }
}

// Returns -1 without launching when the LUT lacks the whole-pixel pattern the MASK instance assumes (the caller then
// runs lanczos_hls_kernel).  The library's own LUT always has it for the configurations below.
template <int C, int A, int N, int MASK>
int launch_hls_tile(const HlsParams &p, int n_frames, cudaStream_t s) {
    using G = HlsGeo<C, A, N>;
    bool pattern = p.lut[0] == (1 << 8);
    for (int k = 1; k <= A; k++) pattern = pattern && p.lut[k * N] == (((MASK >> k) & 1) ? -1 : 0);
    if (!pattern) return -1;
    dim3 grid((p.out_w + G::TW - 1) / G::TW, (p.out_h + G::TH - 1) / G::TH, n_frames);
    lanczos_hls_tile_kernel<C, A, N, MASK><<<grid, 256, 0, s>>>(p);
    return (int)cudaGetLastError();
}

}  // namespace

int launch_hls(const uint8_t *in, uint8_t *out, long long in_pitch, long long out_pitch, long long in_fs,
               long long out_fs, int n_frames, int in_w, int in_h, int out_w, int out_h, int channels, int a, int n,
               int bp, const int *lut, int *kernel_id, cudaStream_t s) {
    HlsParams p{};
    p.in = in; p.out = out; p.in_pitch = in_pitch; p.out_pitch = out_pitch;
    p.in_frame_stride = in_fs; p.out_frame_stride = out_fs;
    p.in_w = in_w; p.in_h = in_h; p.out_w = out_w; p.out_h = out_h; p.a = a; p.n = n; p.bp = bp;
    for (int i = 0; i <= a * n; i++) p.lut[i] = lut[i];
    if (bp == 8) {      // 16-bit intermediates: the tiled kernel (the reference's template BIT_PRECISION is 8)
        // a = 3: floor(L(2) * 2^BP) = -1 (sin(2 pi) < 0 in double), the other whole-pixel entries are 0; a = 2: all 0
        int rc = -1;
#define HLS_CASE(c, aa, nn, mask) if (channels == c && a == aa && n == nn) rc = launch_hls_tile<c, aa, nn, mask>(p, n_frames, s);
        HLS_CASE(3, 3, 2, 4) HLS_CASE(4, 3, 2, 4) HLS_CASE(1, 3, 2, 4) HLS_CASE(3, 2, 2, 0) HLS_CASE(3, 3, 4, 4) HLS_CASE(3, 2, 4, 0)
#undef HLS_CASE
        if (rc >= 0) {
            *kernel_id = 101;
            return rc;
        }
    }
    *kernel_id = 100;
    dim3 grid((out_w + HT_W - 1) / HT_W, (out_h + HT_H - 1) / HT_H, n_frames);
    switch (channels) {
        case 1: lanczos_hls_kernel<1><<<grid, HT_THREADS, 0, s>>>(p); break;
        case 2: lanczos_hls_kernel<2><<<grid, HT_THREADS, 0, s>>>(p); break;
        case 3: lanczos_hls_kernel<3><<<grid, HT_THREADS, 0, s>>>(p); break;
        default: lanczos_hls_kernel<4><<<grid, HT_THREADS, 0, s>>>(p); break;
    }
    return (int)cudaGetLastError();
}

}  // namespace lzb
