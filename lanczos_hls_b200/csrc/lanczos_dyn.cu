// lanczos_dyn.cu -- any-ratio member of the second-generation kernels (ratio period N <= 32, e.g. 17/10).
//
// Same structure as lanczos_v6.cu (see there for what each piece replaces in the reference): every warp owns one
// strip of 128 output byte-columns, its own TMA stages, its own shared-memory ring of horizontal results and
// its own mbarriers; rows stream through in chunks of RB input rows.  What differs:
//   * H pass: a lane owns one 32-bit word of the strip (the same 4 byte-columns it owns in the V pass).  Its
//     tap offsets and its 4 x 2a phase weights are fixed for the whole strip, so they are looked up once
//     (plan tables i0x / polyphase table) and kept in registers; per row it does 4 x 2a byte loads from the
//     staged input row, FHADD conversions and FFMAs.  No compile-time knowledge of the horizontal phase
//     pattern is needed (17/10 RGB has a 51-byte period that fits no vector width).
//   * V pass: the systolic scheme of lanczos_v6.cu with 4-byte columns; the vertical phase pattern is static
//     (template N, D), the loop body is one ratio period (lcm(D,2) input rows).
//   * Phase-0 samples (output coordinate on an input sample) are always evaluated with the reference's double
//     arithmetic: for ratios like 17/10 the coordinate xx/SCALE is not exactly integral in double, so the
//     reference's weights there are 1-eps and +-1e-13 and its result is v or v-1 depending on all six taps.
//     In the H pass these samples sit in fixed byte columns of the strip: one lane per (column, row) after the
//     row loop.  In the V pass they are whole output rows (every N-th): v_fix_dyn.
// Exactness of everything else: fp32 chains from -guard, truncation compared at +guard, exact double
// re-evaluation (full_TB.h:58-63 / :71-75) when they differ.  MODE 1 = LANCZOS_FLAG_TOLERANCE_1LSB (V pass plain fp32).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <cuda.h>

#include "../../include/lanczos_b200.h"
#include "fast_common.cuh"

namespace lzb {

namespace {

struct DynParams : StripParams {
    const int32_t *i0x;       // [out_w] first tap pixel per output pixel (plan AxisTables)
    const double *wdx, *wdy;  // per-coordinate double weights (exact evaluation)
    float guard;              // rigorous fp32 error bound (x1.06) of ascending-order chains with the phase table
    int p0_filter;            // 1: phase-0 coordinates are exactly integral and the residues have the a = 3 pattern,
                              //    so the "cannot flip" test of lanczos_v6.cu (K = 3/8) decides most phase-0 samples
    float wtab[32 * 8];       // polyphase table [N][8] (padded to 8 taps), times 2^24
    unsigned long long *strict_counter;
};

template <int C, int A, int N, int D>
struct GeoD {
    static constexpr int VB = 4;                         // byte-columns per lane
    static constexpr int SWB = 32 * VB;                  // strip width in output bytes = ring pitch
    static constexpr int TAPS = 2 * A;
    static constexpr int U = lcm2(D);                    // input rows per V loop iteration (one ratio period, even)
    static constexpr int RB = U * cdiv(TAPS > 6 ? TAPS : 6, U);    // input rows per chunk (>= 2a - 1: see the ring)
    static constexpr int REGIONS = 2;
    static constexpr int RING = REGIONS * RB;
    static constexpr int STAGES = 4;
    // input pixels a strip can touch: its (SWB/C + 2) output pixels span that many * D/N input pixels, plus taps
    static constexpr int IN_PX = ((SWB / C + 2) * D) / N + 2 + TAPS;
    static constexpr int BOX_B = 16 * cdiv(IN_PX * C + 15, 16);   // + 15: the box starts on a 16-byte boundary
    static constexpr int STAGE_B = 128 * cdiv(RB * BOX_B, 128);
    static constexpr int S0 = (((1 - 2 * A) % D) + D) % D;
    static constexpr int YROWS = N * RB / D;             // output rows completed per chunk
    static_assert(TAPS - 1 <= RB, "tap rows must not reach further back than one ring region");
    static_assert(BOX_B / 4 <= 256, "TMA box too wide");
    static_assert(N <= 32, "phase table too large for kernel params");
    static_assert(cdiv(S0 * N, D) + YROWS <= 32, "fix mask (bit per output row) too small");
};

// fma.rn.f32 WITHOUT .ftz whatever the compilation flags say (-use_fast_math would flush the denormal operand)
__device__ __forceinline__ float fma_keep_denormals(float a, float b, float c) {
    float d;
    asm("fma.rn.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

__device__ __forceinline__ float2 ffma2_keep_denormals(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}

template <class G>
struct __align__(128) SmemD {             // one per warp
    uint8_t in[G::STAGES][G::STAGE_B];    // TMA destinations, row lr at lr * BOX_B
    uint8_t ring[G::RING][G::SWB];        // H-pass results (uint8), row r lives in slot (r - rs) % RING
    unsigned long long full[G::STAGES];
};


// exact evaluation of the bytes of one output row whose fp32 truncation is in doubt, and of whole phase-0 rows
struct VFixD {
    const uint8_t *col;       // this lane's column in ring row 0
    uint8_t *ocol;            // this lane's column in output row `ybase`
    long long opitch;
    int ybase, rs, nbytes;
    uint32_t rows;            // bit yy: output row ybase + yy
};

template <int A, int N, int D, int RING, int SWB>
__device__ __noinline__ int v_fix_dyn(const DynParams &p, const VFixD a) {
    constexpr int TAPS = 2 * A;
    int n_strict = 0;
#pragma unroll 1
    for (uint32_t m = a.rows; m; m &= m - 1) {
        const int yy = __ffs(m) - 1;
        const int y = a.ybase + yy;
        const int ph = (y * D) % N;
        const int s0 = ((y * D) / N - A + 1 - a.rs) % RING;       // ring slot of the first tap row (full_TB.h:72)
        uint8_t *orow = a.ocol + (long long)yy * a.opitch;
        uint32_t tw[TAPS];
#pragma unroll
        for (int k = 0; k < TAPS; k++) tw[k] = *reinterpret_cast<const uint32_t *>(a.col + ((s0 + k) % RING) * SWB);
        uint32_t need = 0xfu;
        if (ph != 0) {
            // the hot path's fp32 chains again (ascending taps, same weights: same bits)
            float acc[4];
#pragma unroll
            for (int i = 0; i < 4; i++) acc[i] = -p.guard;
#pragma unroll
            for (int k = 0; k < TAPS; k++) {
                float x[4];
                word_to_f32x4(tw[k], x[0], x[1], x[2], x[3]);
                const float wk = p.wtab[ph * 8 + k];
#pragma unroll
                for (int i = 0; i < 4; i++) acc[i] = fmaf(x[i], wk, acc[i]);
            }
            const float g2 = 2.f * p.guard;
            const uint32_t dx = quantise4(acc[0], acc[1], acc[2], acc[3]) ^ quantise4(acc[0] + g2, acc[1] + g2, acc[2] + g2, acc[3] + g2);
            need = 0;
#pragma unroll
            for (int e = 0; e < 4; e++)
                if ((dx >> (8 * e)) & 0xffu) need |= 1u << e;
        }
        need &= (a.nbytes >= 4) ? 0xfu : ((1u << a.nbytes) - 1u);
        if (!need) continue;
        double w[TAPS];
#pragma unroll
        for (int k = 0; k < TAPS; k++) w[k] = p.wdy[(long long)y * TAPS + k];
#pragma unroll
        for (int e = 0; e < 4; e++) {
            if (!((need >> e) & 1u)) continue;
            double sum = 0.0;
#pragma unroll
            for (int k = 0; k < TAPS; k++) {
                const double v = __hiloint2double(0x43300000, (int)((tw[k] >> (8 * e)) & 0xffu)) - 4503599627370496.0;
                sum = __dadd_rn(sum, __dmul_rn(v, w[k]));
            }
            orow[e] = quantise_f64(sum);
            n_strict++;
        }
    }
    return n_strict;
}

template <int C, int A, int N, int D, int MODE>
__global__ void __launch_bounds__(32, 16)
lanczos_dyn_kernel(const __grid_constant__ CUtensorMap in_map, const __grid_constant__ DynParams p) {
    using G = GeoD<C, A, N, D>;
    constexpr int TAPS = G::TAPS, SWB = G::SWB, VB = G::VB, RB = G::RB;
    constexpr int NSLOT = nslot<N, D, TAPS>();
    constexpr int CNTMAX = cntmax<N, D>();
    extern __shared__ __align__(128) uint8_t smem_raw[];
    SmemD<G> &sm = *reinterpret_cast<SmemD<G> *>(smem_raw);

    const int lane = threadIdx.x;
    const int strip = blockIdx.x, seg = blockIdx.y, frame = blockIdx.z;
    uint8_t *out_frame = p.out + (long long)frame * p.out_frame_stride;

    // horizontal extent
    const int obyte0 = strip * SWB;
    const int row_bytes = p.out_w * C;
    const int valid_bytes = min(SWB, row_bytes - obyte0);     // > 0 by construction of the grid, multiple of 4
    const int xbyte0 = ((p.i0x[obyte0 / C] * C) >> 4) << 4;   // staged rows start here (16-byte aligned, may be < 0)
    // vertical extent: periods [pv0, pv1) -> output rows [N*pv0, N*pv1), clipped to the band
    const int pv0 = p.vperiod0 + seg * p.seg_periods;
    const int y_end_band = p.out_row0 + p.out_rows;
    const int pv1 = min(pv0 + p.seg_periods, (y_end_band + N - 1) / N);
    const int ys = max(N * pv0, p.out_row0), ye = min(N * pv1, y_end_band);
    if (ys >= ye) return;
    const int rs = D * pv0 - A + 1;                           // first intermediate row pushed
    const int nrows = D * (pv1 - pv0) + TAPS - 1;             // rows to push
    const int nchunks = (nrows + RB - 1) / RB;

    uint32_t full0 = smem_u32(&sm.full[0]);
    asm volatile("" : "+r"(full0));
    if (lane == 0) {
        for (int i = 0; i < G::STAGES; i++) mbar_init(full0 + 8 * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    constexpr uint32_t kStageBytes = RB * G::BOX_B;
    auto issue = [&](int chunk) {
        const uint32_t bar = full0 + 8 * (chunk % G::STAGES);
        mbar_expect_tx(bar, kStageBytes);
        tma_load_3d(smem_u32(&sm.in[chunk % G::STAGES][0]), &in_map, xbyte0 / 4, rs + chunk * RB - p.in_row0, frame, bar);
    };
    if (lane == 0)
        for (int i = 0; i < G::STAGES && i < nchunks; i++) issue(i);

    // ------------------------------ per-lane H geometry (fixed for the strip) ------------------------------
    const bool active = VB * lane < valid_bytes;
    int off[4];                 // byte offset of tap 0 in a staged row
    // A byte loaded with LDS.U8 sits in the low bits of a register: read as fp32 that is the DENORMAL b * 2^-149,
    // and FFMA takes denormal operands at full rate.  With weights times 2^100 the chain runs in units of 2^-49
    // pixels: every intermediate is the same mantissa as in pixel units with the exponent shifted (nothing
    // underflows: the smallest term is ~2^-62), so after one exact multiplication by 2^49 the sum has the very
    // bits of the PRMT/FHADD formulation used elsewhere -- and the per-tap conversion instruction is gone.
    constexpr float kDenScale = 7.555786372591432e22f;    // 2^76: wtab already carries 2^24
    constexpr float kDenUnscale = 5.62949953421312e14f;  // 2^49
    constexpr float kDenGuard = 1.7763568394002505e-15f; // 2^-49
    float wq[4][TAPS];          // phase weights (times 2^100) of the lane's 4 samples
    uint32_t p0mask = 0;        // byte lanes (0xff each) that hold phase-0 samples
#pragma unroll
    for (int e = 0; e < 4; e++) {
        const int ob = min(obyte0 + VB * lane + e, row_bytes - 1);
        const int xx = ob / C, c = ob - xx * C;
        const int ph = (xx * D) % N;
        off[e] = p.i0x[xx] * C + c - xbyte0;
#pragma unroll
        for (int k = 0; k < TAPS; k++) wq[e][k] = p.wtab[ph * 8 + k] * kDenScale;   // exact: a power of two
        if (ph == 0) p0mask |= 0xffu << (8 * e);
    }
    // C = 3: the lane's fourth byte is the channel of its first byte one pixel on, and its taps start 0 or 1 pixel
    // later (upscaling), i.e. they are six of the seven bytes off[0] + 3k, k = 0..6.  Its weights are spread over
    // those seven positions (a zero at the unused end: fma(t, 0, acc) == acc, same bits) and its six loads are gone.
    constexpr bool SHARE = (C == 3);
    float w3s[TAPS + 1];
#pragma unroll
    for (int k = 0; k <= TAPS; k++) w3s[k] = 0.f;
    if (SHARE) {
        const int d3 = (off[3] - off[0]) / C;      // 0 or 1 for every lane that owns columns
#pragma unroll
        for (int k = 0; k <= TAPS; k++) {
            const int src = k - d3;
            float w = 0.f;
#pragma unroll
            for (int j = 0; j < TAPS; j++) w = (src == j) ? wq[3][j] : w;
            w3s[k] = w;
        }
    }
    // phase-0 byte columns of the strip: pixels xx = N*m, all channels;
    // enumerate them on the fly: column index q -> output byte column (or -1)
    auto p0_column = [&](int q) -> int {
        // the strip starts at pixel obyte0 / C (possibly in the middle of it); candidates are pixels
        // px = floor(obyte0 / C / N) * N + j * N for j = 0, 1, ...
        const int base_px = ((obyte0 / C) / N) * N;
        const int j = q / C, c = q - j * C;
        const int ob = (base_px + j * N) * C + c;
        return (ob >= obyte0 && ob < obyte0 + valid_bytes) ? ob : -1;
    };
    constexpr int P0Q = (SWB / (N * C) + 2) * C;              // candidate columns to scan
    // after the row loop lane l takes the (column, row) pairs t = l, l + 32, ...: the same pairs in every chunk, so
    // what each needs is packed into one register now -- row << 20 | strip byte column << 12 | tap-0 byte offset
    // in the staged row -- or -1 when the candidate column lies outside the strip
    constexpr int P0_ITEMS = (P0Q * RB + 31) / 32;
    static_assert(G::BOX_B < 4096 && SWB <= 256 && RB < 2048, "packing of the phase-0 work items");
    int p0_item[P0_ITEMS];
#pragma unroll
    for (int i = 0; i < P0_ITEMS; i++) {
        const int t = lane + 32 * i;
        const int q = t / RB, lr = t - q * RB;
        const int ob = (t < P0Q * RB) ? p0_column(q) : -1;
        p0_item[i] = -1;
        if (ob >= 0) {
            const int xx = ob / C, c = ob - xx * C;
            p0_item[i] = (lr << 20) | ((ob - obyte0) << 12) | (p.i0x[xx] * C + c - xbyte0);
        }
    }

    int n_strict = 0;
    const float guard = p.guard, g2 = 2.f * p.guard;

    // ------------------------------ H pass of one chunk ------------------------------
    auto h_pass = [&](int chunk) {
        const int st = chunk % G::STAGES;
        mbar_wait(full0 + 8 * st, (chunk / G::STAGES) & 1);
        const int slot0 = (chunk % G::REGIONS) * RB;
        if (active) {
#pragma unroll 2
            for (int lr = 0; lr < RB; lr++) {
                const uint8_t *row = &sm.in[st][lr * G::BOX_B];
                float xa[4];
                if (SHARE) {
                    float t[TAPS + 1];
#pragma unroll
                    for (int k = 0; k <= TAPS; k++) t[k] = __uint_as_float((uint32_t)row[off[0] + k * C]);
                    float a0 = -guard * kDenGuard, a3 = a0;
#pragma unroll
                    for (int k = 0; k < TAPS; k++) a0 = fma_keep_denormals(t[k], wq[0][k], a0);
#pragma unroll
                    for (int k = 0; k <= TAPS; k++) a3 = fma_keep_denormals(t[k], w3s[k], a3);
                    xa[0] = a0 * kDenUnscale;
                    xa[3] = a3 * kDenUnscale;
                }
                // the other samples two at a time: one FFMA2 per tap for both (each with its own weights; same rounding
                // as two FFMAs, one issue slot)
#pragma unroll
                for (int e = SHARE ? 1 : 0; e < (SHARE ? 3 : 4); e += 2) {
                    float2 acc = make_float2(-guard * kDenGuard, -guard * kDenGuard);
#pragma unroll
                    for (int k = 0; k < TAPS; k++)
                        acc = ffma2_keep_denormals(make_float2(__uint_as_float((uint32_t)row[off[e] + k * C]), __uint_as_float((uint32_t)row[off[e + 1] + k * C])),
                                                   make_float2(wq[e][k], wq[e + 1][k]), acc);
                    const float2 r = __fmul2_rn(acc, make_float2(kDenUnscale, kDenUnscale));
                    xa[e] = r.x;
                    xa[e + 1] = r.y;
                }
                const uint32_t qa = quantise4(xa[0], xa[1], xa[2], xa[3]);
                const uint32_t qb = quantise4(xa[0] + g2, xa[1] + g2, xa[2] + g2, xa[3] + g2);
                uint8_t *dst = &sm.ring[slot0 + lr][VB * lane];
                *reinterpret_cast<uint32_t *>(dst) = qa;
                const uint32_t dm = (qa ^ qb) & ~p0mask;        // phase-0 bytes are redone below in any case
                if (dm) {
                    // rare: truncation in doubt -> this lane evaluates the byte like the reference (full_TB.h:58-63)
#pragma unroll 1
                    for (int e = 0; e < 4; e++) {
                        if (!((dm >> (8 * e)) & 0xffu)) continue;
                        const int xx = (obyte0 + VB * lane + e) / C;
                        dst[e] = exact_taps<TAPS>(row + off[e], C, [&](int k) { return p.wdx[(long long)xx * TAPS + k]; });
                        n_strict++;
                    }
                }
            }
        }
        __syncwarp();   // the words written above are patched byte-wise by other lanes now
        // phase-0 samples: fixed byte columns of the strip, every row; one (column, row) per lane and round
#pragma unroll
        for (int i = 0; i < P0_ITEMS; i++) {
            const int it = p0_item[i];
            if (it < 0) continue;
            const int lr = it >> 20, col = (it >> 12) & 0xff;
            const uint8_t *tap0 = &sm.in[st][lr * G::BOX_B] + (it & 0xfff);
            if (p.p0_filter) {
                // the reference returns the centre value v unless the negative residues at +-2 pixels outweigh half
                // the spacing of doubles below v (plan.cpp): 3 b <= 8 v on both sides proves that they do not
                const int v = tap0[(A - 1) * C], b0 = tap0[(A - 3) * C], b4 = tap0[(A + 1) * C];
                if (3 * max(b0, b4) <= 8 * v) {
                    sm.ring[slot0 + lr][col] = (uint8_t)v;
                    continue;
                }
            }
            const int xx = (obyte0 + col) / C;
            sm.ring[slot0 + lr][col] = exact_taps<TAPS>(tap0, C, [&](int k) { return p.wdx[(long long)xx * TAPS + k]; });
            n_strict++;
        }
    };

    // ------------------------------ V-pass state ------------------------------
    float acc[NSLOT][VB];
#pragma unroll
    for (int j = 0; j < NSLOT; j++)
#pragma unroll
        for (int i = 0; i < VB; i++) acc[j][i] = 0.f;
    const float guard_v = MODE == 0 ? p.guard : 0.f;
    const long long opitch = p.out_pitch;
    const uint8_t *vcol = &sm.ring[0][VB * lane];
    const int t0_first = (rs - A - G::S0) / D;                 // exact division (also for negative values)
    int ybase = N * t0_first;                                  // output row of bit 0 of `fixrows` for the current chunk
    uint8_t *ocol = out_frame + obyte0 + VB * lane + (long long)(ybase - p.out_row0) * opitch;

    auto v_pass = [&](int chunk) {
        const int bslot = (chunk % G::REGIONS) * RB;
        const uint8_t *vrow = vcol + bslot * SWB;
        const int wrapoff = (bslot == 0) ? G::RING * SWB : 0;
        const bool interior = (ybase >= ys) && (ybase + G::YROWS + N <= ye);
        uint32_t fixrows = 0;                                  // bit yy: look at output row ybase + yy again
        auto body = [&](auto check_tag) {
            constexpr bool CHECK = decltype(check_tag)::value;
            const uint8_t *vit = vrow;
            uint8_t *op = ocol + (long long)ylo<N, D>(G::S0) * opitch;   // next output row (rows come out in order)
            int yit = ybase;
#pragma unroll 1
            for (int it = 0; it < RB / G::U; it++) {
                uint32_t fl = 0;
#pragma unroll
                for (int u = 0; u < G::U; u++) {
                    const int s0 = (G::S0 + u) % D, tq = (G::S0 + u) / D;   // completing centre = D*(t + tq) + s0
                    const int cnt0 = cnt<N, D>(s0);
                    const uint32_t w = *reinterpret_cast<const uint32_t *>(vit + u * SWB);
                    float x[VB];
                    word_to_f32x4(w, x[0], x[1], x[2], x[3]);
                    // ---- systolic step: every pending output row takes its next tap from this row ----
                    float res[CNTMAX][VB];
                    {
                        int q = 0;
#pragma unroll
                        for (int dc = 0; dc < TAPS; dc++) {
                            const int sdc = (s0 + dc) % D;
                            const int k = TAPS - 1 - dc;
#pragma unroll
                            for (int yr = ylo<N, D>(sdc); yr < yhi<N, D>(sdc); yr++) {
                                const int ph = (yr * D) % N;
                                if (ph == 0) continue;
                                const float2 wk2 = make_float2(p.wtab[ph * 8 + k], p.wtab[ph * 8 + k]);
#pragma unroll
                                for (int i = 0; i < VB; i += 2) {
                                    const float2 x2 = make_float2(x[i], x[i + 1]);
                                    const float2 a2 = (dc < TAPS - 1) ? make_float2(acc[q][i], acc[q][i + 1]) : make_float2(-guard_v, -guard_v);
                                    const float2 r2 = __ffma2_rn(x2, wk2, a2);
                                    if (dc == 0) { res[q][i] = r2.x; res[q][i + 1] = r2.y; }
                                    else { acc[q - cnt0][i] = r2.x; acc[q - cnt0][i + 1] = r2.y; }
                                }
                                q++;
                            }
                        }
                    }
                    // ---- rows that received their last tap ----
                    {
                        int q = 0;
#pragma unroll
                        for (int yr = ylo<N, D>(s0); yr < yhi<N, D>(s0); yr++) {
                            const int ph = (yr * D) % N;
                            const int yoff = N * tq + yr;                 // output row relative to yit
                            uint32_t qv;
                            bool doubt = false;
                            if (ph == 0) {
                                // phase 0: start from the centre tap; the reference's value is that or one less, v_fix_dyn decides
                                auto ring_row = [&](int o) {              // ring row `o` rows from this iteration's first
                                    const uint8_t *r = vit + o * SWB;
                                    if (o < 0 && it * G::U + o < 0) r += wrapoff;
                                    return *reinterpret_cast<const uint32_t *>(r);
                                };
                                qv = ring_row(u - A);
                                doubt = true;
                                if (A == 3 && p.p0_filter) {
                                    // v - 0.375 b >= 0 for the rows 2 above and 2 below the centre, as in lanczos_v6.cu:
                                    // one fp16 FMA per test on the raw fp16-subnormal bytes, the sign is exact
                                    const uint32_t wa = ring_row(u - A - 2), wb = ring_row(u - A + 2);
                                    const uint32_t kR = 0xB600B600u;      // -0.375
                                    uint32_t z = 0;
#pragma unroll
                                    for (int hsel = 0; hsel < 2; hsel++) {
                                        const uint32_t sel = hsel ? 0x4342u : 0x4140u;
                                        const uint32_t hv = __byte_perm(qv, 0u, sel);
                                        z |= hfma2(__byte_perm(wa, 0u, sel), kR, hv) | hfma2(__byte_perm(wb, 0u, sel), kR, hv);
                                    }
                                    doubt = (z & 0x80008000u) != 0u;
                                }
                            } else {
                                qv = quantise4(res[q][0], res[q][1], res[q][2], res[q][3]);
                                if (MODE == 0) {
                                    const float g2v = 2.f * p.guard;
                                    doubt = qv != quantise4(res[q][0] + g2v, res[q][1] + g2v, res[q][2] + g2v, res[q][3] + g2v);
                                }
                                q++;
                            }
                            uint8_t *orow = op;
                            op += opitch;
                            if (CHECK && (yit + yoff < ys || yit + yoff >= ye)) continue;
                            if (MODE == 0 && doubt) fl |= 1u << yoff;
                            *reinterpret_cast<uint32_t *>(orow) = qv;
                        }
                    }
                }
                if (MODE == 0) fixrows |= fl << (it * (N * G::U / D));
                vit += G::U * SWB;
                yit += N * G::U / D;
            }
        };
        if (interior) body(std::false_type{}); else body(std::true_type{});
        if (MODE == 0 && fixrows) {
            VFixD a;
            a.col = vcol; a.ocol = ocol; a.opitch = opitch; a.ybase = ybase; a.rs = rs;
            a.nbytes = min(VB, valid_bytes - VB * lane);
            a.rows = fixrows;
            n_strict += v_fix_dyn<A, N, D, G::RING, SWB>(p, a);
        }
        ybase += G::YROWS;
        ocol += (long long)G::YROWS * opitch;
    };

    // ------------------------------ pipeline ------------------------------
    for (int chunk = 0; chunk < nchunks; chunk++) {
        h_pass(chunk);
        __syncwarp();
        if (lane == 0 && chunk + G::STAGES < nchunks) issue(chunk + G::STAGES);
        if (active) v_pass(chunk);
        __syncwarp();
    }
    if (p.strict_counter && n_strict) atomicAdd(p.strict_counter, (unsigned long long)n_strict);
}

template <int C, int A, int N, int D, int MODE>
int launch_dyn_one(const KParams &k, const FastHostTables &t, LaunchShape *shape, cudaStream_t s) {
    using G = GeoD<C, A, N, D>;
    const int row_bytes = k.out_w * C;
    const int strips = (row_bytes + G::SWB - 1) / G::SWB;
    // every strip's input must fit the staged row: check with the host copy of the tap table
    for (int sI = 0; sI < strips; sI++) {
        const int ob0 = sI * G::SWB, ob1 = std::min(row_bytes, ob0 + G::SWB) - 1;
        const int xb0 = ((t.i0x_host[ob0 / C] * C) >> 4) << 4;
        const int last = (t.i0x_host[ob1 / C] + 2 * A) * C;      // one past the last byte read
        if (last - xb0 > G::BOX_B) return -1;
    }
    CUtensorMap map;
    if (!encode_input_map(&map, k, G::BOX_B, G::RB)) return -1;
    auto kern = lanczos_dyn_kernel<C, A, N, D, MODE>;
    const size_t smem = sizeof(SmemD<G>) + 128;
    static std::atomic<int> ctas_per_sm[64] = {};
    const Residency res = resident_ctas(ctas_per_sm, kern, smem);
    if (res.ctas == 0) return -1;
    const int vperiod0 = k.out_row0 / N;
    const int vperiods = (k.out_row0 + k.out_rows + N - 1) / N - vperiod0;
    const SegPlan sp = plan_segments(vperiods, D, A, G::RB, (long long)strips * k.n_frames, res.ctas, 512);

    DynParams p{};
    set_strip_params(p, k, vperiod0, sp.seg_periods);
    p.i0x = k.i0x; p.wdx = k.wdx; p.wdy = k.wdy;
    p.guard = k.guard_asc;
    // the cheap phase-0 test needs: coordinates exactly integral in double on both axes (then the weights there are
    // the whole-pixel residues for every coordinate), a = 3 with negative residues exactly at +-2 pixels, K <= 3/8
    {
        int km = 0;
        bool small = true;
        for (int q = 0; q < 2 * A; q++) {
            if (t.align_k[q] != 0.f) km |= 1 << q;
            if (t.align_k[q] > 0.374f) small = false;
        }
        p.p0_filter = (A == 3 && km == 0x11 && small && t.exact_x && t.exact_y) ? 1 : 0;
    }
    fill_wtab(p.wtab, t, A, N);
    p.strict_counter = k.strict_counter;

    dim3 grid(strips, sp.segs, k.n_frames);
    *shape = LaunchShape{(int)grid.x, (int)grid.y, (int)grid.z, sp.seg_periods, G::RB, res.ctas};
    kern<<<grid, 32, smem, s>>>(map, p);
    return (int)cudaGetLastError();
}

}  // namespace

// Returns 0 on launch, >0 cudaError, -1 when no instance applies (caller falls back to the generic kernel).
// The instances are split over two translation units (lanczos_dyn.cu: LZD_PART 0, lanczos_dyn2.cu: LZD_PART 1)
// so that they compile in parallel.
#ifndef LZD_PART
#define LZD_PART 0
#endif
#if LZD_PART == 0
int launch_dyn_part1(const KParams &k, const FastHostTables &t, int *kernel_id, LaunchShape *shape, cudaStream_t s);
int launch_dyn(const KParams &k, const FastHostTables &t, int *kernel_id, LaunchShape *shape, cudaStream_t s) {
#else
int launch_dyn_part1(const KParams &k, const FastHostTables &t, int *kernel_id, LaunchShape *shape, cudaStream_t s) {
#endif
    if (!strip_layout_ok(k) || !t.i0x_host) return -1;
    const int mode = (k.flags & LANCZOS_FLAG_TOLERANCE_1LSB) ? 1 : 0;
    const int C = k.channels, A = k.a, N = k.scale_n, D = k.scale_d;
#define LZD_CASE(c, a, n, d, id)                                                   \
    if (C == c && A == a && N == n && D == d) {                                     \
        *kernel_id = id;                                                            \
        return mode == 0 ? launch_dyn_one<c, a, n, d, 0>(k, t, shape, s) : launch_dyn_one<c, a, n, d, 1>(k, t, shape, s); \
    }
#if LZD_PART == 0
    LZD_CASE(3, 3, 17, 10, 5)
    LZD_CASE(3, 3, 3, 2, 6)
    LZD_CASE(3, 3, 3, 1, 7)
    LZD_CASE(1, 3, 17, 10, 11)
    // the reference author's own sample configuration (lanczos.h:13-28: 162x89 -> 486x267, 3x, LANCZOS_A 2): interleaved
    // RGB, and one-channel planes (the layout of lanczos_expected itself, through lanczos_b200_upscale_planar / _expected)
    LZD_CASE(3, 2, 3, 1, 12)
    LZD_CASE(1, 2, 3, 1, 13)
    LZD_CASE(3, 3, 4, 1, 14)
    LZD_CASE(1, 3, 3, 1, 15)
    return launch_dyn_part1(k, t, kernel_id, shape, s);
#else
    LZD_CASE(3, 3, 5, 3, 16)
    LZD_CASE(3, 3, 7, 4, 17)
    LZD_CASE(2, 3, 2, 1, 18)
    LZD_CASE(3, 4, 2, 1, 19)
    LZD_CASE(3, 1, 2, 1, 20)
    LZD_CASE(4, 3, 3, 1, 21)
    LZD_CASE(4, 3, 4, 1, 22)
    LZD_CASE(3, 2, 3, 2, 23)
    LZD_CASE(1, 3, 4, 1, 24)
    return -1;
#endif
#undef LZD_CASE
}

}  // namespace lzb
