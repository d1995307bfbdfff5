// lanczos_v6.cu -- specialised fused H->V Lanczos kernels for sm_100a, second generation.
//
// What it replaces in the reference (software-path arithmetic, HLS-path structure):
//   cyclic_buffer/cyclic_buffer.h:4-69  2a(+1)-line cyclic buffer   -> shared-memory ring of H-pass rows
//   worker.cpp:138-155 ColWorkers::exec (vertical MAC per column)    -> systolic V pass: 2a-1 partial sums per
//                                                                       column in registers, one FFMA each per row
//   worker.cpp:225-247 RowWorkers::exec (horizontal MAC)             -> H pass on TMA-staged rows
//   lanczos.cpp:68-83  process_channel block loop (DATAFLOW)          -> chunk loop: H(c+1) overlaps V(c) through
//                                                                       mbarriers, no CTA-wide barrier
//   kernel.cpp:40-58   coefficient LUT                                -> polyphase table in the constant bank
//   full_TB.h:55-77    the arithmetic that must be matched bit for bit
//
// One CTA = one strip of <= VB*NT output byte-columns x one vertical segment, streamed in chunks of RB input rows.
//   1. TMA (cp.async.bulk.tensor 3-D: x, y, frame; out-of-bounds = 0 = the reference's dropped taps) stages
//      RB input rows + halo bytes into shared memory, double buffered on mbarriers.
//   2. H pass (one item per thread and chunk): PH ratio periods of one row.  8-byte conflict-free LDS, bytes ->
//      fp32 via PRMT + FHADD (fp16-subnormal trick), 2a-tap FFMA chains with constant-bank weights for the
//      interpolated samples only, smallest weights first (tighter rounding bound).  Phase-0 samples (copies)
//      never pass through fp32: PRMT splices the raw input bytes next to the F2IP-quantised interpolated
//      bytes; 16-byte STS into the ring.
//   3. V pass, systolic: a thread owns VB byte-columns.  Per new ring row: one LDS.64, bytes -> fp32, then every
//      pending output row of the column takes its next tap (acc[j-1] = fma(x, w, acc[j]): the FFMA's
//      destination does the window shift, so the loop body is one ratio period and the code stays small enough
//      for the instruction cache); the row that received its last tap is quantised and stored (STG.64).
//      The phase-0 "cannot flip" test runs on the fp16x2 pipe with exact small-integer arithmetic
//      (8*v - 3*b[+-2] >= 0 per side, a conservative form of plan.cpp's filter).
// Exactness: sums start at -guard; a sample whose truncation differs between x-guard and x+guard is
// recomputed with the reference's double arithmetic (full_TB.h:58-63) by the thread that found it.
// Phase-0 samples (output coordinate on an input sample: the reference returns the centre value v or v - 1) are
// copies of v where the cheap filter proves that, and are otherwise decided by an EXACT fp32 restatement of the
// reference's double sum (phase0_chain2; proved by enumeration in plan.cpp verify_phase0_chain): in line in the H
// pass (the converted bytes are in registers), once per chunk and out of line in the V pass (v_fix_phase0_chunk).
// MODE 1 (LANCZOS_FLAG_TOLERANCE_1LSB): the V pass is plain fp32 (no guard, no phase-0 test); the H pass
// stays exact, so every output byte is within 1 LSB of the reference.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <type_traits>
#include <cuda.h>

#include "../../include/lanczos_b200.h"
#include "fast_common.cuh"

namespace lzb {

namespace {

// strict_counter leads so that every other field keeps the constant-bank offset mod 16 of the layout the kernel was
// tuned with: with other orders ptxas gave some instances one register and a few instructions more or less.
struct V6Params : StripParams {
    unsigned long long *strict_counter;
    const double *wdx, *wdy;  // per-coordinate double weights (exact recomputation, non-uniform phases)
    float guard_h, guard_v;   // rigorous fp32 error bounds (x1.05) of the two summation orders
    int uniform_x, uniform_y; // double weights identical for all coordinates of a phase -> wdtab usable
    int strict_v_identity;    // 0 with LANCZOS_FLAG_FAST_ALIGNED
    int independent;          // LANCZOS_FLAG_INDEPENDENT: launched with programmatic dependent launch, no wait for the previous kernel
    int alias_rows, alias_top_row;   // in-place top rows done inside this kernel (0 = none / separate kernel)
    float align_k[8];         // phase-0 "cannot flip" constants
    // phase-0 second look (a = 3): the reference's double sum restated exactly in fp32 (plan.cpp verify_phase0_chain):
    // {W0, W1, 1, W3, W4} times 2^24 (the kernels' pixel values carry 2^-24), W_k = fl32(w_k * 2^29)
    float p0c[5];
    float wtab[32 * 8];       // polyphase table [N][8] (padded to 8 taps), N <= 32, times 2^24
    double wdtab[8 * 8];      // double polyphase table [N][8] for N <= 8 (valid when uniform_*)
};

__host__ __device__ constexpr int cmax6(int a, int b) { return a > b ? a : b; }
__host__ __device__ constexpr int gcd6(int a, int b) { return b == 0 ? a : gcd6(b, a % b); }

template <int C, int A, int N, int D, int PH, int MODE>
struct Geo6 {
    static constexpr int VB = 8;                        // byte-columns per V thread
    static constexpr int TAPS = 2 * A;
    static constexpr int IN_B = PH * D * C;             // input bytes owned by one H item
    static constexpr int OUT_B = PH * N * C;            // output bytes produced by one H item
    static constexpr int NI = PH * (N - 1) * C;         // interpolated (phase != 0) samples per H item
    static constexpr int ND = (NI + 3) / 4;             // ... packed 4 per word
    static constexpr int HALO_L = (A - 1) * C;
    static constexpr int B_LAST = ((N - 1) * D) / N;
    static constexpr int HALO_R = cmax6(0, (B_LAST + A + 1 - D) * C);
    static constexpr int PAD_L = 16 * ((HALO_L + 15) / 16);       // TMA box starts PAD_L bytes left of the strip
    static constexpr int WIN_B = HALO_L + IN_B + HALO_R;          // bytes one H item reads
    static constexpr int MIS = (PAD_L - HALO_L) % 8;              // window start inside its first 8-byte unit
    static constexpr int WIN0 = PAD_L - HALO_L - MIS;             // first 8-byte unit (byte offset) of group 0
    static constexpr int NW2 = (MIS + WIN_B + 7) / 8;             // 8-byte loads per H item
    // A warp's strip is SWV = 256 output bytes wide and starts at a multiple of 256: every row piece the V pass
    // stores is two whole 128-byte lines.  (Strips of 5 H items = 240 bytes left every other 32-byte sector and
    // every 128-byte line shared between two warps: tools/wbench.cu measures 4.0 TB/s for that store pattern on
    // this part against 6.8 TB/s for 256-byte pieces, and the V pass alone was bound by it.)  H items are OUT_B
    // bytes wide and aligned to OUT_B, so the H pass of a strip covers the MAX_GROUPS items that contain it.
    // MODE 1 (plain fp32 V pass) is short of H-pass time, not of store bandwidth: five whole H items, no overlap
    // (+7 % on uniform noise in that mode, measured; +-0 on image-like content)
    static constexpr int SWV = (MODE == 1) ? 5 * OUT_B : 32 * VB;
    static constexpr int VOFF_MAX = OUT_B - gcd6(SWV, OUT_B);     // largest offset of a strip inside its first H item
    static constexpr int MAX_GROUPS = cdiv(VOFF_MAX + SWV, OUT_B);   // H items per row of a warp's strip (6 for 48-byte items)
    static constexpr int SW_MAX = MAX_GROUPS * OUT_B;             // ring pitch in bytes (288)
    // a TMA box must start on a 16-byte boundary of the row: strips whose input starts 8 bytes off get a box
    // that starts 8 bytes early (XSHIFT_MAX extra bytes per row)
    static constexpr int XSHIFT_MAX = (IN_B % 16 != 0) ? 8 : 0;   // H items start at multiples of IN_B input bytes
    static constexpr int BOX_B = 16 * cdiv(XSHIFT_MAX + cmax6(PAD_L + MAX_GROUPS * IN_B + HALO_R, WIN0 + (MAX_GROUPS - 1) * IN_B + 8 * NW2), 16);
    static constexpr int HB = 32 / MAX_GROUPS;                    // rows one round of H items covers (one item per lane)
    static constexpr int HROUNDS = 2;                             // H rounds per chunk
    static constexpr int RB = HB * HROUNDS;                       // input rows per chunk
    static constexpr int REGIONS = 2;                             // ring regions of RB rows: V(c) reads region c and the tail of c-1
    static constexpr int RING = REGIONS * RB;                     // intermediate rows kept in smem
    static constexpr int STAGE_B = 128 * ((RB * BOX_B + 127) / 128);  // TMA destinations must be 128-byte aligned
    static constexpr int STAGES = 3;                              // TMA stages in flight
    // the first row pushed by a segment is rs = D*pv0 - A + 1, so (row - A) mod D is static per chunk row
    static constexpr int S0 = (((1 - 2 * A) % D) + D) % D;
    static constexpr int U = lcm2(D);                             // rows per V loop iteration (even: filter delay line parity)
    static constexpr int YROWS = N * RB / D;                      // output rows completed per chunk
    static_assert(IN_B % 8 == 0, "H item input must be 8-byte aligned");
    static_assert(OUT_B % 16 == 0, "H item output must be 16-byte aligned");
    static_assert(OUT_B % VB == 0 && HB * MAX_GROUPS <= 32 && HB >= 1, "one H item per lane and round, one V column per lane");
    static_assert(RB % U == 0, "chunk must be a whole number of V loop iterations");
    static_assert(TAPS - 1 <= RB, "tap rows must not reach further back than one ring region");
    static_assert(BOX_B / 4 <= 256, "TMA box too wide");
    static_assert(N <= 32, "phase table too large for kernel params");
    static_assert(YROWS + N * (S0 + A + 1) / D + 2 <= 64, "fix mask (bit per output row) too small");
    static_assert(cdiv(S0 * N, D) + YROWS <= 32, "rows fixed per chunk must fit 32 bits");
    static_assert(ND <= 31, "H fix mask (bit per packed word) too small");
    static_assert(D <= 2, "phase-0 filter delay line assumes the +-2 rows are phase-0 centres themselves");
};

template <class G>
struct __align__(128) Smem6 {             // one per CTA
    uint8_t in[G::STAGES][G::STAGE_B];    // TMA destinations, row lr at lr * BOX_B
    uint8_t ring[G::RING][G::SW_MAX];     // H-pass results (uint8), row r lives in slot (r - rs) % RING
    unsigned long long full[G::STAGES];   // TMA stage filled
};

// Four bytes from up to four source words, positions known at compile time after unrolling: one PRMT for
// the first two distinct sources, one more per further source.
template <int NSRC>
__device__ __forceinline__ uint32_t gather4(const uint32_t (&arr)[NSRC], const int (&id)[4], const int (&bp)[4]) {
    uint32_t res = 0;
    bool started = false;
    int done = 0;
#pragma unroll
    for (int u = 0; u < 4; u++) {
        if ((done >> u) & 1) continue;
        const int ida = id[u];
        if (!started) {
            int idb = -1;
#pragma unroll
            for (int v = 0; v < 4; v++)
                if (v > u && id[v] != ida && idb < 0) idb = id[v];
            uint32_t sel = 0;
#pragma unroll
            for (int v = 0; v < 4; v++) {
                if (id[v] == ida) { sel |= (uint32_t)bp[v] << (4 * v); done |= 1 << v; }
                else if (idb >= 0 && id[v] == idb) { sel |= (uint32_t)(4 + bp[v]) << (4 * v); done |= 1 << v; }
            }
            res = __byte_perm(arr[ida], idb >= 0 ? arr[idb] : 0u, sel);
            started = true;
        } else {
            uint32_t sel = 0;
#pragma unroll
            for (int v = 0; v < 4; v++) {
                if (id[v] == ida) { sel |= (uint32_t)(4 + bp[v]) << (4 * v); done |= 1 << v; }
                else sel |= (uint32_t)v << (4 * v);
            }
            res = __byte_perm(res, arr[ida], sel);
        }
    }
    return res;
}

// double_to_uint8 (full_TB.h:29-37) on one fp32 value, as F2IP does it: clamp to [0,255], truncate toward zero
__device__ __forceinline__ uint32_t quantise_f32(float x) {
    const int i = __float2int_rz(x);
    return (uint32_t)min(max(i, 0), 255);
}

// summation order of the H-pass chains: outermost (smallest) weights first, the two central taps last
template <int TAPS> __host__ __device__ constexpr int tap_order6(int i) { return (i & 1) ? TAPS - 1 - i / 2 : i / 2; }

// Phase-0 second look (a = 3): the reference's double sum b0*w0 + b1*w1 + v + b3*w3 + b4*w4 (full_TB.h:58-63 /
// :71-75 at a coordinate that falls on an input sample; ascending taps, tap 5 never changes it) restated in fp32.
// The grid of floats around the integer v is the grid of doubles scaled by 2^29, so the sum with residues scaled by
// 2^29 rounds the way the reference's does at every step; plan.cpp verify_phase0_chain enumerates every reachable
// state of the sum to prove that the fp32 rounding of the scaled residues never changes a decision (kernels with a
// phase-0 test are not launched otherwise).  x[k] = the five bytes * 2^-24 (two samples), pc = V6Params.p0c.
// The truncation of the result is the reference's output: v, or v - 1 when the negative residues win.
__device__ __forceinline__ float2 phase0_chain2(const float2 (&x)[5], const float *pc) {
    float2 s = __fmul2_rn(x[0], make_float2(pc[0], pc[0]));
#pragma unroll
    for (int k = 1; k < 5; k++) s = __ffma2_rn(x[k], make_float2(pc[k], pc[k]), s);
    return s;
}
__device__ __forceinline__ float phase0_chain1(const float (&x)[5], const float *pc) {
    float s = __fmul_rn(x[0], pc[0]);
#pragma unroll
    for (int k = 1; k < 5; k++) s = __fmaf_rn(x[k], pc[k], s);
    return s;
}

// Shared-memory loads by 32-bit shared address: the slow paths are out of line, where a generic pointer
// would turn every access into a generic LD.
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}

// ---------------------------------------------------------------------------------------------
// slow paths: executed by the thread that found a sample in doubt, kept out of line so that the hot loop
// stays small.  Both restate full_TB.h:58-63 / :71-75 exactly (exact_taps).
// ---------------------------------------------------------------------------------------------
struct HFixArgs {
    const uint8_t *in_row;    // staged input row of the item (byte 0 = ibyte0 - PAD_L)
    uint8_t *ring_row;        // ring row of the item
    int gbyte0;               // strip-relative output byte of the item's first byte
    int obyte0, ibyte0, valid_bytes;
    uint32_t fix_g;           // bit per packed word of interpolated samples
    float guard;
};

template <class G, int C, int A, int N, int D, int PH>
__device__ __noinline__ int h_fix(const V6Params &p, const HFixArgs a) {
    constexpr int TAPS = 2 * A;
    constexpr int NI = PH * (N - 1) * C;
    constexpr int PAD_L = G::PAD_L;
    int n_strict = 0;
    auto fix_byte = [&](int b) {
        if (a.gbyte0 + b >= a.valid_bytes) return;
        const int ob = a.obyte0 + a.gbyte0 + b;                  // global output byte column
        const int xx = ob / C, c = ob - xx * C;
        const int first = (xx * D) / N - A + 1;                  // first tap pixel (full_TB.h:59)
        const int ph = (xx * D) % N;
        const uint8_t *tap0 = a.in_row + PAD_L + first * C + c - a.ibyte0;
        // the hot path's fp32 chain again (same order, same weights: same bits): only a sample whose
        // truncation really is in doubt needs the double evaluation
        float acc = -a.guard;
#pragma unroll
        for (int i = 0; i < TAPS; i++) {
            const int k = tap_order6<TAPS>(i);
            acc = fmaf((float)tap0[k * C] * (1.f / 16777216.f), p.wtab[ph * 8 + k], acc);
        }
        if (quantise_f32(acc) == quantise_f32(acc + 2.f * a.guard)) return;
        uint8_t r;
        if (p.uniform_x && N <= 8) r = exact_taps<TAPS>(tap0, C, [&](int k) { return p.wdtab[ph * 8 + k]; });
        else r = exact_taps<TAPS>(tap0, C, [&](int k) { return p.wdx[(long long)xx * TAPS + k]; });
        a.ring_row[b] = r;
        n_strict++;
    };
#pragma unroll 1
    for (uint32_t m = a.fix_g; m; m &= m - 1) {
        const int dw = __ffs(m) - 1;
#pragma unroll 1
        for (int e = 0; e < 4; e++) {
            const int s = 4 * dw + e;
            if (s >= NI) break;
            const int per = s / ((N - 1) * C), rem = s - per * ((N - 1) * C);
            fix_byte((per * N + 1) * C + rem);
        }
    }
    return n_strict;
}

// bit 0 of byte e (e = 0..3) -> bit e
__device__ __forceinline__ uint32_t lsb4_to_bits(uint32_t x) {
    return (((x & 0x01010101u) * 0x01020408u) >> 24) & 0xfu;
}

// full_TB.h:71-75 for byte `col_e` of one output row: NT taps from consecutive ring rows starting at slot0
template <int NT, int RING, int SWM, class W>
__device__ __forceinline__ uint32_t exact_ring(uint32_t col_e, int slot0, W weight) {
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < NT; k++) {
        int sl = slot0 + k;
        if (sl >= RING) sl -= RING;
        const double v = __hiloint2double(0x43300000, (int)lds_u8(col_e + sl * SWM)) - 4503599627370496.0;
        sum = __dadd_rn(sum, __dmul_rn(v, weight(k)));
    }
    return quantise_f64(sum);
}

// ---- V-pass slow path: one call per loop iteration in which some lane found something -------------------
// The hot loop stores every row as it comes out of the fp32 pipeline and only collects, per row, what says
// "look again": for an interpolated row the XOR of its two truncations (x - guard, x + guard; a byte in doubt
// differs by one, so bit 0 of the byte is set), for a phase-0 row (copy of a centre row) the sign bits of the
// fp16x2 "cannot flip" tests.  v_fix_iter then re-reads the row it stored, replaces the bytes in question by what
// the reference's double arithmetic gives (full_TB.h:71-75), and stores it again (same lane, program order).
template <int A, int N, int D, int VU, int S0> __host__ __device__ constexpr int viter_interp_rows() {
    int n = 0;
    for (int u = 0; u < VU; u++) n += cnt<N, D>((S0 + u) % D);
    return n;
}
template <int A, int N, int D, int VU, int S0> __host__ __device__ constexpr int viter_centre_rows() {
    int n = 0;
    for (int u = 0; u < VU; u++) n += ((S0 + u + A) % D == 0) ? 1 : 0;
    return n;
}
template <int NI>
struct VIterFlags {
    uint32_t dx[NI > 0 ? NI : 1], dy[NI > 0 ? NI : 1];   // interpolated rows of the iteration, in the order they complete
};

// bytes of an interpolated row: NT = 2a taps from ring slots slot0 .. (ascending rows = ascending taps)
template <int A, int N, int D, int RING, int SWM>
__device__ __forceinline__ int fix_interp_bytes(const V6Params &p, uint32_t col, int slot_r, int y, uint32_t need, uint2 &q) {
    constexpr int TAPS = 2 * A;
    const int ph = (y * D) % N;
    int slot0 = slot_r - (TAPS - 1);
    if (slot0 < 0) slot0 += RING;
    int n = 0;
#pragma unroll 1
    for (; need; need &= need - 1) {
        const int e = __ffs(need) - 1;
        uint32_t v;
        if (p.uniform_y && N <= 8) v = exact_ring<TAPS, RING, SWM>(col + e, slot0, [&](int k) { return p.wdtab[ph * 8 + k]; });
        else v = exact_ring<TAPS, RING, SWM>(col + e, slot0, [&](int k) { return p.wdy[(long long)y * TAPS + k]; });
        const int sh = 8 * (e & 3);
        if (e < 4) q.x = (q.x & ~(0xffu << sh)) | (v << sh);
        else q.y = (q.y & ~(0xffu << sh)) | (v << sh);
        n++;
    }
    return n;
}

// Phase-0 second look of the V pass, once per chunk: when the hot filter flagged any phase-0 row of the chunk, ALL of
// them are redone with the exact fp32 chain (phase0_chain2's arithmetic: the reference's double sum restated, v or
// v - 1) and stored again.  The centres that complete in chunk rows 0 .. RB-1 use ring rows -4 .. RB-1 (a row goes
// out when row c + 2 has arrived; the tail of the previous ring region is still there; rows before the segment's
// first belong to output rows outside [ys, ye), which are skipped).  Every ring row is loaded once per pass and feeds
// the sums of the up to five centres it is a tap of.
//   * four byte-columns per pass, passes not unrolled: the caller's partial sums stay in registers across this call,
//     so whatever this function needs beyond ~30 registers is spilled around it -- and ptxas then also spills inside
//     the hot loop (measured: +4 % on image-like content with six converted rows of 4 columns held at once);
//   * a byte loaded with LDS.U8 is, read as fp32, the denormal b * 2^-149, and FFMA takes denormal operands at full
//     rate: with the constants times 2^101 the chain runs on b * 2^-24 like the hot path's values (every intermediate
//     a normal number: the same roundings), then one exact multiplication by 2^24.
// col: shared address of the lane's column in ring row 0; bslot: ring slot of the chunk's first row; ocol: the lane's
// column in output row ybase (the row the period of the chunk's first iteration starts at).
template <int A, int N, int D, int S0, int RB, int RING, int SWM>
__device__ __noinline__ void v_fix_phase0_chunk(const V6Params &p, uint32_t col, int bslot, int ybase, uint8_t *ocol, long long opitch,
                                                int nbytes, int ys, int ye) {
    static_assert(A == 3, "written for the +-2 residues of a = 3");
    float kd[5];
#pragma unroll
    for (int k = 0; k < 5; k++) kd[k] = p.p0c[k] * 2.535301200456459e30f;       // 2^101, exact
    // rows -4 .. -1 are the last four of the other ring region (REGIONS = 2: bslot is 0 or RB)
    const uint32_t a_prev = col + (bslot == 0 ? RING - 4 : bslot - 4) * SWM + 4 * SWM, a_cur = col + bslot * SWM;
    auto pass = [&](auto all_tag) {
        constexpr bool ALL = decltype(all_tag)::value;      // every row of the chunk lies inside [ys, ye): no row tests
#pragma unroll 1
        for (int half = 0; half < 2; half++) {
            if (4 * half >= nbytes) break;
            float2 sum[RB][2];                   // sums of the centre that completes at chunk row j (alive for five rows)
            uint8_t *orow = ocol + 4 * half;
            int yprev = 0;
#pragma unroll
            for (int jj = -4; jj < RB; jj++) {
                bool used = false;
#pragma unroll
                for (int j = 0; j < RB; j++)
                    if ((S0 + j + A) % D == 0 && jj >= j - 4 && jj <= j) used = true;
                if (!used) continue;
                const uint32_t a = (jj < 0 ? a_prev : a_cur) + 4 * half + jj * SWM;
                const float2 xa = make_float2(__uint_as_float(lds_u8(a)), __uint_as_float(lds_u8(a + 1)));
                const float2 xb = make_float2(__uint_as_float(lds_u8(a + 2)), __uint_as_float(lds_u8(a + 3)));
#pragma unroll
                for (int j = 0; j < RB; j++) {
                    if ((S0 + j + A) % D != 0) continue;
                    const int k = jj - (j - 4);
                    if (k < 0 || k > 4) continue;
                    const float2 kk = make_float2(kd[k], kd[k]);
                    if (k == 0) { sum[j][0] = __fmul2_rn(xa, kk); sum[j][1] = __fmul2_rn(xb, kk); }
                    else { sum[j][0] = __ffma2_rn(xa, kk, sum[j][0]); sum[j][1] = __ffma2_rn(xb, kk, sum[j][1]); }
                    if (k == 4) {
                        const int yoff = N * ((S0 + j + A - 2) / D);
                        orow += (long long)(yoff - yprev) * opitch;
                        yprev = yoff;
                        const float2 u2 = make_float2(16777216.f, 16777216.f);
                        const float2 ra = __fmul2_rn(sum[j][0], u2), rb = __fmul2_rn(sum[j][1], u2);
                        const uint32_t q = quantise4(ra.x, ra.y, rb.x, rb.y);
                        // rows outside [ys, ye) (warm-up rows, rows of the next segment) are skipped
                        if (ALL || (ybase + yoff >= ys && ybase + yoff < ye)) *reinterpret_cast<uint32_t *>(orow) = q;
                    }
                }
            }
        }
    };
    if ((ybase >= ys) && (ybase + N * ((S0 + RB - 1 + A - 2) / D) < ye)) pass(std::true_type{}); else pass(std::false_type{});
}

// col: shared address of the lane's column in ring row 0; slot_it: ring slot of the iteration's first row; yit / op:
// output row the iteration's period starts at and the lane's column in that row.  Returns the number of samples
// evaluated in double.
template <int A, int N, int D, int VU, int S0, int RING, int SWM, bool ST64>
__device__ __noinline__ int v_fix_iter(const V6Params &p, uint32_t col, int slot_it, int yit, uint8_t *op, long long opitch,
                                       const VIterFlags<viter_interp_rows<A, N, D, VU, S0>()> f, int nbytes, int ys, int ye) {
    const uint32_t vmask = nbytes >= 8 ? 0xffu : ((1u << nbytes) - 1u);
    int n = 0, qi = 0;
    auto redo = [&](int yoff, auto fix) {
        const int y = yit + yoff;
        if (y < ys || y >= ye) return;                     // never stored (warm-up rows, rows of the next segment)
        uint8_t *orow = op + (long long)yoff * opitch;
        uint2 q;
        if (ST64) q = *reinterpret_cast<const uint2 *>(orow);
        else { q.x = *reinterpret_cast<const uint32_t *>(orow); q.y = nbytes > 4 ? *reinterpret_cast<const uint32_t *>(orow + 4) : 0u; }
        n += fix(y, q);
        if (ST64) *reinterpret_cast<uint2 *>(orow) = q;
        else { *reinterpret_cast<uint32_t *>(orow) = q.x; if (nbytes > 4) *reinterpret_cast<uint32_t *>(orow + 4) = q.y; }
    };
#pragma unroll
    for (int u = 0; u < VU; u++) {
        const int s0 = (S0 + u) % D, tq = (S0 + u) / D;
#pragma unroll
        for (int yr = ylo<N, D>(s0); yr < yhi<N, D>(s0); yr++) {
            if ((yr * D) % N == 0) continue;
            if ((f.dx[qi] | f.dy[qi]) != 0u) {
                const uint32_t need = (lsb4_to_bits(f.dx[qi]) | (lsb4_to_bits(f.dy[qi]) << 4)) & vmask;
                redo(N * tq + yr, [&](int y, uint2 &q) { return fix_interp_bytes<A, N, D, RING, SWM>(p, col, slot_it + u, y, need, q); });
            }
            qi++;
        }
    }
    return n;
}

// The reference's column pass runs in place from the bottom row up (full_TB.h:67-77): output row yy reads rows
// first..last of the same plane, and every row i > yy of that window already holds its FINAL value.  Only the
// first alias_rows rows are affected.  After chunk 1 the ring still holds the (bit-exact) horizontal results of
// rows 0..2*RB-A, so the warp that owns the strip replays the recurrence for its columns in double arithmetic.
struct AliasArgs {
    const uint8_t *col;       // this thread's column in ring row 0 (slot of intermediate row rs)
    uint8_t *ocol;            // this thread's column in output row 0
    long long opitch;
    int rs, nbytes;
};

template <int A, int N, int D, int RB, int SWM, int VB>
__device__ __noinline__ void alias_fix(const V6Params &p, const AliasArgs a) {
    constexpr int TAPS = 2 * A;
    constexpr int TOP = (2 * RB - A) < 12 ? (2 * RB - A) : 12;   // last intermediate row used (the ring holds -(A-1) .. 2*RB-A after chunk 1)
    static_assert(VB == 8 && TOP - 1 < 16, "alias_fix handles one 8-byte column, rows 0..15");
    // the segment starts at output row 0, so intermediate row i sits in ring slot i + A - 1 (rs = -(A-1)).
    // Rows outside the image hold zeros (TMA fill), which add +-0 to the sum exactly like the reference's
    // clipped window (full_TB.h:72).
    uint2 fin[TOP + 1];                             // final values of rows already replaced
#pragma unroll
    for (int i = 0; i <= TOP; i++) fin[i] = make_uint2(0u, 0u);
#pragma unroll
    for (int yy = TOP - 1; yy >= 0; yy--) {
        if (yy > p.alias_top_row) continue;
        const int first = (yy * D) / N - A + 1;
        const int ph = (yy * D) % N;
        double sum[VB];
#pragma unroll
        for (int e = 0; e < VB; e++) sum[e] = 0.0;
#pragma unroll
        for (int k = 0; k < TAPS; k++) {
            const int i = first + k;
            if (i > TOP) continue;                  // cannot happen for rows the host lets this path handle
            const uint2 v = (i > yy) ? fin[i] : *reinterpret_cast<const uint2 *>(a.col + (i + A - 1) * SWM);
            const double w = (p.uniform_y && N <= 8) ? p.wdtab[ph * 8 + k] : p.wdy[(long long)yy * TAPS + k];
#pragma unroll
            for (int e = 0; e < VB; e++) {
                const uint32_t word = e < 4 ? v.x : v.y;
                const double vd = __hiloint2double(0x43300000, (int)((word >> (8 * (e & 3))) & 0xffu)) - 4503599627370496.0;
                sum[e] = __dadd_rn(sum[e], __dmul_rn(vd, w));
            }
        }
        uint32_t q[VB];
#pragma unroll
        for (int e = 0; e < VB; e++) q[e] = quantise_f64(sum[e]);
        fin[yy] = make_uint2(q[0] | (q[1] << 8) | (q[2] << 16) | (q[3] << 24), q[4] | (q[5] << 8) | (q[6] << 16) | (q[7] << 24));
        if (yy < p.alias_rows) {
            uint8_t *orow = a.ocol + (long long)yy * a.opitch;
#pragma unroll
            for (int e = 0; e < VB; e++)
                if (e < a.nbytes) orow[e] = (uint8_t)q[e];
        }
    }
}

// one warp per CTA, 16 resident per SM: the register allocation aims for 128 per thread
template <int C, int A, int N, int D, int PH, int KM, int MODE, bool ST64>
__global__ void __launch_bounds__(32, 16)
lanczos_v6_kernel(const __grid_constant__ CUtensorMap in_map, const __grid_constant__ V6Params p) {
    using G = Geo6<C, A, N, D, PH, MODE>;
    constexpr int TAPS = G::TAPS;
    constexpr int SWM = G::SW_MAX;
    constexpr int VB = G::VB;
    constexpr int CEN = A - 1;                                  // centre tap of a phase-0 sample
    constexpr int NSLOT = nslot<N, D, TAPS>();
    constexpr int CNTMAX = cntmax<N, D>();
#ifdef LZB_ABL_NOVFILTER     // ablation builds (timing experiments only, results are wrong): see tools/ablate.sh
    constexpr bool FILTER = false;
#else
    constexpr bool FILTER = (MODE == 0) && (KM != 0);
#endif
    // input rows per V loop iteration: one (even) ratio period (two in MODE 1 at D = 1 measured +2 % on 1080p, -5 % on 4K)
    constexpr int VU = G::U;
    static_assert(KM == 0 || (A == 3 && KM == 0x11), "phase-0 row filter is written for the +-2 residues of a = 3");
    extern __shared__ __align__(128) uint8_t smem_raw[];
    Smem6<G> &sm = *reinterpret_cast<Smem6<G> *>(smem_raw);
    const int tid = threadIdx.x;
    const int strip = blockIdx.x, seg = blockIdx.y, frame = blockIdx.z;
    // programmatic dependent launch: let the next kernel of the stream start as soon as SMs free up; unless the caller
    // declared the frames independent, wait here until everything before this kernel on the stream has completed
    // (both are no-ops for a launch without the attribute)
    asm volatile("griddepcontrol.launch_dependents;");
    if (!p.independent) asm volatile("griddepcontrol.wait;" ::: "memory");
    if (strip * G::SWV >= p.out_w * C) return;
    uint8_t *out_frame = p.out + (long long)frame * p.out_frame_stride;

    // horizontal extent
    const int vbyte0 = strip * G::SWV;                        // first output byte column of the strip (V pass, stores)
    const int row_bytes = p.out_w * C;
    const int valid_bytes = min(G::SWV, row_bytes - vbyte0);  // > 0 by construction of the grid
    const int obyte0 = (vbyte0 / G::OUT_B) * G::OUT_B;        // first output byte column of the H items that cover it
    const int voff = vbyte0 - obyte0;                         // 0, 16 or 32 for 48-byte items
    const int groups = min(G::MAX_GROUPS, (voff + valid_bytes + G::OUT_B - 1) / G::OUT_B);
    const int hvalid = min(groups * G::OUT_B, row_bytes - obyte0);   // bytes of the H items inside the image
    const int ibyte0 = (obyte0 / (N * C)) * (D * C);          // first input byte column of the H items
    const int xshift = (ibyte0 - G::PAD_L) & 15;              // 0 or 8: the TMA box starts that many bytes early
    // vertical extent: periods [pv0, pv1) -> output rows [N*pv0, N*pv1), clipped to the band
    const int pv0 = p.vperiod0 + seg * p.seg_periods;
    const int y_end_band = p.out_row0 + p.out_rows;
    const int pv1 = min(pv0 + p.seg_periods, (y_end_band + N - 1) / N);
    const int ys = max(N * pv0, p.out_row0), ye = min(N * pv1, y_end_band);
    if (ys >= ye) return;
    const int rs = D * pv0 - A + 1;                           // first intermediate row pushed
    const int nrows = D * (pv1 - pv0) + TAPS - 1;             // rows to push
    const int nchunks = (nrows + G::RB - 1) / G::RB;

    uint32_t full0 = smem_u32(&sm.full[0]);
    // keep the address in a register: without this it is re-derived from the CTA's shared window at every use
    asm volatile("" : "+r"(full0));
    if (tid == 0) {
        for (int i = 0; i < G::STAGES; i++) mbar_init(full0 + 8 * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    constexpr uint32_t kStageBytes = G::RB * G::BOX_B;
    auto issue = [&](int chunk) {
        const uint32_t bar = full0 + 8 * (chunk % G::STAGES);
        mbar_expect_tx(bar, kStageBytes);
        tma_load_3d(smem_u32(&sm.in[chunk % G::STAGES][0]), &in_map, (ibyte0 - G::PAD_L - xshift) / 4, rs + chunk * G::RB - p.in_row0, frame, bar);
    };
    if (tid == 0) {
        for (int i = 0; i < G::STAGES && i < nchunks; i++) issue(i);
    }

    // ------------------------------ H pass of one chunk ------------------------------
    int n_strict = 0;
    const float guard_h = p.guard_h, g2h = 2.f * p.guard_h;
    // lane -> (row, group) of its H item; the mapping is the same for every chunk
    int h_src0, h_dst0;
    {
        const int lr = tid / groups, g = tid - lr * groups;
        h_src0 = lr * G::BOX_B + xshift + G::WIN0 + g * G::IN_B;
        h_dst0 = lr * SWM + g * G::OUT_B;
        asm volatile("" : "+r"(h_src0), "+r"(h_dst0));
    }
    auto h_pass = [&](int chunk) {
        const int st = chunk % G::STAGES;
        mbar_wait(full0 + 8 * st, (chunk / G::STAGES) & 1);
        const int slot0 = (chunk % G::REGIONS) * G::RB;          // ring slot of this chunk's first row
#pragma unroll 1
        for (int hr = 0; hr < G::HROUNDS; hr++) {
            if (tid >= G::HB * groups) break;
            const int item = hr * G::HB * groups + tid;
            const int src_off = h_src0 + hr * (G::HB * G::BOX_B), dst_off = h_dst0 + hr * (G::HB * SWM);
            const uint2 *src = reinterpret_cast<const uint2 *>(&sm.in[st][src_off]);
            // srcw[0 .. 2*NW2): raw input words; srcw[2*NW2 ..): quantised interpolated samples, 4 per word
            uint32_t srcw[2 * G::NW2 + G::ND];
            uint32_t fix_g = 0;        // bit per packed word of interpolated samples: truncation in doubt
            uint32_t zor = 0;          // sign bit: some phase-0 sample may flip
            float f[G::NW2 * 8];
#pragma unroll
            for (int wi = 0; wi < G::NW2; wi++) {
                const uint2 w = src[wi];
                srcw[2 * wi] = w.x;
                srcw[2 * wi + 1] = w.y;
                word_to_f32x4(w.x, f[8 * wi], f[8 * wi + 1], f[8 * wi + 2], f[8 * wi + 3]);
                word_to_f32x4(w.y, f[8 * wi + 4], f[8 * wi + 5], f[8 * wi + 6], f[8 * wi + 7]);
            }
            // phase-0 samples are copies of the centre tap; "cannot flip" filter of plan.cpp:
            // v - sum K_k*b_k >= 0 over the negative residues -> the reference returns v as well
#ifndef LZB_ABL_NOHFILTER
            if (KM != 0) {
#pragma unroll
                for (int per = 0; per < PH; per++)
#pragma unroll
                    for (int c = 0; c < C; c += 2) {
                        const int base = G::MIS + per * D * C + c;
                        if (c + 1 < C) {
                            float2 z = make_float2(f[base + CEN * C], f[base + CEN * C + 1]);
#pragma unroll
                            for (int k = 0; k < TAPS; k++)
                                if ((KM >> k) & 1) z = __ffma2_rn(make_float2(f[base + k * C], f[base + k * C + 1]), make_float2(-p.align_k[k], -p.align_k[k]), z);
                            zor |= __float_as_uint(z.x) | __float_as_uint(z.y);
                        } else {
                            float z = f[base + CEN * C];
#pragma unroll
                            for (int k = 0; k < TAPS; k++)
                                if ((KM >> k) & 1) z = fmaf(f[base + k * C], -p.align_k[k], z);
                            zor |= __float_as_uint(z);
                        }
                    }
                if ((int)zor < 0) {
                    float cr[PH * C];
#pragma unroll
                    for (int per = 0; per < PH; per++)
#pragma unroll
                        for (int c = 0; c < C; c += 2) {
                            const int base = G::MIS + per * D * C + c;
                            if (c + 1 < C) {
                                float2 xs[5];
#pragma unroll
                                for (int k = 0; k < 5; k++) xs[k] = make_float2(f[base + k * C], f[base + k * C + 1]);
                                const float2 r = phase0_chain2(xs, p.p0c);
                                cr[per * C + c] = r.x;
                                cr[per * C + c + 1] = r.y;
                            } else {
                                float xs[5];
#pragma unroll
                                for (int k = 0; k < 5; k++) xs[k] = f[base + k * C];
                                cr[per * C + c] = phase0_chain1(xs, p.p0c);
                            }
                        }
#pragma unroll
                    for (int wi = 0; wi < 2 * G::NW2; wi++) {
                        float rr[4] = {0.f, 0.f, 0.f, 0.f};
                        uint32_t sel = 0x3210u;
                        bool any = false;
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const int j = 4 * wi + e - G::MIS - CEN * C;      // input byte of the item, 0 = its first own byte
                            if (j >= 0 && j < PH * D * C && (j / C) % D == 0) {
                                rr[e] = cr[((j / C) / D) * C + j % C];
                                sel = (sel & ~(0xfu << (4 * e))) | ((uint32_t)(4 + e) << (4 * e));
                                any = true;
                            }
                        }
                        if (any) {
                            const uint32_t q = quantise4(rr[0], rr[1], rr[2], rr[3]);
                            srcw[wi] = (sel == 0x7654u) ? q : __byte_perm(srcw[wi], q, sel);
                        }
                    }
                }
            }
#endif
            // window byte k (k = 0 is HALO_L bytes left of the item's own input) = f[MIS + k] * 2^24
            // interpolated samples in output order (sample s: period s / ((N-1)*C), then phase, then channel).
            // Channels c and c + 1 (c even) of a pixel use the same weights and their window bytes are neighbours:
            // they share one FFMA2 chain (one issue slot and 1.8 pipe cycles for two FMAs instead of 2 x 1.15, same
            // rounding as two FFMAs).  A window byte is only ever the first or only ever the second element of such
            // a pair, so the converted values sit in aligned register pairs without copies.
            float xa[4 * G::ND], xb[4 * G::ND];
#pragma unroll
            for (int s = 0; s < 4 * G::ND; s++) {
                if (s >= G::NI) { xa[s] = xb[s] = 0.f; continue; }
                const int per = s / ((N - 1) * C), rem = s % ((N - 1) * C);
                const int r = 1 + rem / C, c = rem % C;
                const int ph = (r * D) % N;
                const int base = G::MIS + (per * D + (r * D) / N) * C + c;   // f index of tap 0
                if (c % 2 == 0 && c + 1 < C) {
                    float2 acc = make_float2(-guard_h, -guard_h);
#pragma unroll
                    for (int i = 0; i < TAPS; i++) {
                        const int k = tap_order6<TAPS>(i);
                        acc = __ffma2_rn(make_float2(f[base + k * C], f[base + k * C + 1]), make_float2(p.wtab[ph * 8 + k], p.wtab[ph * 8 + k]), acc);
                    }
                    const float2 accb = __fadd2_rn(acc, make_float2(g2h, g2h));
                    xa[s] = acc.x; xa[s + 1] = acc.y;
                    xb[s] = accb.x; xb[s + 1] = accb.y;
                } else if (c % 2 == 0) {
                    float acc = -guard_h;
#pragma unroll
                    for (int i = 0; i < TAPS; i++) {
                        const int k = tap_order6<TAPS>(i);
                        acc = fmaf(f[base + k * C], p.wtab[ph * 8 + k], acc);
                    }
                    xa[s] = acc;
                    xb[s] = acc + g2h;
                }
            }
#pragma unroll
            for (int dw = 0; dw < G::ND; dw++) {
                const uint32_t qa = quantise4(xa[4 * dw], xa[4 * dw + 1], xa[4 * dw + 2], xa[4 * dw + 3]);
                const uint32_t qb = quantise4(xb[4 * dw], xb[4 * dw + 1], xb[4 * dw + 2], xb[4 * dw + 3]);
                srcw[2 * G::NW2 + dw] = qa;
                if (qa != qb) fix_g |= 1u << dw;
            }
            // splice copies (raw input bytes) and interpolated bytes into the output words
            uint8_t *drow = &sm.ring[slot0][dst_off];
            uint4 *dst = reinterpret_cast<uint4 *>(drow);
#pragma unroll
            for (int v4 = 0; v4 < G::OUT_B / 16; v4++) {
                uint32_t o4[4];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int ow = 4 * v4 + q;
                    int id[4], bp[4];
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        const int o = 4 * ow + e;
                        const int px = o / C, c = o % C;
                        const int per = px / N, r = px % N;
                        if (r == 0) {
                            const int bi = G::MIS + (per * D + CEN) * C + c;
                            id[e] = bi / 4;
                            bp[e] = bi % 4;
                        } else {
                            const int s = per * (N - 1) * C + (r - 1) * C + c;
                            id[e] = 2 * G::NW2 + s / 4;
                            bp[e] = s % 4;
                        }
                    }
                    o4[q] = gather4(srcw, id, bp);
                }
                dst[v4] = make_uint4(o4[0], o4[1], o4[2], o4[3]);
            }
            // rare: a truncation in doubt -> this thread looks again
            if (fix_g != 0) {
                HFixArgs a;
                const int lr = item / groups, g = item - lr * groups;
                a.in_row = &sm.in[st][lr * G::BOX_B + xshift]; a.ring_row = drow; a.gbyte0 = g * G::OUT_B;
                a.obyte0 = obyte0; a.ibyte0 = ibyte0; a.valid_bytes = hvalid;
                a.fix_g = fix_g; a.guard = guard_h;
                n_strict += h_fix<G, C, A, N, D, PH>(p, a);
            }
        }
    };

    // ------------------------------ V-pass state ------------------------------
    // partial sums of the output rows that are still collecting taps (value * 1, pixel units)
    float acc[NSLOT][VB];
#pragma unroll
    for (int j = 0; j < NSLOT; j++)
#pragma unroll
        for (int i = 0; i < VB; i++) acc[j][i] = 0.f;
    // Delay line of the phase-0 centre rows: a phase-0 output row (copy of centre row c) is stored when row c + 2
    // arrives, together with the verdict of the "cannot flip" test on both of its +-2 neighbours.
    //   FILTER: zA = the centre rows as fp16x2 words (bytes * 2^-24), zP = sign bits of the test against row c - 2
    //   else:   wP = the centre rows as packed bytes
    constexpr int ZD = (D == 1) ? 2 : 1;                       // D = 1: rows r-1 and r-2 are both centres
    uint32_t zA[ZD][VB / 2], zP[ZD];
    uint2 wP[ZD];
#pragma unroll
    for (int j = 0; j < ZD; j++) {
#pragma unroll
        for (int i = 0; i < VB / 2; i++) zA[j][i] = 0u;
        zP[j] = 0u;
        wP[j] = make_uint2(0u, 0u);
    }
    const bool v_active = VB * tid < valid_bytes;
    const bool v_second = VB * tid + 4 < valid_bytes;          // second word of the column inside the image (only !ST64)
    const float guard_v = MODE == 0 ? p.guard_v : 0.f, g2v = 2.f * p.guard_v;
    const long long opitch = p.out_pitch;
    const uint8_t *vcol = &sm.ring[0][voff + VB * tid];        // this thread's column of the ring
    uint32_t vcol_s = smem_u32(vcol);                          // ... as a 32-bit shared address (what the V loop works with)
    asm volatile("" : "+r"(vcol_s));
    const int t0_first = (rs - A - G::S0) / D;                 // exact division (also for negative values)
    int ybase = N * t0_first;                                  // output row that period t of the chunk's first iteration starts at
    uint8_t *ocol = out_frame + vbyte0 + VB * tid + (long long)(ybase - p.out_row0) * opitch;   // column in row ybase

    constexpr int NI_IT = viter_interp_rows<A, N, D, VU, G::S0>();
    const uint32_t zmask = p.strict_v_identity ? 0x80008000u : 0u;   // LANCZOS_FLAG_FAST_ALIGNED: phase-0 rows stay plain copies

    auto v_pass = [&](int chunk, bool noisy) -> bool {
        const int bslot = (chunk % G::REGIONS) * G::RB;
        const uint8_t *vrow = vcol + bslot * SWM;
        // rows [ybase, ybase + YROWS + N * (A + 2) / D] can be stored by this chunk
        const bool interior = (ybase - N >= ys) && (ybase + G::YROWS + N * (A + 2) <= ye);
        uint32_t zchunk = 0;                                   // sign bits: some phase-0 row of the chunk may flip (FILTER)
        auto body = [&](auto check_tag) {
            constexpr bool CHECK = decltype(check_tag)::value;
            const uint8_t *vit = vrow;                         // first row of the iteration
            uint8_t *op = ocol;                                // output row yit of this lane's column
            int yit = ybase;
#pragma unroll 1
            for (int it = 0; it < G::RB / VU; it++) {
                VIterFlags<NI_IT> fl;                          // what says "look again" (MODE 0), see v_fix_iter
                int qi = 0;
#pragma unroll
                for (int u = 0; u < VU; u++) {
                    const int s0 = (G::S0 + u) % D, tq = (G::S0 + u) / D;   // completing centre = D*(t + tq) + s0
                    const int cnt0 = cnt<N, D>(s0);
                    const uint2 w = *reinterpret_cast<const uint2 *>(vit + u * SWM);
                    const uint32_t h0 = __byte_perm(w.x, 0u, 0x4140), h1 = __byte_perm(w.x, 0u, 0x4342);
                    const uint32_t h2 = __byte_perm(w.y, 0u, 0x4140), h3 = __byte_perm(w.y, 0u, 0x4342);
                    float x[VB];
#ifdef LZB_ABL_NOCONV           // ablation: no byte -> fp32 conversion
                    x[0] = __uint_as_float(h0); x[1] = __uint_as_float(h0 + 1); x[2] = __uint_as_float(h1); x[3] = __uint_as_float(h1 + 1);
                    x[4] = __uint_as_float(h2); x[5] = __uint_as_float(h2 + 1); x[6] = __uint_as_float(h3); x[7] = __uint_as_float(h3 + 1);
#else
                    x[0] = h2_lo_to_f32(h0); x[1] = h2_hi_to_f32(h0); x[2] = h2_lo_to_f32(h1); x[3] = h2_hi_to_f32(h1);
                    x[4] = h2_lo_to_f32(h2); x[5] = h2_hi_to_f32(h2); x[6] = h2_lo_to_f32(h3); x[7] = h2_hi_to_f32(h3);
#endif
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
#ifdef LZB_ABL_TAPS             // ablation: only the first and the last LZB_ABL_TAPS/2 taps are computed
                                if (dc >= LZB_ABL_TAPS / 2 && dc < TAPS - LZB_ABL_TAPS / 2) { q++; continue; }
#endif
                                // two columns per FFMA2 (one issue slot for two FMAs; same rounding as two FFMAs)
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
                    auto store_row = [&](int yoff, const uint2 qv) {
#ifdef LZB_ABL_NOSTORE
                        if (qv.x != 0x12345678u) return;
#endif
                        if (CHECK && (yit + yoff < ys || yit + yoff >= ye)) return;
                        uint8_t *orow = op + (long long)yoff * opitch;
                        if (ST64) {
                            *reinterpret_cast<uint2 *>(orow) = qv;
                        } else {
                            *reinterpret_cast<uint32_t *>(orow) = qv.x;
                            if (v_second) *reinterpret_cast<uint32_t *>(orow + 4) = qv.y;
                        }
                    };
                    // ---- this row r is a phase-0 centre: the phase-0 output row of centre r - 2 goes out now ----
                    // (rows r - 2 and r + 2 of a centre are centres themselves: D <= 2).  With b = bytes * 2^-24
                    // (fp16 subnormals) and v the centre, one FMA per side and byte pair on the fp16x2 pipe:
                    //   v[r-2] - 0.375*b[r]  (this row is the +2 neighbour)  and  v[r] - 0.375*b[r-2]  (kept in zP
                    //   until row r + 2 arrives).  The exact value (a multiple of 2^-27) is rounded once, to a multiple
                    //   of 2^-24, and rounding never changes the sign; 0.375 >= plan.cpp's K_k: a set sign bit means
                    //   "the reference may return v - 1" (v_fix_iter looks again).
                    // (noisy, warp-uniform: the phase-0 rows of this chunk are all redone by v_fix_phase0_chunk anyway, see the
                    // pipeline loop: no filter, no copies here)
                    if ((s0 + A) % D == 0 && !noisy) {
                        const int zs = (ZD == 2) ? (u & 1) : 0;       // D = 1: slot of row r-2 = slot this row overwrites
                        uint2 qv;
                        if (FILTER) {
                            const uint32_t kR = 0xB600B600u;              // -0.375
                            const uint32_t hn[4] = {h0, h1, h2, h3};
                            uint32_t zpost = zP[zs], zpre = 0;
                            qv.x = __byte_perm(zA[zs][0], zA[zs][1], 0x6420);
                            qv.y = __byte_perm(zA[zs][2], zA[zs][3], 0x6420);
#pragma unroll
                            for (int i = 0; i < VB / 2; i++) {
                                zpost |= hfma2(hn[i], kR, zA[zs][i]);
                                zpre |= hfma2(zA[zs][i], kR, hn[i]);
                                zA[zs][i] = hn[i];
                            }
                            // (rows outside [ys, ye) -- warm-up rows, rows of the next segment -- are never stored: no second look)
                            if (!CHECK || (yit + N * ((G::S0 + u + A - 2) / D) >= ys && yit + N * ((G::S0 + u + A - 2) / D) < ye)) zchunk |= zpost;
                            zP[zs] = zpre;
                        } else {
                            qv = wP[zs];
                            wP[zs] = w;
                        }
                        store_row(N * ((G::S0 + u + A - 2) / D), qv);
                    }
                    // ---- interpolated rows that received their last tap ----
                    {
                        int q = 0;
#pragma unroll
                        for (int yr = ylo<N, D>(s0); yr < yhi<N, D>(s0); yr++) {
                            const int ph = (yr * D) % N;
                            if (ph == 0) continue;
                            uint2 qv;
                            qv.x = quantise4(res[q][0], res[q][1], res[q][2], res[q][3]);
                            qv.y = quantise4(res[q][4], res[q][5], res[q][6], res[q][7]);
#ifndef LZB_ABL_NOVGUARD
                            if (MODE == 0) {
                                const float2 gg = make_float2(g2v, g2v);
                                const float2 b01 = __fadd2_rn(make_float2(res[q][0], res[q][1]), gg), b23 = __fadd2_rn(make_float2(res[q][2], res[q][3]), gg);
                                const float2 b45 = __fadd2_rn(make_float2(res[q][4], res[q][5]), gg), b67 = __fadd2_rn(make_float2(res[q][6], res[q][7]), gg);
                                fl.dx[qi] = qv.x ^ quantise4(b01.x, b01.y, b23.x, b23.y);
                                fl.dy[qi] = qv.y ^ quantise4(b45.x, b45.y, b67.x, b67.y);
                            }
#else
                            if (MODE == 0) { fl.dx[qi] = 0; fl.dy[qi] = 0; }
#endif
                            q++;
                            qi++;
                            store_row(N * tq + yr, qv);
                        }
                    }
                }
                if (MODE == 0) {
                    // rare: some row of this iteration needs a second look (every row has been stored already)
                    uint32_t any = 0;
#pragma unroll
                    for (int j = 0; j < NI_IT; j++) any |= fl.dx[j] | fl.dy[j];
                    if (any != 0u)
                        n_strict += v_fix_iter<A, N, D, VU, G::S0, G::RING, SWM, ST64>(
                            p, vcol_s, (int)((uint32_t)(vit - vcol) / (uint32_t)SWM), yit, op, opitch, fl, valid_bytes - VB * tid, ys, ye);
                }
                vit += VU * SWM;
                yit += N * VU / D;
                op += (long long)(N * VU / D) * opitch;
            }
        };
        bool flagged = false;
        if constexpr (FILTER) {
            if (interior) body(std::false_type{}); else body(std::true_type{});
            flagged = noisy || (zchunk & zmask) != 0u;
            // the reference may return v - 1 somewhere in the phase-0 rows of this chunk -> all of them again, exactly
            // (rare on image-like content; in noisy mode this IS how the phase-0 rows are produced)
            if (flagged)
                v_fix_phase0_chunk<A, N, D, G::S0, G::RB, G::RING, SWM>(p, vcol_s, bslot, ybase, ocol, opitch, valid_bytes - VB * tid, ys, ye);
        } else {
            if (interior) body(std::false_type{}); else body(std::true_type{});
        }
        ybase += G::YROWS;
        ocol += (long long)G::YROWS * opitch;
        return flagged;
    };

    // ------------------------------ pipeline ------------------------------
    constexpr int kNoisyAfter = 2;     // flagged chunks in a row after which a warp stops filtering phase-0 rows
    bool noisy = false;
    int flagged_run = 0;
    for (int chunk = 0; chunk < nchunks; chunk++) {
#ifndef LZB_ABL_NOH
        h_pass(chunk);
#else
        mbar_wait(full0 + 8 * (chunk % G::STAGES), (chunk / G::STAGES) & 1);
#endif
        __syncwarp();
        // every lane has read the TMA stage of this chunk: refill it with chunk + STAGES
        if (tid == 0 && chunk + G::STAGES < nchunks) issue(chunk + G::STAGES);
#ifndef LZB_ABL_NOV
        bool flagged = false;
        if (v_active) flagged = v_pass(chunk, noisy);
        // Content that keeps flagging the phase-0 filter (noise, dark noise): after two flagged chunks in a row the warp
        // stops filtering for the rest of its segment -- the chunk-wise exact pass produces the phase-0 rows, the hot loop
        // only the interpolated ones (warp-uniform; a warp works on one strip x segment of one frame).  One loop body
        // with a uniform branch around the filter: separate loop bodies for the two modes grew the chunk loop from 16 to
        // 23 KB of code and cost image-like content 2.6 % (measured), the branch costs it 0.5 %.
        if constexpr (FILTER) {
            if (!noisy) {
                flagged_run = __any_sync(0xffffffffu, flagged) ? flagged_run + 1 : 0;
                noisy = flagged_run >= kNoisyAfter;
            }
        }
#endif
        // in-place top rows of the reference: replayed exactly once rows 0..alias_top_row+A are in the ring
        if (p.alias_rows > 0 && ys == 0 && v_active && chunk == (nchunks > 1 ? 1 : 0)) {
            AliasArgs a;
            a.col = vcol; a.ocol = out_frame + vbyte0 + VB * tid; a.opitch = opitch; a.rs = rs;
            a.nbytes = min(VB, valid_bytes - VB * tid);
            alias_fix<A, N, D, G::RB, SWM, VB>(p, a);
        }
        __syncwarp();
    }
    if (p.strict_counter && n_strict) atomicAdd(p.strict_counter, (unsigned long long)n_strict);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// Vertical segments of a launch over vperiods ratio periods, cols = strips x frames CTA columns and slots resident CTAs
// (one warp each) on sms SMs.  Every segment re-runs 2a-1 warm-up rows and works in whole chunks of RB rows, and the
// time of a chunk depends on how many warps share an SM sub-partition: measured on 1080p->2160p single frames
// (segment-count sweep, B200) it is ~(1.6 + 1.7 w) us for w = 1..4 resident warps -- two warps already reach 92 % of
// the issue rate of four.  Small jobs minimise chunks x sum over waves of that time; batches, which run many waves,
// minimise waves x rows per segment (plan_segments).
SegPlan plan_v6_segments(int vperiods, int D, int A, int RB, long long cols, long long slots, int sms, bool independent) {
    constexpr int kMaxSegs = 256;
    if (cols * 4 > slots) return plan_segments(vperiods, D, A, RB, cols, slots, kMaxSegs);
    // small job (a frame or a few): everything is resident at once, latency counts
    const int max_segs = max_segments(vperiods, D, RB);
    int segs;
    if (independent) {
        // LANCZOS_FLAG_INDEPENDENT: successive small launches of a stream overlap like the frames of a batch, so what
        // counts is throughput, not the latency of one launch: about four launches' worth of warps resident at a time
        // (measured on 1080p single frames, profiles/r02b_segs_independent.txt: 13 segments 11.6 us per frame,
        // 27 segments -- what the latency model picks -- 13.3 us, 3 segments 16.2 us)
        segs = std::max(1, std::min(max_segs, (int)std::lround((double)slots / (4.0 * (double)cols))));
    } else {
        auto chunk_time = [&](double warps) { return 1.6 + 1.7 * std::max(1.0, warps / (4.0 * sms)); };
        segs = cheapest_segments(vperiods, max_segs, kMaxSegs, [&](int per, int sg) {
            const double chunks = std::ceil((double)(per * D + 2 * A - 1) / RB);
            const long long ctas = cols * sg;
            const long long full_waves = ctas / slots, rem = ctas - full_waves * slots;
            return chunks * ((double)full_waves * chunk_time((double)slots) + (rem > 0 ? chunk_time((double)rem) : 0.0));
        });
    }
    return split_periods(vperiods, segs);
}

template <int C, int A, int N, int D, int PH, int KM, int MODE, bool ST64>
int launch_v6_one(const KParams &k, const FastHostTables &t, int *alias_in_kernel, LaunchShape *shape, cudaStream_t s) {
    using G = Geo6<C, A, N, D, PH, MODE>;
    CUtensorMap map;
    if (!encode_input_map(&map, k, G::BOX_B, G::RB)) return -1;
    auto kern = lanczos_v6_kernel<C, A, N, D, PH, KM, MODE, ST64>;
    const size_t smem = sizeof(Smem6<G>) + 128;
    static std::atomic<int> ctas_per_sm[64] = {};
    const Residency res = resident_ctas(ctas_per_sm, kern, smem);
    if (res.ctas == 0) return -1;
    const int strips = (k.out_w * C + G::SWV - 1) / G::SWV;   // one strip of SWV = 256 output bytes per warp
    const long long cols = (long long)strips * k.n_frames;
    const int vperiod0 = k.out_row0 / N;
    const int vperiods = (k.out_row0 + k.out_rows + N - 1) / N - vperiod0;
    const SegPlan sp = plan_v6_segments(vperiods, D, A, G::RB, cols, res.ctas, res.sms, (k.flags & LANCZOS_FLAG_INDEPENDENT) != 0);

    V6Params p{};
    set_strip_params(p, k, vperiod0, sp.seg_periods);
    p.wdx = k.wdx; p.wdy = k.wdy;
    p.guard_h = k.guard_outer; p.guard_v = k.guard_asc;
    p.uniform_x = t.uniform_x; p.uniform_y = t.uniform_y;
    p.strict_v_identity = (k.flags & LANCZOS_FLAG_FAST_ALIGNED) ? 0 : 1;
    // in-place top rows inside the kernel: the band must start at row 0 with input row 0 present, and every
    // intermediate row the recurrence touches must still be in the ring after chunk 1 (rows -(a-1) .. 2*RB-a)
    *alias_in_kernel = 0;
    if (k.alias_rows > 0 && k.out_row0 == 0 && k.in_row0 == 0 && k.alias_in_rows <= std::min(2 * G::RB - A, 12) + 1 && k.alias_top_row <= std::min(2 * G::RB - A, 12) - 1 &&
        k.alias_rows <= k.out_rows) {
        p.alias_rows = k.alias_rows;
        p.alias_top_row = k.alias_top_row;
        *alias_in_kernel = 1;
    }
    for (int i = 0; i < 8; i++) p.align_k[i] = i < 2 * A ? t.align_k[i] : 0.f;
    for (int i = 0; i < 5; i++) p.p0c[i] = t.p0_chain ? t.p0_chain[i] * 16777216.f : 0.f;   // x 2^24, exact
    fill_wtab(p.wtab, t, A, N);
    for (int ph = 0; ph < N && ph < 8; ph++)
        for (int q = 0; q < 8; q++) p.wdtab[ph * 8 + q] = q < 2 * A ? t.phase_wd[ph * 2 * A + q] : 0.0;
    p.strict_counter = k.strict_counter;

    dim3 grid(strips, sp.segs, k.n_frames);
    *shape = LaunchShape{(int)grid.x, (int)grid.y, (int)grid.z, sp.seg_periods, G::RB, res.ctas};
    p.independent = (k.flags & LANCZOS_FLAG_INDEPENDENT) ? 1 : 0;
    if (p.independent) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = grid;
        cfg.blockDim = dim3(32);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = s;
        cudaLaunchAttribute attr{};
        attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr.val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = &attr;
        cfg.numAttrs = 1;
        return (int)cudaLaunchKernelEx(&cfg, kern, map, p);
    }
    kern<<<grid, 32, smem, s>>>(map, p);
    return (int)cudaGetLastError();
}

}  // namespace

// Returns 0 on launch, >0 cudaError, -1 when no specialised kernel applies (caller falls back).
int launch_v6(const KParams &k, const FastHostTables &t, int *kernel_id, int *alias_in_kernel, LaunchShape *shape,
              cudaStream_t s) {
    if (!strip_layout_ok(k)) return -1;
    // 64-bit stores of the V pass
    const bool st64 = (k.out_w * k.channels) % 8 == 0 && k.out_pitch % 8 == 0 && (reinterpret_cast<uintptr_t>(k.out) & 7) == 0 &&
                      (k.n_frames <= 1 || k.out_frame_stride % 8 == 0);
    if (!t.exact_x || !t.exact_y) return -1;     // phase-0 coordinates not exactly integral in double: other kernels
    const int mode = (k.flags & LANCZOS_FLAG_TOLERANCE_1LSB) ? 1 : 0;
    const int C = k.channels, A = k.a, N = k.scale_n, D = k.scale_d;
    // KM: taps whose phase-0 residue is negative (nonzero filter constant); the host table must agree
    int km = 0;
    for (int q = 0; q < 2 * A; q++)
        if (t.align_k[q] != 0.f) km |= 1 << q;
    // the fp16x2 row filter uses K = 3/8 for every flagged tap
    for (int q = 0; q < 2 * A; q++)
        if (t.align_k[q] > 0.374f) return -1;
#define LZ6_CASE(c, a, n, d, ph, kmask, id)                                                            \
    if (C == c && A == a && N == n && D == d && km == (kmask)) {                                        \
        *kernel_id = id;                                                                                \
        if (mode == 0) return st64 ? launch_v6_one<c, a, n, d, ph, kmask, 0, true>(k, t, alias_in_kernel, shape, s)         \
                                   : launch_v6_one<c, a, n, d, ph, kmask, 0, false>(k, t, alias_in_kernel, shape, s);       \
        return st64 ? launch_v6_one<c, a, n, d, ph, kmask, 1, true>(k, t, alias_in_kernel, shape, s)                        \
                    : launch_v6_one<c, a, n, d, ph, kmask, 1, false>(k, t, alias_in_kernel, shape, s);                      \
    }
    // the phase-0 second look is the exact fp32 chain (phase0_chain2): only with plan.cpp's proof for these weights
    if (km != 0 && !t.p0_chain) return -1;
    // a = 3: sin(2*pi) < 0 in double, so the |d| = 2 taps (k = 0 and k = 4) carry negative residues
    LZ6_CASE(3, 3, 2, 1, 8, 0x11, 1)
#ifndef LZB_V6_DEV   // development builds (tools/build_variant.sh -DLZB_V6_DEV): the headline instance only
    LZ6_CASE(4, 3, 2, 1, 6, 0x11, 2)
    LZ6_CASE(4, 3, 3, 2, 4, 0x11, 3)
    LZ6_CASE(3, 2, 2, 1, 8, 0x0, 4)
    // planar images (lanczos_b200_upscale_planar): every plane is a one-channel frame
    LZ6_CASE(1, 3, 2, 1, 24, 0x11, 8)
    LZ6_CASE(1, 3, 3, 2, 16, 0x11, 9)
    LZ6_CASE(1, 2, 2, 1, 24, 0x0, 10)
#endif
#undef LZ6_CASE
    return -1;
}

}  // namespace lzb
