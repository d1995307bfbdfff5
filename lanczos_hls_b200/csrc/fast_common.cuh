// fast_common.cuh -- the strip pipeline and the device/host helpers shared by the TMA + register-window kernels
// (lanczos_v6.cu: static-phase H pass for a few ratios; lanczos_dyn.cu: any ratio with N <= 32).
#pragma once
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

#include "kernels.cuh"

namespace lzb {
namespace {

// ---------------------------------------------------------------------------------------------
// kernel parameters and the static vertical phase pattern
// ---------------------------------------------------------------------------------------------
// What both kernel families know about a launch: the output window and how it is cut into vertical segments.  The
// kernels read out_row0 + out_rows and vperiod0 + seg_periods together: each pair shares one 8-byte word.
// Columns are byte columns: the window is output bytes [out_byte0, out_byte0 + out_bytes) of a row, and the input rect
// starts at input byte in_byte0 of a row (both global: KParams out_col0 * C and in_col0 * C).  out_byte0 and in_byte0
// are the LAST fields of each family's parameter struct (V6Params, DynParams), set by launch_strips: placed here they
// moved the constant-bank offsets of every other field, and bench.py measured the headline kernel 0.6 % slower.
struct StripParams {
    uint8_t *out;         // output pixel (out_col0, out_row0) of frame 0
    long long out_pitch, out_frame_stride;
    int out_row0, out_rows;
    int seg_periods;      // vertical ratio-periods per segment
    int vperiod0;         // first vertical period covered by the launch (floor(out_row0 / N))
    int out_bytes, in_row0;
};

__host__ __device__ constexpr int cdiv(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ constexpr int lcm2(int d) { return d % 2 == 0 ? d : 2 * d; }

// residue s of a completing centre (c = D*t + s): its output rows are N*t + [ylo, yhi)
template <int N, int D> __host__ __device__ constexpr int ylo(int s) { return cdiv(s * N, D); }
template <int N, int D> __host__ __device__ constexpr int yhi(int s) { return cdiv((s + 1) * N, D); }
template <int N, int D> __host__ __device__ constexpr int cnt(int s) {   // interpolated (phase != 0) rows among them
    int n = 0;
    for (int yr = ylo<N, D>(s); yr < yhi<N, D>(s); yr++) n += ((yr * D) % N != 0) ? 1 : 0;
    return n;
}
template <int N, int D, int TAPS> __host__ __device__ constexpr int nslot() {   // partial sums alive while a row is processed
    int best = 0;
    for (int s0 = 0; s0 < D; s0++) {
        int n = 0;
        for (int dc = 0; dc < TAPS; dc++) n += cnt<N, D>((s0 + dc) % D);
        best = n > best ? n : best;
    }
    return best;
}
template <int N, int D> __host__ __device__ constexpr int cntmax() {   // rows completed by one input row (at least 1)
    int best = 1;
    for (int s = 0; s < D; s++) best = cnt<N, D>(s) > best ? cnt<N, D>(s) : best;
    return best;
}

// ---------------------------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *map, int x, int y, int z, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(z), "r"(bar)
        : "memory");
}

// u8 -> fp32 without the 16/clk I2F unit: PRMT places two bytes into the low bytes of two fp16
// lanes (0x00bb = the fp16 SUBNORMAL b * 2^-24), and one FHADD per byte widens it to fp32 exactly.
// All fp32 pixel values in these kernels therefore carry a factor 2^-24 (kPixScale); the float
// weight tables are pre-multiplied by 2^24 on the host (exact, powers of two), so sums come out in
// pixel units with exactly the rounding they would have unscaled.
constexpr float kPixUnscale = 16777216.f;  // 2^24
__device__ __forceinline__ float h2_lo_to_f32(uint32_t h2) {
    float f;
    asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %1;\n\tadd.rn.f32.f16 %0, lo, 0f00000000;\n\t}" : "=f"(f) : "r"(h2));
    return f;
}
__device__ __forceinline__ float h2_hi_to_f32(uint32_t h2) {
    float f;
    asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %1;\n\tadd.rn.f32.f16 %0, hi, 0f00000000;\n\t}" : "=f"(f) : "r"(h2));
    return f;
}
__device__ __forceinline__ void word_to_f32x4(uint32_t w, float &f0, float &f1, float &f2, float &f3) {
    const uint32_t a = __byte_perm(w, 0u, 0x4140), b = __byte_perm(w, 0u, 0x4342);
    f0 = h2_lo_to_f32(a); f1 = h2_hi_to_f32(a); f2 = h2_lo_to_f32(b); f3 = h2_hi_to_f32(b);
}

__device__ __forceinline__ uint32_t hfma2(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// double_to_uint8 (full_TB.h:29-37) on four fp32 values, packed little-endian: clamp to [0,255],
// truncate toward zero. ptxas fuses each cvt.rzi pair + cvt.pack into ONE F2IP.U8.F32.TRUNC.
__device__ __forceinline__ uint32_t quantise4(float a, float b, float c, float d) {
    const int ia = __float2int_rz(a), ib = __float2int_rz(b), ic = __float2int_rz(c), id = __float2int_rz(d);
    uint32_t hi, r;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, 0;" : "=r"(hi) : "r"(id), "r"(ic));
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(ib), "r"(ia), "r"(hi));
    return r;
}

// The reference's exact sum for one sample whose 2a taps are `stride` bytes apart in shared memory (taps outside the
// image were zero-filled by TMA).  This is exact_add spelled out: with exact_add itself ptxas schedules three kernel
// instances differently (v6 <1,3,2,1,24,17,0,true> +8 instructions, dyn <1,3,4,1,0> +6 in its chunk loop).
template <int TAPS, class W>
__device__ __forceinline__ uint8_t exact_taps(const uint8_t *tap0, int stride, W weight) {
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < TAPS; k++) {
        const double v = __hiloint2double(0x43300000, (int)tap0[k * stride]) - 4503599627370496.0;
        sum = __dadd_rn(sum, __dmul_rn(v, weight(k)));
    }
    return quantise_f64(sum);
}

// ---------------------------------------------------------------------------------------------
// the strip pipeline both families share
// ---------------------------------------------------------------------------------------------
// One warp owns a strip of output byte-columns x one vertical segment.  Chunks of RB input rows are staged by TMA
// (STAGES stages in flight, BOX_B bytes per staged row), the H pass writes them to a shared-memory ring of RING rows
// (PITCH bytes each), and the systolic V pass reads them back, VB byte-columns per lane.  A family describes its
// own choices in F (VB, RB, BOX_B, STAGES, PITCH); StripGeo adds what the pipeline derives from them.
template <int A, int N, int D, class F>
struct StripGeo : F {
    static constexpr int TAPS = 2 * A;
    static constexpr int U = lcm2(D);                             // input rows per V loop iteration (one ratio period, even)
    static constexpr int REGIONS = 2;                             // ring regions of RB rows: V(c) reads region c and the tail of c-1
    static constexpr int RING = REGIONS * F::RB;                  // intermediate rows kept in smem
    static constexpr int STAGE_B = 128 * cdiv(F::RB * F::BOX_B, 128);   // TMA destinations must be 128-byte aligned
    // the first row pushed by a segment is rs = D*pv0 - A + 1, so (row - A) mod D is static per chunk row
    static constexpr int S0 = (((1 - 2 * A) % D) + D) % D;
    static constexpr int YROWS = N * F::RB / D;                   // output rows completed per chunk
    static_assert(F::RB % U == 0, "chunk must be a whole number of V loop iterations");
    static_assert(TAPS - 1 <= F::RB, "tap rows must not reach further back than one ring region");
    static_assert(F::BOX_B / 4 <= 256, "TMA box too wide");
    static_assert(N <= 32, "phase table too large for kernel params");
    static_assert(cdiv(S0 * N, D) + YROWS <= 32, "rows fixed per chunk must fit 32 bits");
};

template <class G>
struct __align__(128) StripSmem {         // one per warp (a CTA is one warp)
    uint8_t in[G::STAGES][G::STAGE_B];    // TMA destinations, row lr at lr * BOX_B
    uint8_t ring[G::RING][G::PITCH];      // H-pass results (uint8), row r lives in slot (r - rs) % RING
    unsigned long long full[G::STAGES];   // TMA stage filled
};
template <class G> constexpr size_t strip_smem_bytes() { return sizeof(StripSmem<G>) + 128; }

// The rows of segment `seg`: ratio periods [pv0, pv1) -> output rows [ys, ye) (N*pv0 .. N*pv1 clipped to the band),
// from the intermediate rows rs .. rs + 2a - 2 + D*(pv1 - pv0) pushed in nchunks chunks of RB rows.
struct SegRows {
    int ys, ye, rs, nchunks;
};
// false when the segment has no rows in the band (the CTA has nothing to do)
template <int A, int N, int D, int RB>
__device__ __forceinline__ bool segment_rows(const StripParams &p, int seg, SegRows &r) {
    const int pv0 = p.vperiod0 + seg * p.seg_periods;
    const int y_end_band = p.out_row0 + p.out_rows;
    const int pv1 = min(pv0 + p.seg_periods, (y_end_band + N - 1) / N);
    r.ys = max(N * pv0, p.out_row0);
    r.ye = min(N * pv1, y_end_band);
    if (r.ys >= r.ye) return false;
    r.rs = D * pv0 - A + 1;                                   // first intermediate row pushed
    const int nrows = D * (pv1 - pv0) + 2 * A - 1;            // rows to push
    r.nchunks = (nrows + RB - 1) / RB;
    return true;
}

// Systolic step of the V pass: every pending output row of the lane's VB byte-columns takes its next tap from the
// converted ring row x, whose completing centre has residue s0 (c = D*t + s0).  acc[j - cnt0] = fma(x, w, acc[j]): the
// FFMA's destination does the window shift, so a V loop iteration is one ratio period of straight-line code.  A row
// takes its first tap from -guard_v; the rows that take their last tap land in res, in the order they complete.
// Two columns per FFMA2 (one issue slot for two FMAs; same rounding as two FFMAs).
// cnt0 = cnt<N, D>(s0), computed by the caller before it loads the ring row: computed here, it moves ptxas's
// schedule of the V loop (headline kernel: 8104 -> 8112 instructions, one V loop 214 -> 221).
template <int N, int D, int TAPS, int VB, int NSLOT, int CNTMAX>
__device__ __forceinline__ void systolic_step(const float (&x)[VB], float (&acc)[NSLOT][VB], float (&res)[CNTMAX][VB], int s0,
                                              int cnt0, float guard_v, const float *wtab) {
    int q = 0;
#pragma unroll
    for (int dc = 0; dc < TAPS; dc++) {
        const int sdc = (s0 + dc) % D;
        const int k = TAPS - 1 - dc;
#pragma unroll
        for (int yr = ylo<N, D>(sdc); yr < yhi<N, D>(sdc); yr++) {
            const int ph = (yr * D) % N;
            if (ph == 0) continue;
#ifdef LZB_ABL_TAPS     // ablation: only the first and the last LZB_ABL_TAPS/2 taps are computed
            if (dc >= LZB_ABL_TAPS / 2 && dc < TAPS - LZB_ABL_TAPS / 2) { q++; continue; }
#endif
            const float2 wk2 = make_float2(wtab[ph * 8 + k], wtab[ph * 8 + k]);
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

using EncodeFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                              const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                              CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode() {
    static EncodeFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeFn>(sym);
    }
    return fn;
}

// ---------------------------------------------------------------------------------------------
// host side of a launch
// ---------------------------------------------------------------------------------------------
// Layout requirements of the TMA map and of the 32-bit accesses: input rect and output window row bytes %4, input
// pitch %16, output pitch %4, 16-byte aligned input base, 4-byte aligned output base, and the same for the frame strides.
inline bool strip_layout_ok(const KParams &k) {
    if ((k.in_cols * k.channels) % 4 != 0 || (k.out_cols * k.channels) % 4 != 0) return false;
    if (k.in_pitch % 16 != 0 || k.out_pitch % 4 != 0) return false;
    if ((reinterpret_cast<uintptr_t>(k.in) & 15) != 0 || (reinterpret_cast<uintptr_t>(k.out) & 3) != 0) return false;
    if (k.n_frames > 1 && (k.in_frame_stride % 16 != 0 || k.out_frame_stride % 4 != 0)) return false;
    return true;
}

// The input rect of the frames as a 3-D tensor of 32-bit words (x, row, frame), read in boxes of box_bytes x box_rows;
// TMA fills what lies outside the rect with zeros.  At the image's edges those are the reference's dropped taps; inside
// the image no window pixel has a tap outside the rect (the caller's rect covers them), so the zeros there only reach
// samples outside the window, which are never stored.
inline bool encode_input_map(CUtensorMap *map, const KParams &k, int box_bytes, int box_rows) {
    EncodeFn encode = get_encode();
    if (!encode) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)(k.in_cols * k.channels / 4), (cuuint64_t)k.in_rows, (cuuint64_t)k.n_frames};
    const cuuint64_t strides[2] = {(cuuint64_t)k.in_pitch, (cuuint64_t)(k.n_frames > 1 ? k.in_frame_stride : k.in_pitch * k.in_rows)};
    const cuuint32_t box[3] = {(cuuint32_t)(box_bytes / 4), (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t *>(k.in), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Resident one-warp CTAs on the current device of one kernel instance that takes `smem` bytes of dynamic shared memory;
// ctas = 0 when the kernel cannot have them (the caller then falls back to another kernel).  `ctas_per_sm` is the
// instance's own cache, one entry per device: every instance of a family has the same function-pointer type, so each
// launcher instantiation keeps its own.  The calls are idempotent, so two threads racing here only repeat them.
struct Residency {
    int sms;
    long long ctas;
};
template <class Kernel>
Residency resident_ctas(std::atomic<int> (&ctas_per_sm)[64], Kernel kern, size_t smem) {
    // what both families are built for (__launch_bounds__(32, 16)); only used when the occupancy query fails
    constexpr int kFallbackCtasPerSm = 16;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    std::atomic<int> &cached = ctas_per_sm[dev & 63];
    int nb = cached.load(std::memory_order_acquire);
    if (nb == 0) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();   // clear the error state: the caller falls back to another kernel
            return {sms, 0};
        }
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, 32, smem) != cudaSuccess || nb < 1) nb = kFallbackCtasPerSm;
        cached.store(nb, std::memory_order_release);
    }
    return {sms, (long long)nb * sms};
}

// Vertical segments: the vperiods ratio periods of a launch split into segs segments of seg_periods periods each
// (the last one may be shorter).
struct SegPlan {
    int segs, seg_periods;
};
inline SegPlan split_periods(int vperiods, int segs) {
    const int seg_periods = cdiv(vperiods, segs);
    return {cdiv(vperiods, seg_periods), seg_periods};
}
// every segment re-runs 2a-1 warm-up rows and works in whole chunks of RB rows: at least 2*RB input rows each
inline int max_segments(int vperiods, int D, int RB) { return std::max(1, vperiods / std::max(1, (2 * RB) / D)); }

// The segment count in 1 .. min(max_segs, cap) of least cost(periods per segment, segments)
template <class Cost>
int cheapest_segments(int vperiods, int max_segs, int cap, Cost cost) {
    int segs = 1;
    double best_cost = 1e300;
    for (int sg = 1; sg <= std::min(max_segs, cap); sg++) {
        const int per = cdiv(vperiods, sg);
        const int sg_eff = cdiv(vperiods, per);
        const double c = cost(per, sg_eff);
        if (c < best_cost - 1e-9) { best_cost = c; segs = sg_eff; }
    }
    return segs;
}

// Segments of a batch (many waves of CTAs): cols = strips x frames CTA columns, slots = resident CTAs of the device.
// It minimises (waves) x (rows per segment + warm-up + pipeline fill); a wave that is not full still costs a full wave
// unless it is the only one.
inline SegPlan plan_segments(int vperiods, int D, int A, int RB, long long cols, long long slots, int cap) {
    const int segs = cheapest_segments(vperiods, max_segments(vperiods, D, RB), cap, [&](int per, int sg) {
        const double rows = (double)per * D + 2 * A - 1 + 0.5 * RB;
        const double waves = std::ceil((double)(cols * sg) / (double)slots);
        return (cols * sg <= slots) ? rows : rows * waves;
    });
    return split_periods(vperiods, segs);
}

// The StripParams of a launch over the window of k
inline void set_strip_params(StripParams &p, const KParams &k, int vperiod0, int seg_periods) {
    p.out = k.out;
    p.out_pitch = k.out_pitch;
    p.out_frame_stride = k.out_frame_stride;
    p.out_bytes = k.out_cols * k.channels;
    p.out_row0 = k.out_row0; p.out_rows = k.out_rows; p.in_row0 = k.in_row0;
    p.seg_periods = seg_periods; p.vperiod0 = vperiod0;
}

// polyphase table [N][8] (padded to 8 taps) times 2^24, see kPixUnscale
inline void fill_wtab(float *wtab, const FastHostTables &t, int A, int N) {
    for (int ph = 0; ph < N; ph++)
        for (int q = 0; q < 8; q++) wtab[ph * 8 + q] = q < 2 * A ? t.phase_w[ph * 2 * A + q] * 16777216.f : 0.f;
}

// The tail of a launch of either family: p arrives with the family's own fields set; this fills the fields every strip
// kernel has, reports the shape and launches kern over strips x segments x frames, one warp per CTA.  `programmatic`:
// the kernel may start before the previous kernel of the stream has finished (programmatic dependent launch).
template <class G, class P, class Kernel>
int launch_strips(Kernel kern, const CUtensorMap &map, P &p, const KParams &k, const FastHostTables &t, int strips,
                  int vperiod0, SegPlan sp, long long ctas, bool programmatic, LaunchShape *shape, cudaStream_t s) {
    set_strip_params(p, k, vperiod0, sp.seg_periods);
    p.out_byte0 = k.out_col0 * k.channels;
    p.in_byte0 = k.in_col0 * k.channels;
    fill_wtab(p.wtab, t, k.a, k.scale_n);
    p.strict_counter = k.strict_counter;
    const dim3 grid(strips, sp.segs, k.n_frames);
    *shape = LaunchShape{(int)grid.x, (int)grid.y, (int)grid.z, sp.seg_periods, G::RB, ctas};
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(32);
    cfg.dynamicSmemBytes = strip_smem_bytes<G>();
    cfg.stream = s;
    cudaLaunchAttribute attr{};
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = programmatic ? 1 : 0;
    return (int)cudaLaunchKernelEx(&cfg, kern, map, p);
}

}  // namespace
}  // namespace lzb
