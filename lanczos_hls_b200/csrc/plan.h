// plan.h -- host-side plan: validated descriptor, rational ratio, weight tables.
//
// Replaces the reference's compile-time configuration and coefficient generator:
//   params.h macros (template lanczos.h:9-31)        -> lanczos_desc, validated at run time
//   gcd.h:1-24 + util_includes/simp (preprocessor gcd) -> std::gcd
//   init_lanczos_kernel / LUT (kernel.cpp:40-58)      -> polyphase table, one row per phase
//   lanczos_kernel(double) (full_TB.h:51-53)          -> per-coordinate double weights used by the
//                                                        exact re-evaluation path
#pragma once
#include <cstdint>
#include <vector>

#include "../../include/lanczos_b200.h"

namespace lzb {

constexpr int kMaxTaps = 8;  // 2*a, a <= 4

// One axis (x: out_w/in_w, y: out_h/in_h) of the separable resampler.
struct AxisTables {
    int out_len = 0, in_len = 0;
    std::vector<int32_t> i0;  // [out_len] first tap = floor(x)-a+1 (may be < 0)
    std::vector<double> wd;   // [out_len][2a] L(x-(i0+k)) exactly as full_TB.h:60 evaluates it
    std::vector<float> wf;    // [out_len][2a] the same rounded to float (fast path)
    bool aligned_exact = true;  // every phase-0 coordinate has x exactly integral in double
    bool uniform_phase = true;  // wd[xx][k] == phase_wd[phase(xx)][k] bit for bit, for every coordinate
    double fast_err = 0;        // rigorous bound on |fp32 fast sum - reference double sum| (ascending taps, |.| sums)
    double err_asc = 0;         // the same, sign-aware partial sums and binade-exact half-ulps, ascending taps
    double err_outer = 0;       // ... outermost taps first (lanczos_v6.cu H pass)
};

struct Plan {
    lanczos_desc d{};  // resolved: ratio reduced, pitches filled
    int taps = 0;      // 2a
    AxisTables x, y;
    std::vector<float> phase_w;  // [scale_n][2a] float polyphase table (phase p = (xx*D) mod N)
    std::vector<double> phase_wd;  // [scale_n][2a] double, for reports
    float guard = 0;             // |sum - nearest integer| below this -> exact re-evaluation
    float guard_asc = 0, guard_outer = 0;   // tighter guards of the second-generation kernels (see AxisTables)
    std::vector<float> align_k;  // [2a] phase-0 "cannot flip" filter constants (see plan.cpp)
    // a = 3, phase-0 coordinates exactly integral: the reference's double sum restated EXACTLY in fp32 (plan.cpp
    // verify_phase0_chain): {W0, W1, 1, W3, W4} with W_k = fl32(w_k * 2^29).  p0_chain_ok = the enumeration over every
    // reachable state of the sum found no difference; kernels that rely on the chain are not used without it.
    float p0_chain[5] = {0, 0, 0, 0, 0};
    bool p0_chain_ok = false;
    // in-place aliasing (full_TB.h:67-77): rows [0,alias_rows) read already-final rows
    int alias_rows = 0;     // K0
    int alias_top_row = -1; // M: largest row read by an aliased row (-1 if none)
    int alias_in_rows = 0;  // input rows the alias emulation needs: 0..alias_in_rows-1
};

// Validate + resolve. Returns LANCZOS_OK or an error code.
int resolve_desc(const lanczos_desc *in, lanczos_desc *out);

// Build all host tables. `out` must outlive device uploads.
int build_plan(const lanczos_desc *desc, Plan *out);

// The phase-0 sum of the reference (a = 3; w = its six double weights at integer distances) against its fp32
// restatement t = b0*W0, y = fma(b1, W1, t), X2 = v + y, X3 = fma(b3, W3, X2), X4 = fma(b4, W4, X3): true when
// trunc(X4) equals the reference's result for EVERY (b0, b1, v, b3, b4), by enumeration of the states of the sum.
bool verify_phase0_chain(const double *w, float *W);

// The reference kernel, full_TB.h:39-53.
double ref_kernel(double x, int a);

// True when the reference's tap origin floor((double)xx / ((double)n/d)) (full_TB.h:57) equals the exact floor(xx*d/n)
// for every output coordinate xx in [from, to): the condition behind LANCZOS_ERR_RATIO_FLOAT.
bool float_floor_exact(int from, int to, int n, int d);

// Input row range needed for a band of output rows (global indices).
void band_rows(const Plan &p, int out_row0, int out_rows, int *in_row0, int *in_rows);

}  // namespace lzb
