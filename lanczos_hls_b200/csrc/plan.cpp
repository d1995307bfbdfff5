// plan.cpp -- descriptor validation, rational ratio, weight tables (host).
// See plan.h for the reference interfaces this replaces.
//
// Compiled with -ffp-contract=off: the double weights must be the very values the
// reference computes at full_TB.h:60 (`lanczos_kernel(x - i)` with x = (double)xx/SCALE).
#include "plan.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include <numeric>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

namespace lzb {

// full_TB.h:39-44
static double sinc_ref(double x) {
    if (x == 0) return 1;
    return std::sin(x) / x;
}

// full_TB.h:51-53 (LANCZOS_A is an int macro: M_PI*x/a divides by (double)a)
double ref_kernel(double x, int a) { return sinc_ref(M_PI * x) * sinc_ref(M_PI * x / a); }

// Phase-0 sum of the reference in fp32 (lanczos_v6.cu phase0 chain; tools/phase0_affine_proof.py is the same proof
// in numpy).  The reference adds, in double and in this order, b0*w0, b1*w1, v*1, b3*w3, b4*w4 (tap 5 is < 1e-25 and
// never changes the sum): residues of ~1e-15 against a centre v whose neighbouring doubles are u = 2^(e-52) apart
// (v in [2^e, 2^(e+1)); u/2 below a power of two).  What comes out, v or v - 1, is decided by how the residues round
// on that grid.  The fp32 grid around the same v is the double grid scaled by exactly 2^29 in every binade (24
// against 53 significand bits; the halving below powers of two and the parity of the last bit included, v being an
// integer < 256), so the same sum with residues scaled by 2^29 makes the same decisions -- unless an fp32 rounding
// error of the scaled residues (W_k carries 24 bits) moves a value across a rounding boundary.  That cannot be argued
// away, but it can be enumerated: the sum after the centre tap is v + k*u/2 with a few dozen possible k, so
//   stage 1: every (v, b0, b1)            -> k2 (16.7 M cases)
//   stage 2: every (v, reachable k2, b3)  -> k3
//   stage 3: every (v, reachable k3, b4)  -> k4 and the truncated result
// are compared between the two arithmetics, each stage starting from the exact common state.
bool verify_phase0_chain(const double *w, float *W) {
    if (!(w[0] < 0 && w[4] < 0 && w[1] > 0 && w[3] > 0 && w[2] == 1.0 && std::fabs(w[5]) < 1e-25)) return false;
    const double S29 = std::ldexp(1.0, 29);
    W[0] = (float)(w[0] * S29); W[1] = (float)(w[1] * S29); W[2] = 1.f; W[3] = (float)(w[3] * S29); W[4] = (float)(w[4] * S29);
    // the same for every plan with these weights: verified once per process
    static std::mutex mu;
    static double seen_w[6];
    static int seen = -1;
    std::lock_guard<std::mutex> lock(mu);
    if (seen >= 0 && std::memcmp(seen_w, w, sizeof seen_w) == 0) return seen == 1;
    auto run = [&]() -> bool {
        std::vector<double> s1(65536);
        std::vector<float> y1(65536);
        for (int b0 = 0; b0 < 256; b0++)
            for (int b1 = 0; b1 < 256; b1++) {
                const double p0 = (double)b0 * w[0], p1 = (double)b1 * w[1];
                s1[b0 * 256 + b1] = p0 + p1;
                const float t = (float)b0 * W[0];
                y1[b0 * 256 + b1] = std::fmaf((float)b1, W[1], t);
            }
        constexpr int KR = 512;                       // states are k in (-KR, KR) half-spacings
        for (int v = 1; v < 256; v++) {
            int e = 0;
            while ((2 << e) <= v) e++;
            const double hs = std::ldexp(1.0, e - 53), HS = hs * S29;
            const double dv = (double)v;
            const float fv = (float)v;
            bool st2[2 * KR] = {}, st3[2 * KR] = {}, st4[2 * KR] = {};
            auto same = [&](double s, float X, bool *mark) {
                const double k64 = (s - dv) / hs, k32 = ((double)X - dv) / HS;
                if (k64 != k32 || k64 != std::rint(k64) || std::fabs(k64) >= KR) return false;
                mark[(int)k64 + KR] = true;
                return true;
            };
            for (int i = 0; i < 65536; i++) {
                const double s2 = s1[i] + dv * w[2];
                const float X2 = fv + y1[i];
                if (!same(s2, X2, st2)) return false;
            }
            for (int stage = 0; stage < 2; stage++) {
                const bool *from = stage ? st3 : st2;
                bool *to = stage ? st4 : st3;
                const int tap = stage ? 4 : 3;
                for (int k = -KR + 1; k < KR; k++) {
                    if (!from[k + KR]) continue;
                    const double s_in = dv + k * hs;
                    const float X_in = (float)(dv + k * HS);
                    if ((double)X_in != dv + k * HS || (s_in - dv) / hs != (double)k) return false;   // the common state is exact in both
                    for (int b = 0; b < 256; b++) {
                        const double s = s_in + (double)b * w[tap];
                        const float X = std::fmaf((float)b, W[tap], X_in);
                        if (!same(s, X, to)) return false;
                        if (stage == 1 && std::trunc(s) != (double)std::trunc(X)) return false;
                    }
                }
            }
        }
        return true;
    };
    const bool ok = run();
    std::memcpy(seen_w, w, sizeof seen_w);
    seen = ok ? 1 : 0;
    return ok;
}

int resolve_desc(const lanczos_desc *in, lanczos_desc *out) {
    if (!in || !out) return LANCZOS_ERR_NULL;
    lanczos_desc d = *in;
    if (d.in_w < 1 || d.in_h < 1 || d.out_w < 1 || d.out_h < 1) return LANCZOS_ERR_DIMS;
    // 2^20 per side keeps every byte offset inside a row and every coordinate product in int32
    if (d.in_w > (1 << 20) || d.in_h > (1 << 20) || d.out_w > (1 << 20) || d.out_h > (1 << 20))
        return LANCZOS_ERR_DIMS;
    if (d.channels < 1 || d.channels > 4) return LANCZOS_ERR_CHANNELS;
    if (d.a < 1 || d.a > kMaxTaps / 2) return LANCZOS_ERR_TAPS;
    if (d.reserved != 0) return LANCZOS_ERR_DIMS;
    if (d.scale_n == 0 && d.scale_d == 0) {
        // lanczos.h:110 SCALE_GCD = gcd(OUT_WIDTH, IN_WIDTH)
        const int g = std::gcd(d.out_w, d.in_w);
        d.scale_n = d.out_w / g;
        d.scale_d = d.in_w / g;
    } else {
        if (d.scale_n < 1 || d.scale_d < 1) return LANCZOS_ERR_RATIO;
        const int g = std::gcd(d.scale_n, d.scale_d);
        d.scale_n /= g;
        d.scale_d /= g;
    }
    if (d.scale_n < d.scale_d) return LANCZOS_ERR_RATIO;  // upscale only (worker.cpp:140)
    if (d.scale_n > (1 << 16)) return LANCZOS_ERR_RATIO;
    // the reference keeps the horizontal result in the first in_h rows of the output plane
    if (d.out_h < d.in_h) return LANCZOS_ERR_DIMS;
    const int64_t in_row = (int64_t)d.in_w * d.channels, out_row = (int64_t)d.out_w * d.channels;
    if (d.in_pitch == 0) d.in_pitch = in_row;
    if (d.out_pitch == 0) d.out_pitch = out_row;
    if (d.in_pitch < in_row || d.out_pitch < out_row) return LANCZOS_ERR_DIMS;
    *out = d;
    return LANCZOS_OK;
}

bool float_floor_exact(int from, int to, int n, int d) {
    const double scale = (double)n / d;  // lanczos.h:112
    for (int xx = from; xx < to; xx++)
        if ((double)((int64_t)xx * d / n) != std::floor((double)xx / scale)) return false;
    return true;
}

static int build_axis(AxisTables &t, int out_len, int in_len, int a, int n, int dd,
                      const std::vector<float> &phase_w, const std::vector<double> &phase_wd) {
    const int taps = 2 * a;
    const double scale = (double)n / dd;  // lanczos.h:112
    if (!float_floor_exact(0, out_len, n, dd)) return LANCZOS_ERR_RATIO_FLOAT;
    t.out_len = out_len;
    t.in_len = in_len;
    t.i0.resize(out_len);
    t.wd.assign((size_t)out_len * taps, 0.0);
    t.wf.assign((size_t)out_len * taps, 0.f);
    t.aligned_exact = true;
    t.uniform_phase = true;
    t.fast_err = 0;
    const double u = std::ldexp(1.0, -24);  // relative half-ulp of fp32
    for (int xx = 0; xx < out_len; xx++) {
        const double x = (double)xx / scale;  // full_TB.h:57,70
        const double fx = std::floor(x);
        const int64_t q = (int64_t)xx * dd / n;
        const int phase = (int)(((int64_t)xx * dd) % n);
        if (phase == 0 && x != fx) t.aligned_exact = false;
        const int first = (int)q - a + 1;
        t.i0[xx] = first;
        double werr_coord = 0, werr_phase = 0, abs_sum = 0, round_err = 0;
        for (int k = 0; k < taps; k++) {
            const int i = first + k;
            const double w = ref_kernel(x - i, a);  // full_TB.h:60
            const float wf = (float)w;
            t.wd[(size_t)xx * taps + k] = w;
            if (w != phase_wd[(size_t)phase * taps + k]) t.uniform_phase = false;
            t.wf[(size_t)xx * taps + k] = wf;
            werr_coord += 255.0 * std::fabs((double)wf - w);
            werr_phase += 255.0 * std::fabs((double)phase_w[(size_t)phase * taps + k] - w);
            // taps are accumulated in ascending order (both kernels): the k-th FMA rounds a partial sum
            // bounded by the prefix of absolute products (+1 covers the -guard start value)
            abs_sum += 255.0 * std::fabs(w);
            round_err += u * (abs_sum + 1.0);
        }
        t.fast_err = std::max(t.fast_err, std::max(werr_coord, werr_phase) + round_err);
        // Tighter bound for the second-generation kernels (phase-table weights, FMA chains from -guard):
        //  * bytes are >= 0, so a partial sum lies in [255 * sum of negative weights, 255 * sum of positive ones];
        //  * one FMA rounds by at most half an ulp of its result: 2^(floor(log2 |result|) - 24);
        //  * the last FMA only matters when the sum is below 256 (anything above is clamped either way);
        //  * the weight error sum_k b_k (wf_k - w_k) is bounded by 255 * max(sum of positive, sum of negative errors).
        for (int order = 0; order < 2; order++) {
            double lo = 0, hi = 0, rerr = 0, dpos = 0, dneg = 0;
            for (int i = 0; i < taps; i++) {
                const int k = order == 0 ? i : ((i & 1) ? taps - 1 - i / 2 : i / 2);
                const double wf = (double)phase_w[(size_t)phase * taps + k];
                if (wf > 0) hi += 255.0 * wf; else lo += 255.0 * wf;
                double m = std::max(-lo, hi) + std::ldexp(1.0, -10);     // + the -guard start value
                if (i == taps - 1) m = std::min(m, 255.999);
                rerr += std::ldexp(1.0, (int)std::floor(std::log2(m)) - 24);
                const double dw = wf - t.wd[(size_t)xx * taps + k];
                if (dw > 0) dpos += dw; else dneg -= dw;
            }
            const double e = rerr + 255.0 * std::max(dpos, dneg);
            if (order == 0) t.err_asc = std::max(t.err_asc, e); else t.err_outer = std::max(t.err_outer, e);
        }
    }
    return LANCZOS_OK;
}

int build_plan(const lanczos_desc *desc, Plan *out) {
    Plan p;
    int rc = resolve_desc(desc, &p.d);
    if (rc != LANCZOS_OK) return rc;
    const int a = p.d.a, n = p.d.scale_n, dd = p.d.scale_d;
    p.taps = 2 * a;
    // polyphase table: phase ph of the period-N pattern is first reached at output xx with
    // (xx*D) mod N == ph; use that coordinate's weights (all coordinates of a phase agree to ~1e-13)
    p.phase_w.assign((size_t)n * p.taps, 0.f);
    p.phase_wd.assign((size_t)n * p.taps, 0.0);
    {
        const double scale = (double)n / dd;
        std::vector<char> seen(n, 0);
        for (int xx = 0; xx < n; xx++) {
            const int ph = (int)(((int64_t)xx * dd) % n);
            if (seen[ph]) continue;
            seen[ph] = 1;
            const double x = (double)xx / scale;
            const int first = (int)((int64_t)xx * dd / n) - a + 1;
            for (int k = 0; k < p.taps; k++) {
                const double w = ref_kernel(x - (first + k), a);
                p.phase_wd[(size_t)ph * p.taps + k] = w;
                p.phase_w[(size_t)ph * p.taps + k] = (float)w;
            }
        }
    }
    // Phase 0 (coordinate exactly on an input sample): the reference's weights are 1 at the centre
    // tap and ~1e-17 sin(k*pi) residues elsewhere (full_TB.h:43 has no |x|<a window).  Its double
    // sum can only fall below v (and truncate to v-1) if the negative residues outweigh half the
    // spacing of doubles below v, which is >= v*2^-54.  Sufficient for "output == v":
    //     sum_k K_k * b_k <= v,   K_k = |w_k| * 2^54 / 0.99 for residues w_k < 0 (else 0).
    p.align_k.assign(p.taps, 0.f);
    for (int k = 0; k < p.taps; k++) {
        const double w = p.phase_wd[k];
        if (k != a - 1 && w < 0) {
            const double K = -w * std::ldexp(1.0, 54) / 0.99;
            if (K > 1e-7) p.align_k[k] = (float)(K * (1.0 + 1e-6));
        }
    }
    // Phase-0 second look of lanczos_v6.cu (a = 3): the reference's sum restated exactly in fp32, see verify_phase0_chain.
    // It holds for the sign pattern of a = 3 only (taps 0 and 4 pull down, 1 and 3 lift, tap 5 is far below half an
    // ulp of 1) and is proved by enumeration for the very weights of this plan.
    if (a == 3) p.p0_chain_ok = verify_phase0_chain(p.phase_wd.data(), p.p0_chain);
    rc = build_axis(p.x, p.d.out_w, p.d.in_w, a, n, dd, p.phase_w, p.phase_wd);
    if (rc != LANCZOS_OK) return rc;
    rc = build_axis(p.y, p.d.out_h, p.d.in_h, a, n, dd, p.phase_w, p.phase_wd);
    if (rc != LANCZOS_OK) return rc;
    // guard band: 1.25x the rigorous fp32 error bound, never below 2^-14
    const double e = std::max(p.x.fast_err, p.y.fast_err);
    p.guard = (float)std::max(1.25 * e, std::ldexp(1.0, -14));
    p.guard_asc = (float)(1.0625 * std::max(p.x.err_asc, p.y.err_asc));
    p.guard_outer = (float)(1.0625 * std::max(p.x.err_outer, p.y.err_outer));

    // in-place aliasing of the vertical pass (full_TB.h:67-77): going bottom-up, row xx reads
    // rows first..last; any row i > xx has already been overwritten with final output.
    p.alias_rows = 0;
    p.alias_top_row = -1;
    p.alias_in_rows = 0;
    if (!(p.d.flags & LANCZOS_FLAG_NO_ALIAS)) {
        auto last_row = [&](int xx) { return std::min(p.d.in_h - 1, p.y.i0[xx] + p.taps - 1); };
        for (int xx = 0; xx < p.d.out_h; xx++)
            if (last_row(xx) > xx) p.alias_rows = xx + 1;
        for (int xx = 0; xx < p.alias_rows; xx++) p.alias_top_row = std::max(p.alias_top_row, last_row(xx));
        for (int xx = 0; xx <= p.alias_top_row; xx++) p.alias_in_rows = std::max(p.alias_in_rows, last_row(xx) + 1);
    }
    *out = std::move(p);
    return LANCZOS_OK;
}

void band_rows(const Plan &p, int out_row0, int out_rows, int *in_row0, int *in_rows) {
    int lo = std::min(p.d.in_h - 1, std::max(0, p.y.i0[out_row0]));
    int hi = std::min(p.d.in_h - 1, p.y.i0[out_row0 + out_rows - 1] + p.taps - 1);
    if (out_row0 < p.alias_rows) {  // the in-place emulation starts from row alias_top_row
        lo = 0;
        hi = std::max(hi, p.alias_in_rows - 1);
    }
    if (hi < lo) hi = lo;  // band entirely below the last input row: nothing is read
    *in_row0 = lo;
    *in_rows = hi - lo + 1;
}

void band_cols(const Plan &p, int out_col0, int out_cols, int *in_col0, int *in_cols) {
    const int lo = std::min(p.d.in_w - 1, std::max(0, p.x.i0[out_col0]));
    int hi = std::min(p.d.in_w - 1, p.x.i0[out_col0 + out_cols - 1] + p.taps - 1);
    if (hi < lo) hi = lo;
    *in_col0 = lo;
    *in_cols = hi - lo + 1;
}

}  // namespace lzb
