/*
 * lanczos_oracle.c -- CPU ORACLE (TEST INFRASTRUCTURE ONLY; see lanczos_oracle.h).
 *
 * Restates the reference software path, reference file LanczosUpscaler/full_TB.h:
 *   double_to_uint8            full_TB.h:29-37   (clamp, then truncate toward zero)
 *   sinc                       full_TB.h:39-44
 *   lanczos_kernel             full_TB.h:51-53   (no |x|<a window test)
 *   lanczos_interpolate_row    full_TB.h:55-65   (x = xx/SCALE, zero borders, no renormalisation)
 *   lanczos_interpolate_col    full_TB.h:67-77   (in place, bottom-up -> top rows alias)
 *   lanczos_expected           full_TB.h:79-96   (all rows of all channels, then all columns)
 *   SCALE                      lanczos.h:112     ((double)SCALE_N/SCALE_D)
 *
 * Build with -O2 -ffp-contract=off and WITHOUT -march=native/-ffast-math: a fused
 * multiply-add in `sum += in[i]*L` changes truncation outcomes.
 *
 * Nothing here is copied from the reference: sizes are runtime values, storage is
 * flat, and the fast variant reorganises the loops (same arithmetic per sample,
 * same summation order, hence bit-identical results).
 */
#include "lanczos_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

/* full_TB.h:29-37 */
static uint8_t quantise(double x) {
    if (x > 255) return 255;
    if (x < 0) return 0;
    return (uint8_t)x;
}

/* full_TB.h:39-44 */
static double sinc_ref(double x) {
    if (x == 0) return 1;
    return sin(x) / x;
}

/* full_TB.h:51-53; `a` is an int macro there, so M_PI*x/a divides by (double)a */
double oracle_kernel(double x, int a) {
    return sinc_ref(M_PI * x) * sinc_ref(M_PI * x / a);
}

/* Tap range of full_TB.h:59 / :72.  The reference evaluates MAX/MIN on doubles. */
static void tap_range(double x, int a, int in_len, int *first, int *last) {
    double lo = floor(x) - a + 1;
    double hi = floor(x) + a;
    if (lo < 0) lo = 0;
    if (hi > in_len - 1) hi = in_len - 1;
    *first = (int)lo;
    *last = (int)hi;
}

static int check_args(int channels, int in_w, int in_h, int out_w, int out_h,
                      int a, int n, int d) {
    if (channels < 1 || in_w < 1 || in_h < 1 || out_w < 1 || out_h < 1) return -1;
    if (a < 1 || n < 1 || d < 1) return -1;
    /* the in-place column pass keeps the H result in the first in_h rows of the
     * output plane (full_TB.h:85), so the output must be at least that tall */
    if (out_h < in_h) return -1;
    return 0;
}

/* ---- literal variant ----------------------------------------------------- */

/* full_TB.h:55-65 */
static void interpolate_row(const uint8_t *in, uint8_t *out, int in_w, int out_w,
                            int a, double scale) {
    for (int xx = 0; xx < out_w; xx++) {
        double x = (double)xx / scale;
        double sum = 0;
        int first, last;
        tap_range(x, a, in_w, &first, &last);
        for (int i = first; i <= last; i++) {
            sum += in[i] * oracle_kernel(x - i, a);
        }
        out[xx] = quantise(sum);
    }
}

/* full_TB.h:67-77: `src` and `dst` are the same plane for VERBATIM */
static void interpolate_col(const uint8_t *src, uint8_t *dst, int col, int in_h,
                            int out_w, int out_h, int a, double scale) {
    for (int xx = out_h - 1; xx >= 0; xx--) {
        double x = (double)xx / scale;
        double sum = 0;
        int first, last;
        tap_range(x, a, in_h, &first, &last);
        for (int i = first; i <= last; i++) {
            sum += src[(size_t)i * out_w + col] * oracle_kernel(x - i, a);
        }
        dst[(size_t)xx * out_w + col] = quantise(sum);
    }
}

int oracle_expected_planar(const uint8_t *in, uint8_t *out, int channels,
                           int in_w, int in_h, int out_w, int out_h, int a,
                           int scale_n, int scale_d, int variant) {
    if (check_args(channels, in_w, in_h, out_w, out_h, a, scale_n, scale_d)) return -1;
    const double scale = (double)scale_n / scale_d; /* lanczos.h:112 */
    const size_t in_plane = (size_t)in_w * in_h, out_plane = (size_t)out_w * out_h;
    uint8_t *tmp = NULL;
    if (variant == ORACLE_CLEAN) {
        tmp = (uint8_t *)malloc(out_plane * channels);
        if (!tmp) return -2;
    }
    /* the reference's output array is a zero-initialised global (full_TB.h:21) */
    memset(out, 0, out_plane * channels);
    /* full_TB.h:83-87 */
    for (int i = 0; i < in_h; i++)
        for (int j = 0; j < channels; j++)
            interpolate_row(in + j * in_plane + (size_t)i * in_w,
                            out + j * out_plane + (size_t)i * out_w, in_w, out_w, a, scale);
    if (tmp) memcpy(tmp, out, out_plane * channels);
    /* full_TB.h:89-93 */
    for (int i1 = 0; i1 < out_w; i1++)
        for (int j = 0; j < channels; j++)
            interpolate_col(tmp ? tmp + j * out_plane : out + j * out_plane,
                            out + j * out_plane, i1, in_h, out_w, out_h, a, scale);
    free(tmp);
    return 0;
}

/* ---- fast variant: per-coordinate weights, row-wise sweeps, OpenMP ------- */

typedef struct {
    int first, last; /* inclusive tap range, already clipped */
    double w[16];    /* w[k] = L(x - (first+k)) */
} coord_t;

static coord_t *build_coords(int out_len, int in_len, int a, double scale) {
    coord_t *c = (coord_t *)malloc(sizeof(coord_t) * (size_t)out_len);
    if (!c) return NULL;
    for (int xx = 0; xx < out_len; xx++) {
        double x = (double)xx / scale;
        tap_range(x, a, in_len, &c[xx].first, &c[xx].last);
        for (int i = c[xx].first, k = 0; i <= c[xx].last; i++, k++)
            c[xx].w[k] = oracle_kernel(x - i, a);
    }
    return c;
}

/* Output rows [row0, row0 + rows) of the planar result; the other rows of `out` are scratch.  Only the input rows
 * those rows read go through the horizontal pass.  In place (VERBATIM) a top row reads rows below it that already
 * hold final output (full_TB.h:67-77), so the vertical pass starts at the first row that reads no row below itself
 * and walks up from there like the full sweep does: every row the band reads has the value the full sweep gives it. */
static int expected_planar_rows(const uint8_t *in, uint8_t *out, int channels, int in_w, int in_h, int out_w,
                                int out_h, int a, int scale_n, int scale_d, int variant, int threads, int row0,
                                int rows) {
    if (check_args(channels, in_w, in_h, out_w, out_h, a, scale_n, scale_d)) return -1;
    if (row0 < 0 || rows < 0 || row0 + rows > out_h) return -1;
    if (a > 8) return -1;
    const double scale = (double)scale_n / scale_d;
    const size_t in_plane = (size_t)in_w * in_h, out_plane = (size_t)out_w * out_h;
    coord_t *cx = build_coords(out_w, in_w, a, scale);
    coord_t *cy = build_coords(out_h, in_h, a, scale);
    uint8_t *tmp = NULL;
    if (variant == ORACLE_CLEAN) tmp = (uint8_t *)malloc(out_plane * channels);
    if (!cx || !cy || (variant == ORACLE_CLEAN && !tmp)) {
        free(cx); free(cy); free(tmp);
        return -2;
    }
#ifdef _OPENMP
    if (threads <= 0) threads = omp_get_max_threads();
#else
    threads = 1;
#endif
    memset(out, 0, out_plane * channels);
    if (rows == 0) {
        free(cx); free(cy); free(tmp);
        return 0;
    }
    /* vertical rows yy_lo..yy_hi (bottom-up), horizontal rows h_lo..h_hi; first/last grow with the output row, so
     * yy_hi is the first row at or below the band that reads no row below itself */
    const int yy_lo = row0;
    int yy_hi = row0 + rows - 1;
    while (cy[yy_hi].last > yy_hi) yy_hi = cy[yy_hi].last;
    const int h_lo = cy[yy_lo].first, h_hi = cy[yy_hi].last;
    /* horizontal pass: rows are independent */
#pragma omp parallel for num_threads(threads) schedule(static) collapse(2)
    for (int j = 0; j < channels; j++) {
        for (int i = h_lo; i <= h_hi; i++) {
            const uint8_t *src = in + j * in_plane + (size_t)i * in_w;
            uint8_t *dst = out + j * out_plane + (size_t)i * out_w;
            for (int xx = 0; xx < out_w; xx++) {
                const coord_t *c = &cx[xx];
                double sum = 0;
                for (int t = c->first, k = 0; t <= c->last; t++, k++) sum += src[t] * c->w[k];
                dst[xx] = quantise(sum);
            }
        }
    }
    if (tmp) memcpy(tmp, out, out_plane * channels);
    /* vertical pass: columns are independent; every column walks xx from the bottom
     * up exactly like full_TB.h:69, so sweeping whole row segments bottom-up per
     * column block gives the same values (including the top-row aliasing). */
    const int blk = 256;
    const int nblk = (out_w + blk - 1) / blk;
#pragma omp parallel for num_threads(threads) schedule(dynamic) collapse(2)
    for (int j = 0; j < channels; j++) {
        for (int b = 0; b < nblk; b++) {
            const int c0 = b * blk, c1 = (c0 + blk < out_w) ? c0 + blk : out_w;
            uint8_t *plane = out + j * out_plane;
            const uint8_t *src = tmp ? tmp + j * out_plane : plane;
            double acc[256];
            for (int xx = yy_hi; xx >= yy_lo; xx--) {
                const coord_t *c = &cy[xx];
                for (int col = c0; col < c1; col++) acc[col - c0] = 0;
                for (int t = c->first, k = 0; t <= c->last; t++, k++) {
                    const uint8_t *r = src + (size_t)t * out_w;
                    const double w = c->w[k];
                    for (int col = c0; col < c1; col++) acc[col - c0] += r[col] * w;
                }
                uint8_t *d = plane + (size_t)xx * out_w;
                for (int col = c0; col < c1; col++) d[col] = quantise(acc[col - c0]);
            }
        }
    }
    free(cx); free(cy); free(tmp);
    return 0;
}

int oracle_expected_planar_fast(const uint8_t *in, uint8_t *out, int channels,
                                int in_w, int in_h, int out_w, int out_h, int a,
                                int scale_n, int scale_d, int variant, int threads) {
    return expected_planar_rows(in, out, channels, in_w, in_h, out_w, out_h, a, scale_n, scale_d, variant, threads,
                                0, out_h);
}

/* ---- interleaved front end (full_TB.h:127-138, :146-165) ------------------ */

int oracle_upscale_interleaved_rows(const uint8_t *in, int64_t in_pitch,
                                    uint8_t *out_band, int64_t out_pitch,
                                    int channels, int in_w, int in_h, int out_w,
                                    int out_h, int a, int scale_n, int scale_d,
                                    int variant, int threads, int row0, int rows) {
    if (check_args(channels, in_w, in_h, out_w, out_h, a, scale_n, scale_d)) return -1;
    if (row0 < 0 || rows < 0 || row0 + rows > out_h) return -1;
    if (in_pitch == 0) in_pitch = (int64_t)in_w * channels;
    if (out_pitch == 0) out_pitch = (int64_t)out_w * channels;
    const size_t in_plane = (size_t)in_w * in_h, out_plane = (size_t)out_w * out_h;
    uint8_t *pin = (uint8_t *)malloc(in_plane * channels);
    uint8_t *pout = (uint8_t *)malloc(out_plane * channels);
    if (!pin || !pout) { free(pin); free(pout); return -2; }
    for (int y = 0; y < in_h; y++)
        for (int x = 0; x < in_w; x++)
            for (int c = 0; c < channels; c++)
                pin[c * in_plane + (size_t)y * in_w + x] = in[y * in_pitch + (int64_t)x * channels + c];
    int rc = expected_planar_rows(pin, pout, channels, in_w, in_h, out_w, out_h, a, scale_n, scale_d, variant,
                                  threads, row0, rows);
    if (rc == 0) {
        for (int y = 0; y < rows; y++)
            for (int x = 0; x < out_w; x++)
                for (int c = 0; c < channels; c++)
                    out_band[y * out_pitch + (int64_t)x * channels + c] =
                        pout[c * out_plane + (size_t)(row0 + y) * out_w + x];
    }
    free(pin); free(pout);
    return rc;
}

int oracle_upscale_interleaved(const uint8_t *in, int64_t in_pitch, uint8_t *out,
                               int64_t out_pitch, int channels, int in_w, int in_h,
                               int out_w, int out_h, int a, int scale_n, int scale_d,
                               int variant, int threads) {
    return oracle_upscale_interleaved_rows(in, in_pitch, out, out_pitch, channels, in_w, in_h,
                                           out_w, out_h, a, scale_n, scale_d, variant, threads,
                                           0, out_h);
}

/* ---- synthetic data + hash (SURVEY.md 8d, Appendix A) --------------------- */

void oracle_fill_xorshift(uint8_t *dst, int64_t n, uint64_t seed) {
    uint64_t s = seed;
    for (int64_t i = 0; i < n; i++) {
        s ^= s << 13;
        s ^= s >> 7;
        s ^= s << 17;
        dst[i] = (uint8_t)(s >> 32);
    }
}

uint64_t oracle_fnv1a64(const uint8_t *p, int64_t n) {
    uint64_t h = 1469598103934665603ULL;
    for (int64_t i = 0; i < n; i++) {
        h ^= p[i];
        h *= 1099511628211ULL;
    }
    return h;
}

int oracle_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
