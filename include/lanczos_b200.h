/*
 * lanczos_b200.h -- C ABI of the B200-native Lanczos upscaler.
 *
 * Drop-in boundary for the *software path* of PKBeam/Lanczos-HLS.  Every entry
 * point cites the reference interface it replaces (file:line relative to the
 * reference tree).  Plain pointers and sizes only; no C++ or torch types.
 *
 * Conventions kept from the reference:
 *   - 8-bit pixels, channel-interleaved, channel 0 first / lowest byte
 *     (worker.cpp:35-43, full_TB.h:130), raster order in and out
 *     (full_TB.h:127-138, lanczos.cpp:56-62);
 *   - SCALE = SCALE_N/SCALE_D = OUT/IN in lowest terms (lanczos.h:112, gcd.h:23-24);
 *     output coordinate xx maps to input coordinate xx*D/N, origin aligned, no
 *     half-pixel offset (full_TB.h:57,70);
 *   - LANCZOS_A taps each side (lanczos.h:26), window = input samples
 *     floor(x)-A+1 .. floor(x)+A, samples outside the image dropped (zero border),
 *     no weight renormalisation (full_TB.h:59,72);
 *   - horizontal pass first, quantised to uint8 by clamp-then-truncate
 *     (full_TB.h:29-37), then the vertical pass on that uint8 intermediate;
 *   - the vertical pass of the reference runs in place, bottom-up
 *     (full_TB.h:67-77), so the first few output rows read rows that already hold
 *     final output.  That is the reference's observable result and the default
 *     here; LANCZOS_FLAG_NO_ALIAS selects the ping-pong result instead.
 *
 * All `lanczos_b200_*` compute entry points run on the GPU only.  There is no CPU
 * fallback: without a usable CUDA device they return LANCZOS_ERR_CUDA.
 */
#ifndef LANCZOS_B200_H
#define LANCZOS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LANCZOS_B200_ABI_VERSION 1

/* ---- error codes (the reference has none: lanczos() is void and the test bench's
 *      EXIT_FAILURE for bad dimensions, full_TB.h:110-123, is ignored by main.cpp:18) */
enum {
    LANCZOS_OK              = 0,
    LANCZOS_ERR_NULL        = -1, /* null descriptor or buffer */
    LANCZOS_ERR_DIMS        = -2, /* non-positive or oversize dimensions / pitches too small */
    LANCZOS_ERR_CHANNELS    = -3, /* channels not in 1..4 (reference NUM_CHANNELS, lanczos.h:25) */
    LANCZOS_ERR_TAPS        = -4, /* a not in 1..4 (reference LANCZOS_A, lanczos.h:26) */
    LANCZOS_ERR_RATIO       = -5, /* scale_n/scale_d not positive, not in lowest terms after
                                     reduction, or a downscale (worker.cpp:140 assumes 1/SCALE < 1) */
    LANCZOS_ERR_RATIO_FLOAT = -6, /* floor((double)xx/SCALE) != floor(xx*D/N) for some output
                                     coordinate: the reference itself picks a shifted window there */
    LANCZOS_ERR_BAND        = -7, /* row band or window outside the image or its input pixels not supplied */
    LANCZOS_ERR_CUDA        = -8, /* CUDA runtime/driver error (see lanczos_b200_last_cuda_error) */
    LANCZOS_ERR_NOMEM       = -9,
    LANCZOS_ERR_ALIGN       = -10 /* packed-word stream shim only supports 3 channels */
};

/* ---- flags */
enum {
    /* Vertical pass reads the untouched horizontal result for every row (ping-pong).
     * Default (flag clear) reproduces the reference's in-place top rows, full_TB.h:67-77. */
    LANCZOS_FLAG_NO_ALIAS = 1u << 0,
    /* Skip the exact double-precision re-evaluation of integer-aligned output rows in the
     * vertical pass.  Output then differs from the reference by at most 1 LSB, and only at
     * samples whose coordinate lands exactly on an input sample (phase 0), where the
     * reference returns v-1 when its ~1e-17 sin(k*pi) residues sum below v. */
    LANCZOS_FLAG_FAST_ALIGNED = 1u << 1,
    /* Force the generic (any ratio) kernel even when a specialised one exists. */
    LANCZOS_FLAG_GENERIC_KERNEL = 1u << 2,
    /* Tolerance mode of BASELINE.json's north star ("at most 1 LSB per channel, exact-match
     * fraction stated"): the horizontal pass stays bit-exact, the vertical pass is evaluated in
     * plain fp32 without the exact re-evaluation of near-integer sums and of integer-aligned rows.
     * Every output byte is within 1 LSB of the reference; the exact-match fraction is reported by
     * bench.py and asserted in tests/ (> 0.999 on image-like content). */
    LANCZOS_FLAG_TOLERANCE_1LSB = 1u << 3,
    /* Device-buffer entry points only: the caller promises that this call reads nothing that earlier work on the same
     * CUDA stream is still writing, and writes nothing that earlier work is still reading or writing -- independent
     * frames of a video, one call per frame, each with its OWN output buffer (two consecutive calls into the same
     * output buffer may overlap in time).  The kernel is then launched
     * with programmatic dependent launch and does not wait for the previous kernel of the stream, so consecutive
     * single-frame calls overlap on the GPU like the frames of one batch launch instead of running back to back
     * (BASELINE configs[1] read literally: one 1080p frame per call).  Later work on the stream still waits for the
     * call as usual.  Without the flag a call is ordered after everything before it on its stream, like any kernel. */
    LANCZOS_FLAG_INDEPENDENT = 1u << 4
};

/* Runtime replacement for the reference's compile-time params.h macros
 * (template lanczos.h:9-31: IN_WIDTH, IN_HEIGHT, OUT_WIDTH, OUT_HEIGHT,
 * NUM_CHANNELS, LANCZOS_A; plus SCALE_N, SCALE_D used at lanczos.h:47-48,112). */
typedef struct lanczos_desc {
    int32_t in_w, in_h;    /* IN_WIDTH, IN_HEIGHT   */
    int32_t out_w, out_h;  /* OUT_WIDTH, OUT_HEIGHT (independent loop bounds, full_TB.h:56,69) */
    int32_t channels;      /* NUM_CHANNELS, 1..4    */
    int32_t a;             /* LANCZOS_A, 1..4       */
    int32_t scale_n;       /* SCALE_N; 0 = derive N/D from out_w/in_w by gcd (stb.cpp:9-12) */
    int32_t scale_d;       /* SCALE_D               */
    int64_t in_pitch;      /* bytes between input rows;  0 = in_w*channels  */
    int64_t out_pitch;     /* bytes between output rows; 0 = out_w*channels */
    uint32_t flags;        /* LANCZOS_FLAG_*        */
    uint32_t reserved;     /* must be 0             */
} lanczos_desc;

/* Counters of the last call on this host thread (for reports and tests). */
typedef struct lanczos_stats {
    int64_t kernel_launches;   /* kernels of this library launched by the call */
    int64_t strict_samples;    /* samples re-evaluated in exact double arithmetic (0 unless
                                  the plan was created with statistics enabled) */
    int32_t kernel_id;         /* which main kernel ran: 0 generic, 1.. specialised */
    int32_t alias_rows;        /* top rows produced by the in-place emulation */
} lanczos_stats;

/* Launch shape of the last call on this host thread (for reports and tests), taken from the FIRST main-kernel launch
 * of the call.  The host-buffer drivers run one device call per frame or band: there it describes the last of them. */
typedef struct lanczos_launch {
    int32_t grid_x, grid_y, grid_z;  /* gridDim of the main kernel; grid_z = frames (planes) of its frame group */
    int32_t seg_periods;             /* ratio periods (N output rows) per vertical segment; 0 for generic and HLS kernels */
    int32_t chunk_rows;              /* input rows per pipeline chunk of a segment; 0 for generic and HLS kernels */
    int32_t main_launches;           /* main-kernel launches of the call: one per frame group of at most 65,535 frames */
    int64_t resident_ctas;           /* resident CTAs of the device the segment plan assumed; 0 for generic and HLS */
} lanczos_launch;

/* ---- single frame, device buffers.
 * Replaces `void lanczos(stream_t in, stream_t out)` (lanczos.h:121-126) and its software
 * twin `lanczos_expected(byte[C][IN_H][IN_W], byte[C][OUT_H][OUT_W])` (full_TB.h:79-82).
 * `d_in`/`d_out` are device pointers on `device`; the call is asynchronous on `cuda_stream`
 * (a cudaStream_t, NULL = default stream). */
int lanczos_b200_upscale(const lanczos_desc *desc, const uint8_t *d_in, uint8_t *d_out,
                         int device, void *cuda_stream);

/* ---- batch of independent frames with the same descriptor (BASELINE configs 3 and 4).
 * Frame f lives at d_in + f*in_frame_stride / d_out + f*out_frame_stride
 * (0 = in_pitch*in_h / out_pitch*out_h). One launch covers a group of up to 65,535 frames (CUDA's limit on a grid's
 * y and z dimensions): larger batches run as consecutive groups on the same stream, each with its own launch. */
int lanczos_b200_upscale_batch(const lanczos_desc *desc, const uint8_t *d_in, uint8_t *d_out,
                               int32_t n_frames, int64_t in_frame_stride,
                               int64_t out_frame_stride, int device, void *cuda_stream);

/* ---- planar device buffers: the layout of the reference's software twin itself,
 * `lanczos_expected(byte img_in[C][IN_H][IN_W], byte img_out[C][OUT_H][OUT_W])` (full_TB.h:20-21, 79-96).
 * `desc->channels` = planes per frame; `in_pitch`/`out_pitch` = row pitch of a plane in bytes (0 = width).
 * Plane q (q = frame*channels + c) lives at d_in + q*in_plane_stride / d_out + q*out_plane_stride
 * (0 = pitch*height). Every plane is resampled as a one-channel image, like the reference's per-channel loops
 * (full_TB.h:83-95); the planes of all frames are one batch of n_frames*channels one-channel frames (grouped like
 * lanczos_b200_upscale_batch), which must not exceed INT32_MAX (else LANCZOS_ERR_DIMS). */
int lanczos_b200_upscale_planar(const lanczos_desc *desc, const uint8_t *d_in, uint8_t *d_out,
                                int32_t n_frames, int64_t in_plane_stride, int64_t out_plane_stride,
                                int device, void *cuda_stream);

/* ---- one row band of a large image (BASELINE config 5; SURVEY.md 8e).
 * Computes output rows [out_row0, out_row0+out_rows) of the image described by `desc`.
 * `d_in_band` points at input row `in_row0` of the image and holds `in_rows` rows; they must
 * cover lanczos_b200_band_input_rows().  `d_out_band` points at output row out_row0.
 * Phases use the global row index, so bands concatenate to the single-GPU result bit for bit. */
int lanczos_b200_upscale_band(const lanczos_desc *desc, const uint8_t *d_in_band,
                              uint8_t *d_out_band, int32_t out_row0, int32_t out_rows,
                              int32_t in_row0, int32_t in_rows, int device, void *cuda_stream);

/* Input rows [*in_row0, *in_row0+*in_rows) needed for output rows [out_row0, out_row0+out_rows):
 * floor(r0*D/N)-A+1 .. floor((r1-1)*D/N)+A clipped to the image (full_TB.h:72), widened for a
 * band that contains the in-place top rows. */
int lanczos_b200_band_input_rows(const lanczos_desc *desc, int32_t out_row0, int32_t out_rows,
                                 int32_t *in_row0, int32_t *in_rows);

/* ---- any rectangle (window) of the output image: a viewport, a tile, part of each video frame.
 * Every pixel of a window equals the pixel at the same coordinates of the whole-image result, bit for bit (phases
 * and weights follow the global column and row), and only the input pixels the window reads are needed: the
 * rectangle of lanczos_b200_region_input_rect.  A row band is the full-width window.
 *
 * lanczos_b200_region_input_rect: the input rect [*in_x0, *in_x0+*in_w) x [*in_y0, *in_y0+*in_h) that the output
 * window [out_x0, out_x0+out_w) x [out_y0, out_y0+out_h) reads.  Rows are lanczos_b200_band_input_rows of the
 * window's rows (widened for a window that contains the in-place top rows); columns are the same rule on the x-axis,
 * clipped to the image, with *in_x0 then moved left until in_x0*channels is a multiple of 16 (a view into a
 * 16-byte-aligned image with a 16-byte pitch keeps the alignment the fast kernels need).
 * LANCZOS_ERR_BAND when the window is empty or not inside the output image. */
int lanczos_b200_region_input_rect(const lanczos_desc *desc, int32_t out_x0, int32_t out_y0, int32_t out_w,
                                   int32_t out_h, int32_t *in_x0, int32_t *in_y0, int32_t *in_w, int32_t *in_h);

/* lanczos_b200_upscale_region: device buffers, asynchronous on `cuda_stream`.  `d_in_rect` points at input pixel
 * (in_x0, in_y0) and holds in_w x in_h pixels; `d_out_window` points at the window's first pixel.  desc->in_pitch and
 * desc->out_pitch are the row pitches of these two buffers (0 = dense rows of the rect and of the window), so a view
 * into a full image passes the full image's pitch.  Frames as in lanczos_b200_upscale_batch (stride 0 = pitch x rows
 * of the rect / window; groups of at most 65,535 frames); planar images pass channels = 1 and plane strides.
 * LANCZOS_ERR_BAND when the window or the rect lies outside the image, or the rect does not contain the columns and
 * rows the window reads (region_input_rect's rect before the 16-byte rounding of in_x0).  An empty window is a no-op.
 * The fast kernels need what they need for whole images, applied to the rect and the window; the static-phase kernels
 * also need (out_x0*channels) on their H-item grid (16 bytes for RGB in exact mode) and fall back otherwise. */
int lanczos_b200_upscale_region(const lanczos_desc *desc, const uint8_t *d_in_rect, uint8_t *d_out_window,
                                int32_t out_x0, int32_t out_y0, int32_t out_w, int32_t out_h, int32_t in_x0,
                                int32_t in_y0, int32_t in_w, int32_t in_h, int32_t n_frames, int64_t in_frame_stride,
                                int64_t out_frame_stride, int device, void *cuda_stream);

/* lanczos_b200_upscale_host_region: a window of a HOST image.  `h_in` is the whole image (desc->in_pitch its pitch,
 * 0 = dense); only the input rect is copied to the device and only the window back, to `h_out_window` with row pitch
 * out_window_pitch (0 = dense).  Synchronous: returns when `h_out_window` is complete. */
int lanczos_b200_upscale_host_region(const lanczos_desc *desc, const uint8_t *h_in, uint8_t *h_out_window,
                                     int32_t out_x0, int32_t out_y0, int32_t out_w, int32_t out_h,
                                     int64_t out_window_pitch, int device);

/* ---- end to end with HOST buffers: what sim_tb does around the two calls
 * (full_TB.h:127-165) minus the PNG codec.  Frames are split into chunks that are copied
 * host->device, upscaled and copied back on `n_streams` CUDA streams so that copies overlap
 * compute.  Host buffers should be pinned (lanczos_b200_host_alloc) for full PCIe speed.
 * Synchronous: returns when `h_out` is complete. */
int lanczos_b200_upscale_host(const lanczos_desc *desc, const uint8_t *h_in, uint8_t *h_out,
                              int32_t n_frames, int64_t in_frame_stride,
                              int64_t out_frame_stride, int device, int32_t n_streams);

/* ---- one large host image over several GPUs of this process, one stream per GPU, row bands
 * with redundantly read halo rows, no collectives (SURVEY.md 8e).  devices[i] are CUDA ordinals. */
int lanczos_b200_upscale_host_bands(const lanczos_desc *desc, const uint8_t *h_in, uint8_t *h_out,
                                    const int32_t *devices, int32_t n_devices);

/* ---- planar twin: exactly the argument layout of the reference's
 * `lanczos_expected(byte img_in[C][IN_H][IN_W], byte img_out[C][OUT_H][OUT_W])`
 * (full_TB.h:79-82) with HOST arrays; interleaves on the device. Pitches in `desc` are ignored. */
int lanczos_b200_expected(const lanczos_desc *desc, const uint8_t *h_in_planar,
                          uint8_t *h_out_planar, int device);

/* ---- packed-word raster stream shim for the HLS top function
 * `lanczos(hls::stream<ap_uint<24>>&, hls::stream<ap_uint<24>>&)` (lanczos.h:121-126,
 * packing worker.cpp:35-43: channel i in bits [8i+7:8i]).  Consumes exactly in_w*in_h words and
 * produces exactly out_w*out_h words (host memory, one 32-bit word per pixel, top byte 0).
 * Software-path arithmetic; channels must be 3. */
int lanczos_b200_stream(const lanczos_desc *desc, const uint32_t *h_in_words,
                        uint32_t *h_out_words, int device);

/* ---- fixed-point "HLS mode" (SURVEY.md 8f): the integer arithmetic of the reference's HLS path,
 * `lanczos()` = process_channel (lanczos.cpp:68-98): vertical pass first, LUT weights indexed by
 * |out*SCALE_D - in*SCALE_N| (kernel.cpp:50-67), exact integer MAC + de-ring clamp to the two central
 * taps (worker.cpp:45-115), zero borders above/left and replicated borders below/right
 * (worker.cpp:170-198,239-275).  Integer scales only (scale_d == 1, a*scale_n <= 127);
 * bit_precision = BIT_PRECISION (lanczos.h:28), 1..12.  Results are bit-exact against oracle/hls_oracle.c, whose
 * per-sample arithmetic is pinned to the reference's own worker.cpp:10-130 (compiled against an integer-backed
 * ap_fixed shim, oracle/Makefile target refhls).  The LUT is floor(L(x)*2^BP) with L in double: the reference's
 * hls::sinpi values are not available, so the LUT content is UNPINNED.  Device buffers, asynchronous. */
int lanczos_b200_upscale_hls(const lanczos_desc *desc, const uint8_t *d_in, uint8_t *d_out,
                             int32_t bit_precision, int32_t n_frames, int64_t in_frame_stride,
                             int64_t out_frame_stride, int device, void *cuda_stream);
/* The LUT of init_lanczos_kernel (kernel.cpp:40-45): a*scale_n+1 entries in units of 2^-bit_precision. */
int lanczos_b200_hls_lut(int32_t a, int32_t scale_n, int32_t bit_precision, int32_t *lut, int32_t capacity);

/* ---- helpers */
/* Reduce out/in to lowest terms like the reference's gcd() (stb.cpp:9-12, lanczos.h:110). */
int lanczos_b200_reduce_ratio(int32_t out_len, int32_t in_len, int32_t *scale_n, int32_t *scale_d);
/* Validate a descriptor and fill in derived defaults (ratio, pitches) in *resolved. */
int lanczos_b200_resolve(const lanczos_desc *desc, lanczos_desc *resolved);
/* Host-side weight of the reference kernel, L(x) = sinc(pi x) sinc(pi x / a) (full_TB.h:39-53). */
double lanczos_b200_kernel(double x, int32_t a);
/* Polyphase table of the plan: `phases` rows of 2a float weights (row p = phase p of the N-periodic
 * ratio, kernel.cpp:40-45's LUT restated per phase). Returns the number of phases or an error. */
int lanczos_b200_phase_table(const lanczos_desc *desc, float *weights, int32_t capacity_floats);
/* Introspection for tests: the five fp32 constants {W0, W1, 1, W3, W4}, W_k = fl32(w_k * 2^29), of the phase-0 second
 * look.  For an output coordinate exactly on an input sample the reference's double sum (full_TB.h:58-63, weights 1 at
 * the centre and sin(k*pi) residues ~1e-17 elsewhere) truncates to the centre value v or to v-1; the kernels decide
 * which with the fp32 chain t = b0*W0, y = fma(b1,W1,t), X = v + y, X = fma(b3,W3,X), X = fma(b4,W4,X), result =
 * trunc(X), which the plan proves equal to the reference for every (b0,b1,v,b3,b4) by enumerating the states of the
 * sum (plan.cpp verify_phase0_chain; tests/test_phase0_chain.py repeats the proof in numpy).  Returns 1 when the plan
 * verified the chain (a = 3), 0 when there is none (other a; the specialised kernels then need no second look or
 * are not used), or an error. */
int lanczos_b200_phase0_chain(const lanczos_desc *desc, float *consts5);
/* Number of top output rows that the reference's in-place pass aliases (0 with NO_ALIAS). */
int lanczos_b200_alias_rows(const lanczos_desc *desc);

int lanczos_b200_device_count(void);
void *lanczos_b200_host_alloc(size_t bytes);           /* pinned host memory */
void lanczos_b200_host_free(void *p);
void *lanczos_b200_device_alloc(int device, size_t bytes);
void lanczos_b200_device_free(int device, void *p);
int lanczos_b200_memcpy_h2d(int device, void *d_dst, const void *h_src, size_t bytes);
int lanczos_b200_memcpy_d2h(int device, void *h_dst, const void *d_src, size_t bytes);
int lanczos_b200_synchronize(int device);

void lanczos_b200_enable_stats(int on);                 /* count strict samples (slower) */
int lanczos_b200_get_stats(lanczos_stats *out);
int lanczos_b200_get_launch(lanczos_launch *out);       /* read only: see lanczos_launch */
const char *lanczos_b200_strerror(int code);
const char *lanczos_b200_last_cuda_error(void);
int lanczos_b200_abi_version(void);
void lanczos_b200_clear_plans(void);                    /* drop cached weight tables */

#ifdef __cplusplus
}
#endif
#endif /* LANCZOS_B200_H */
