/* abi_consumer.cpp -- a compiled C-ABI consumer (VERDICT r1 #9, SURVEY.md 8b).
 * oracle/Makefile (target `consumer`) compiles this file once per params.h configuration (-DIN_WIDTH= ...) and links it
 * against liblanczos_b200.so: one translation unit in which the reference's static planar arrays (full_TB.h:20-21) are
 * handed, as they are, to the binding INTEGRATION.md section 2 tells a maintainer to add.  Struct layout, linkage and
 * argument meaning of include/lanczos_b200.h are therefore checked by a C++ compiler, not by a ctypes mirror.  The
 * executable prints the FNV-1a-64 of its output; tests/test_abi_consumer.py compares it under -m gpu with the hash of
 * lanczos_expected's output for the same input as the CPU oracle computes it (tests/golden/abi_consumer_hashes.txt). */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "lanczos_b200.h"

#if !defined(IN_WIDTH) || !defined(IN_HEIGHT) || !defined(OUT_WIDTH) || !defined(OUT_HEIGHT) || \
    !defined(NUM_CHANNELS) || !defined(LANCZOS_A) || !defined(SCALE_N) || !defined(SCALE_D)
#error "pass -DIN_WIDTH= -DIN_HEIGHT= -DOUT_WIDTH= -DOUT_HEIGHT= -DNUM_CHANNELS= -DLANCZOS_A= -DSCALE_N= -DSCALE_D="
#endif
typedef uint8_t byte;                                                /* full_TB.h:18: ap_uint<8> used as 8-bit storage */

static byte img_in[NUM_CHANNELS][IN_HEIGHT][IN_WIDTH];             /* full_TB.h:20 */
static byte img_out_b200[NUM_CHANNELS][OUT_HEIGHT][OUT_WIDTH];     /* full_TB.h:21 */

/* INTEGRATION.md section 2, verbatim */
void lanczos_expected_b200(byte img_in[NUM_CHANNELS][IN_HEIGHT][IN_WIDTH],
                           byte img_out[NUM_CHANNELS][OUT_HEIGHT][OUT_WIDTH]) {
    lanczos_desc d = {};
    d.in_w = IN_WIDTH;   d.in_h = IN_HEIGHT;
    d.out_w = OUT_WIDTH; d.out_h = OUT_HEIGHT;
    d.channels = NUM_CHANNELS;
    d.a = LANCZOS_A;
    d.scale_n = SCALE_N; d.scale_d = SCALE_D;
    int rc = lanczos_b200_expected(&d, (const uint8_t *)img_in, (uint8_t *)img_out, /*device=*/0);
    if (rc != LANCZOS_OK) { printf("lanczos_b200: %s (%s)\n", lanczos_b200_strerror(rc), lanczos_b200_last_cuda_error()); exit(EXIT_FAILURE); }
}

int main(int argc, char **argv) {
    /* synthetic input in place of the PNG load of sim_tb (full_TB.h:127-138): xorshift64 noise, or dark noise 0..15 */
    const int dark = argc > 1 && !strcmp(argv[1], "dark");
    uint64_t s = 0x9E3779B97F4A7C15ull;
    for (int c = 0; c < NUM_CHANNELS; c++)
        for (int y = 0; y < IN_HEIGHT; y++)
            for (int x = 0; x < IN_WIDTH; x++) {
                s ^= s << 13; s ^= s >> 7; s ^= s << 17;
                img_in[c][y][x] = (byte)(dark ? (s >> 24) & 15 : (s >> 24) & 255);
            }
    if (lanczos_b200_abi_version() != LANCZOS_B200_ABI_VERSION) { printf("ABI version mismatch\n"); return 2; }
    lanczos_expected_b200(img_in, img_out_b200);     /* the drop-in for full_TB.h:141 */
    uint64_t h = 1469598103934665603ull;             /* FNV-1a-64 of the planar output */
    for (size_t i = 0; i < sizeof(img_out_b200); i++) { h ^= ((const uint8_t *)img_out_b200)[i]; h *= 1099511628211ull; }
    printf("abi_consumer %dx%d -> %dx%d c=%d a=%d %d/%d %s: fnv1a64 %016llx\n", IN_WIDTH, IN_HEIGHT, OUT_WIDTH, OUT_HEIGHT,
           NUM_CHANNELS, LANCZOS_A, SCALE_N, SCALE_D, dark ? "dark" : "noise", (unsigned long long)h);
    return 0;
}
