/* host/batch.c -- stereobatch: whole stereo pairs sharded over every GPU of the box, from C.
 *
 * BASELINE config 4 in the reference's own terms: the host scatters each GPU's pairs from pinned
 * memory, every GPU runs the whole algorithm's steps 1-2 (edges, match / box sum / winner-take-all)
 * on its pairs, the disparity maps (`web`) come back; no exchange between GPUs (SURVEY 8e).  The
 * reference has no batch program; this one exists to exercise the multi-GPU entry of the C ABI
 * (sm_multi_*, include/stereo_b200.h) without Python.
 *
 *   stereobatch WIDTH HEIGHT NUM_SHIFTS SQUARE_WIDTH N_PAIRS [wrap|ghost] [u8|u16|i32] [n_gpus] [min_shift]
 *
 * Input: the synthetic textured pairs of SURVEY 8(d) (seed 1234 + 2k for pair k), threshold 0.15.  With min_shift
 * (m) the contexts search the shifts [m, m + NUM_SHIFTS) (sm_multi_create_range) and the pairs carry the disparities
 * m + (hd mod NUM_SHIFTS) instead of hd mod NUM_SHIFTS; without it the run is the reference's range [0, NUM_SHIFTS).
 * Output line (stdout):
 *   gpus = G, pairs = N, elapsed = S, pairs_per_s = P, mde_per_s = M, web_crc32 = XXXXXXXX
 * `elapsed` covers H2D, edges, hot path and D2H of all pairs (second of two runs); the CRC is zlib's
 * over the web array as returned (i32 or u16 little endian, or u8).  u16 runs sm_multi_run_batch16, whose hot
 * kernel writes the 16-bit web itself.
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <zlib.h>

#include "stereo_b200.h"

#define CHECK(call)                                                          \
    do {                                                                     \
        int rc_ = (call);                                                    \
        if (rc_ != SM_OK) {                                                  \
            fprintf(stderr, "error: %s: %s\n", #call, sm_last_error());      \
            exit(EXIT_FAILURE);                                              \
        }                                                                    \
    } while (0)

static uint64_t splitmix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

/* SURVEY 8(d): flat gray with 1-in-8 speckle; right = left shifted by a per-tile disparity */
static uint8_t left_at(uint64_t seed, int x, int y)
{
    const uint64_t K = 0xD6E8FEB86659FD93ull;
    uint64_t hk = splitmix64(seed * K + ((uint64_t)y << 20) + (uint64_t)x);
    return ((hk >> 8) & 7) == 0 ? (uint8_t)(hk & 0xFF) : 128;
}

static void synth_pair(uint64_t seed, int w, int h, int m, int d, uint8_t *left, uint8_t *right)
{
    const uint64_t K = 0xD6E8FEB86659FD93ull;
    const int tw = 4 * d > 240 ? 4 * d : 240, th = 120;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            uint64_t hd = splitmix64((seed + 1) * K + (uint64_t)(y / th) * 4096 + (uint64_t)(x / tw));
            int disp = m + (int)(hd % (uint64_t)d);
            int xs = ((x - disp) % w + w) % w;
            left[(size_t)y * w + x] = left_at(seed, x, y);
            right[(size_t)y * w + x] = left_at(seed, xs, y);
        }
}

static double now(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

int main(int argc, char **argv)
{
    if (argc < 6) {
        fprintf(stderr,
                "usage: %s width height num_shifts square_width n_pairs [wrap|ghost] [u8|u16|i32] [n_gpus] [min_shift]\n",
                argv[0]);
        return 1;
    }
    const int w = atoi(argv[1]), h = atoi(argv[2]), d = atoi(argv[3]), sw = atoi(argv[4]), n = atoi(argv[5]);
    const int variant = (argc > 6 && strcmp(argv[6], "ghost") == 0) ? SM_GHOST : SM_WRAP;
    const int u8 = argc > 7 && strcmp(argv[7], "u8") == 0, u16 = argc > 7 && strcmp(argv[7], "u16") == 0;
    const size_t elem = u8 ? 1 : (u16 ? 2 : 4); /* bytes per web element */
    int ngpu = sm_device_count();
    if (ngpu < 1) {
        fprintf(stderr, "error: no CUDA device: %s\n", sm_last_error());
        return 1;
    }
    if (argc > 8 && atoi(argv[8]) >= 1 && atoi(argv[8]) < ngpu) ngpu = atoi(argv[8]);
    const int ms = argc > 9 ? atoi(argv[9]) : 0;
    if (w < 1 || h < 1 || d < 1 || sw < 1 || n < 1 || ms < 0) {
        fprintf(stderr, "error: arguments must be positive (min_shift non-negative)\n");
        return 1;
    }
    const size_t npix = (size_t)w * h;
    uint8_t *first, *second;
    void *web;
    CHECK(sm_host_alloc((void **)&first, npix * n));
    CHECK(sm_host_alloc((void **)&second, npix * n));
    CHECK(sm_host_alloc(&web, npix * n * elem));
    for (int k = 0; k < n; k++) synth_pair(1234 + 2 * (uint64_t)k, w, h, ms, d, first + npix * k, second + npix * k);

    int devices[64];
    for (int g = 0; g < ngpu && g < 64; g++) devices[g] = g;
    sm_multi *m;
    if (argc > 9)
        CHECK(sm_multi_create_range(&m, devices, ngpu, w, h, ms, d, sw, variant));
    else
        CHECK(sm_multi_create(&m, devices, ngpu, w, h, d, sw, variant));
    double t1 = 0.0;
    for (int run = 0; run < 2; run++) { /* first run: buffers, kernels */
        t1 = now();
        if (u16)
            CHECK(sm_multi_run_batch16(m, n, first, second, 0.15, (uint16_t *)web, NULL));
        else
            CHECK(sm_multi_run_batch(m, n, first, second, 0.15, web, u8, NULL));
    }
    double t2 = now();
    unsigned long crc = crc32(0L, Z_NULL, 0);
    const size_t bytes = npix * n * elem;
    for (size_t off = 0; off < bytes; off += (size_t)1 << 30) {
        size_t len = bytes - off < ((size_t)1 << 30) ? bytes - off : ((size_t)1 << 30);
        crc = crc32(crc, (const unsigned char *)web + off, (unsigned)len);
    }
    printf("gpus = %d, pairs = %d, elapsed = %f, pairs_per_s = %.1f, mde_per_s = %.4g, web_crc32 = %08lx\n", ngpu, n,
           t2 - t1, n / (t2 - t1), (double)npix * d * n / (t2 - t1), crc);
    CHECK(sm_multi_destroy(m));
    sm_host_free(first);
    sm_host_free(second);
    sm_host_free(web);
    return 0;
}
