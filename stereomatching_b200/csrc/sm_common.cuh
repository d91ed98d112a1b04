// sm_common.cuh -- shared declarations of libstereo_b200 (internal, C++/CUDA).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/stereo_b200.h"

namespace smb {

// ---- error plumbing ---------------------------------------------------------
// The reference prints and exits on any CUDA failure (helper_cuda.h:890-905); the
// library records the message per thread and returns a status instead.
void set_error(const char *fmt, ...);

#define SM_CUDA(call)                                                                     \
    do {                                                                                  \
        cudaError_t e__ = (call);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            smb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,                  \
                           cudaGetErrorString(e__));                                      \
            return SM_ERR_CUDA;                                                           \
        }                                                                                 \
    } while (0)

#define SM_REQUIRE(cond, ...)                                                             \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            smb::set_error(__VA_ARGS__);                                                  \
            return SM_ERR_ARG;                                                            \
        }                                                                                 \
    } while (0)

// ---- packed edge planes -------------------------------------------------------
// The hot path never touches the u8 edge maps directly.  A pack kernel turns them
// into three 1-bit-per-pixel planes over a PADDED band:
//     LA = valid & first_edges      LB = valid & ~first_edges      RB = valid & second_edges
// so that   match(u, i) = (RB[u+i] & LA[u]) | (~RB[u+i] & LB[u])
// is the reference's `left_edges[p] == right_edges[p shifted by i]`
// (stereo.c:113-127) for in-image taps and 0 for taps that, in the GHOST variant,
// fall in the zero ghost area of the match image (stereo-ghost.c:93-97).
//   rows   : padded row pr <-> frame row row0 - half + pr,  pr in [0, BH + 2*half)
//   columns: bit index PADL + x,  x in [-half, W + half + D)
// WRAP fills the padding with the toroidally wrapped image (util.h:42-47), GHOST with
// zeros.  After packing, the kernels are variant-agnostic.
// A search range [M, M + D) that starts above zero (min_shift M) is absorbed by the
// producers: bit PADL + x of RB holds the second image at column x + M (under the same
// border policy), so RB[u+i] is shift M + i and the kernels only add M to the winning shift.
//   match(u, i) = [first(u) == second(u + M + i)]
constexpr int PADL = 32;  // left padding in bits (>= half, keeps x = 0 word aligned)

struct PackedGeom {
    int W;     // image width
    int BH;    // output rows of this band
    int ER;    // padded rows = BH + 2*half
    int half;  // square_width / 2
    int D;     // num_shifts
    int WPR;   // 32-bit words per padded row (multiple of 4)
};

inline int packed_words_per_row(int W, int half, int D)
{
    // the bit-sliced kernel reads whole 64-column strips and 64-shift chunks; the slack
    // covers its funnel-shift over-reads and the direct kernel's 64-bit windows
    int bits = PADL + ((W + 63) & ~63) + ((D + 63) & ~63) + half + 160;
    int words = (bits + 31) / 32;
    return (words + 3) & ~3;
}

// Everything a hot-path kernel needs.
struct HotArgs {
    PackedGeom g;
    const uint32_t *LA, *LB, *RB;  // [ER][WPR]
    // frame arrays [FH][W] of int32_t, or of uint16_t for the 16-bit kernels (the same argument layout for both
    // families); band row j -> frame row row0 + j.  The 16-bit direct kernel takes a NULL best (web only)
    void *best, *web;
    int row0;
    // several independent pairs in one launch (blockIdx.z): pair p's planes are plane_stride
    // words further, its outputs out_stride elements further
    int npairs = 1;
    size_t plane_stride = 0, out_stride = 0;
    // the pack kernel that produces LA/LB/RB is the launch just before on the same stream: the
    // main kernel may then start as its programmatic dependent (griddepcontrol), so that its
    // launch and prologue overlap the pack kernel's tail
    bool after_pack = false;
    // one pair per launch: number of row runs per strip (0 = one wave of resident warps)
    int force_segs = 0;
    // resident warps per SM of the bit-sliced kernel this geometry uses (prepare_bitslice; 0 = ask)
    int blocks_per_sm = 0;
    // min_shift: the planes hold shifts [M, M + D), the winner's web is M + 1 + its lane.  (Last, in the struct's
    // tail padding: the offsets of the other fields, and with them the kernels' parameter loads, stay put.)
    int M = 0;
};

// What a hot-path launch ran (SM_INFO_KERNEL_SHAPE, SM_INFO_ROW_RUNS): filled in by the launcher from the
// values it launched with.
struct LaunchRecord {
    int shape = 0;     // sm_shape code
    int row_runs = 0;  // grid.y
};

// launchers (each returns the number of kernels launched, or a negative sm_status)
int launch_pack(const uint8_t *e1, const uint8_t *e2, int FH, int row0, int variant,
                const PackedGeom &g, int M, uint32_t *LA, uint32_t *LB, uint32_t *RB, cudaStream_t s,
                int npairs = 1, size_t edge_stride = 0, size_t plane_stride = 0);
// out16: the 16-bit twin; runner_up (16-bit outputs only): the twin that also stores the runner-up score there;
// web_sub (16-bit outputs only): the twin that also stores the web in sixteenths of a shift there
int launch_direct(const HotArgs &a, cudaStream_t s, bool out16 = false, uint16_t *runner_up = nullptr,
                  uint16_t *web_sub = nullptr);
int launch_bitslice(const HotArgs &a, int num_sms, cudaStream_t s, LaunchRecord *rec);
int launch_bitslice16(const HotArgs &a, int num_sms, cudaStream_t s, LaunchRecord *rec);  // uint16_t outputs
// uint16_t outputs and the runner-up score [pairs][FH][W], pair z a.out_stride elements further
int launch_bitslice_ru(const HotArgs &a, uint16_t *runner_up, int num_sms, cudaStream_t s, LaunchRecord *rec);
// uint16_t outputs and web_sub [pairs][FH][W], pair z a.out_stride elements further; carry: the same layout, needed
// past 64 shifts (the chunk merge's per-pixel state)
int launch_bitslice_sub(const HotArgs &a, uint16_t *web_sub, uint16_t *carry, int num_sms, cudaStream_t s,
                        LaunchRecord *rec);
bool bitslice_supports(int half, int D);
int prepare_bitslice(const HotArgs &a, int num_sms);
int prepare_bitslice16(const HotArgs &a, int num_sms);
int prepare_bitslice_ru(const HotArgs &a, int num_sms);
int prepare_bitslice_sub(const HotArgs &a, int num_sms);
// web_sub = 16 * web + frac must fit 16 bits: min_shift + num_shifts <= SUB_MAX_RANGE for the sub-pixel entries
constexpr int SUB_MAX_RANGE = 4095;
int bitslice_tmem_columns(const HotArgs &a);
int bitslice_pairs_per_launch(const HotArgs &a, int num_sms, int max_pairs);
// force the (lazily loaded) kernels of each translation unit into the context
void warm_edges(int variant);
void warm_pack(int variant);
void warm_direct();
void warm_step3();

template <typename K>
inline void warm_kernel(K k)
{
    cudaFuncAttributes attr;
    (void)cudaFuncGetAttributes(&attr, k);
}
int launch_planes(const HotArgs &a, int shift, uint8_t *match, int32_t *score_all, int32_t *score,
                  cudaStream_t s);

template <typename T>
int launch_edges(const T *img, int W, int FH, int ystart, int nrows, int variant, double threshold,
                 uint8_t *edges, cudaStream_t s);

// integer fast path of the edge detector for 8-bit images: a 766 x 766 bit table per threshold
int launch_edge_lut(double threshold, uint32_t *lut, cudaStream_t s);
size_t edge_lut_words();

// both images of npairs pairs -> packed planes in one launch (edges1/edges2 non-NULL: the byte maps as well; the
// second image's only while M == 0).  M: min_shift, the second image's planes start M columns further
int launch_edges_planes(const uint8_t *img1, const uint8_t *img2, int FH, int row0, int variant, const PackedGeom &g,
                        int M, double threshold, const uint32_t *lut, uint32_t *LA, uint32_t *LB, uint32_t *RB, uint8_t *edges1,
                        uint8_t *edges2, cudaStream_t s, int npairs = 1, size_t image_stride = 0, size_t plane_stride = 0);

int launch_fill_web_holes_step(const int32_t *src, int32_t *dst, int W, int H, cudaStream_t s);
int launch_minmax_arm(int32_t *d_minmax, cudaStream_t s);
int launch_minmax(const int32_t *a, size_t n, int32_t *d_minmax, int cur, cudaStream_t s);
int launch_contour(const int32_t *web, size_t n, const int32_t *d_minmax_slot, int lines, uint8_t *out,
                   cudaStream_t s);
// int32 -> T (uint8_t or uint16_t), element-wise truncation: the caller guarantees that the values fit
template <typename T>
int launch_narrow(const int32_t *src, T *dst, size_t n, cudaStream_t s);

}  // namespace smb
