// k_edges.cu -- step 1, find_all_edges on the device (SURVEY 8f n1).
//
// Replaces find_all_edges<<<>>> of the reference (stereo.cu:83-92 with the four
// detectors stereo.cu:17-81; ghost twin stereo-ghost.cu:84-93).  One thread per pixel,
// FP64 with the reference's exact operation order -- ((a+b)+c)/3.0, (l+r)/2.0,
// fabs(l-r) > min(max(thr*overall,0),1) (stereo.c:16-28) -- written with the
// round-to-nearest intrinsics so that nothing is contracted or reassociated.
// Input is either the 8-bit pixels (converted as image.c:13 does, v/256.0, exact) or
// the reference's own double layout.
#include "sm_common.cuh"

namespace smb {

template <typename T>
__device__ __forceinline__ double to_bright(T v);
template <>
__device__ __forceinline__ double to_bright<uint8_t>(uint8_t v)
{
    return __ddiv_rn((double)v, 256.0);
}
template <>
__device__ __forceinline__ double to_bright<double>(double v)
{
    return v;
}

__device__ __forceinline__ int detect(double a0, double a1, double a2, double b0, double b1,
                                      double b2, double thr)
{
    double l = __ddiv_rn(__dadd_rn(__dadd_rn(a0, a1), a2), 3.0);
    double r = __ddiv_rn(__dadd_rn(__dadd_rn(b0, b1), b2), 3.0);
    double ov = __ddiv_rn(__dadd_rn(l, r), 2.0);
    double lim = __dmul_rn(thr, ov);
    lim = lim > 0.0 ? lim : 0.0;  // CLAMP = MIN(MAX(x, 0), 1), util.h:24-26
    lim = lim < 1.0 ? lim : 1.0;
    return fabs(__dsub_rn(l, r)) > lim;
}

// Rows handled: frame rows ystart .. ystart+nrows-1.  WRAP: taken mod FH (a band's halo
// rows wrap around the frame); GHOST: rows outside the frame are skipped (their edge
// cells are ghost zeros that the pack kernel supplies).
template <typename T, int VARIANT>
__global__ void __launch_bounds__(256) k_edges(const T *__restrict__ img, int W, int FH, int ystart,
                                               int nrows, double thr, uint8_t *__restrict__ edges)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int r = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= W || r >= nrows) return;
    int y = ystart + r;
    if (VARIANT == SM_WRAP) {
        y %= FH;
        if (y < 0) y += FH;
    } else if (y < 0 || y >= FH) {
        return;
    }
    double b[3][3];
#pragma unroll
    for (int dy = -1; dy <= 1; dy++) {
#pragma unroll
        for (int dx = -1; dx <= 1; dx++) {
            int xx = x + dx, yy = y + dy;
            double v;
            if (VARIANT == SM_WRAP) {
                xx = xx < 0 ? xx + W : (xx >= W ? xx - W : xx);
                yy = yy < 0 ? yy + FH : (yy >= FH ? yy - FH : yy);
                v = to_bright<T>(img[(size_t)yy * W + xx]);
            } else {
                // brightness ghost cell = 128.0 (stereo-ghost.c:384-385)
                bool in = xx >= 0 && xx < W && yy >= 0 && yy < FH;
                v = in ? to_bright<T>(img[(size_t)yy * W + xx]) : 128.0;
            }
            b[dy + 1][dx + 1] = v;
        }
    }
#define B(dx, dy) b[(dy) + 1][(dx) + 1]
    int e = detect(B(-1, -1), B(-1, 0), B(-1, 1), B(1, -1), B(1, 0), B(1, 1), thr)       // left_right
            | detect(B(-1, -1), B(0, -1), B(1, -1), B(-1, 1), B(0, 1), B(1, 1), thr)     // top_bottom
            | detect(B(-1, -1), B(0, -1), B(-1, 0), B(1, 0), B(0, 1), B(1, 1), thr)      // upleft_downright
            | detect(B(-1, 1), B(0, 1), B(-1, 0), B(0, -1), B(1, -1), B(1, 0), thr);     // downleft_upright
#undef B
    edges[(size_t)y * W + x] = (uint8_t)e;
}

template <typename T>
int launch_edges(const T *img, int W, int FH, int ystart, int nrows, int variant, double threshold,
                 uint8_t *edges, cudaStream_t s)
{
    dim3 block(64, 4);
    dim3 grid((W + block.x - 1) / block.x, (nrows + block.y - 1) / block.y);
    if (variant == SM_WRAP)
        k_edges<T, SM_WRAP><<<grid, block, 0, s>>>(img, W, FH, ystart, nrows, threshold, edges);
    else
        k_edges<T, SM_GHOST><<<grid, block, 0, s>>>(img, W, FH, ystart, nrows, threshold, edges);
    SM_CUDA(cudaGetLastError());
    return 1;
}

template int launch_edges<uint8_t>(const uint8_t *, int, int, int, int, int, double, uint8_t *,
                                   cudaStream_t);
template int launch_edges<double>(const double *, int, int, int, int, int, double, uint8_t *,
                                  cudaStream_t);

// ---- integer fast path for 8-bit images -----------------------------------------------
// With 8-bit pixels every directional detector depends only on the two integer 3-pixel
// sums L, R in [0, 765] (each brightness is k/256 exactly, so the two additions are exact
// and ((a+b)+c)/3.0 == fl((L/256)/3)) and on the threshold.  k_edge_lut evaluates the
// reference's FP64 expression (stereo.c:16-28) once for all 766 x 766 pairs into a bit
// table; the detector then needs integer adds and four table decisions per pixel.  Pixels whose
// 3x3 stencil leaves the image in the GHOST variant see the 128.0 ghost cells
// (stereo-ghost.c:384-385), which are not 8-bit values: they take the FP64 path.
constexpr int LUT_N = 766, LUT_WORDS = 24;  // 766 bits per row -> 24 words

__global__ void __launch_bounds__(256) k_edge_lut(double thr, uint32_t *__restrict__ lut)
{
    const int L = blockIdx.x;
    for (int wd = threadIdx.x; wd < LUT_WORDS; wd += blockDim.x) {
        uint32_t bits = 0;
        for (int b = 0; b < 32; b++) {
            const int R = wd * 32 + b;
            if (R < LUT_N) {
                const double sl = __ddiv_rn((double)L, 256.0), sr = __ddiv_rn((double)R, 256.0);
                // detect() with the sums already formed: pass them as (s, 0, 0)
                bits |= (uint32_t)detect(sl, 0.0, 0.0, sr, 0.0, 0.0, thr) << b;
            }
        }
        lut[L * LUT_WORDS + wd] = bits;
    }
}

__device__ __forceinline__ int lut_bit(const uint32_t *__restrict__ lut, int L, int R)
{
    return (__ldg(lut + L * LUT_WORDS + (R >> 5)) >> (R & 31)) & 1;
}

// The table as thresholds.  The detector is symmetric in its two sums (|l - r| and (l + r) / 2 are), and for a
// fixed smaller sum m the decision is monotone in the larger one: no edge up to some hi[m], edge above it.  So
//     edge(L, R) = max(L, R) > hi[min(L, R)]
// and the 73 KB bit table (four scattered global loads per pixel) shrinks to 766 sixteen-bit entries that live in
// shared memory.  k_edge_thresholds derives hi[] FROM the bit table and CHECKS both properties against every one
// of its 766 x 766 bits; the flag word it leaves behind tells the detector kernels whether the thresholds stand
// in for the table exactly (they fall back to the bit table otherwise).  Layout behind the bit table:
// [LUT_N * LUT_WORDS] bits | [HI_WORDS] hi[] as u16 pairs | [1] flag.
constexpr int HI_WORDS = (LUT_N + 1) / 2;
constexpr int LUT_HI = LUT_N * LUT_WORDS, LUT_FLAG = LUT_HI + HI_WORDS;

__global__ void k_edge_thresholds_init(uint32_t *__restrict__ lut) { lut[LUT_FLAG] = 1u; }

// one block per smaller sum m, its threads over the larger one
__global__ void __launch_bounds__(256) k_edge_thresholds(uint32_t *__restrict__ lut)
{
    const int m = blockIdx.x;
    __shared__ int first_edge;
    __shared__ int bad;
    if (threadIdx.x == 0) first_edge = LUT_N, bad = 0;
    __syncthreads();
    for (int R = m + (int)threadIdx.x; R < LUT_N; R += blockDim.x)
        if (lut_bit(lut, m, R)) atomicMin(&first_edge, R);
    __syncthreads();
    const int hi = first_edge - 1;  // the largest R >= m without an edge (LUT_N - 1: none fires)
    bool ok = true;
    for (int R = (int)threadIdx.x; R < LUT_N; R += blockDim.x) {
        const int b = lut_bit(lut, m, R);
        ok = ok && b == lut_bit(lut, R, m);            // symmetric
        if (R >= m) ok = ok && b == (R > hi ? 1 : 0);  // monotone above the diagonal
    }
    // hi = m - 1 would be an edge already at L == R: no such detector exists (|l - r| = 0 is never above a
    // non-negative limit), and an unsigned table could not hold it at m = 0; the check keeps it honest
    if (hi < m) ok = false;
    if (!ok) bad = 1;
    __syncthreads();
    if (threadIdx.x == 0) {
        reinterpret_cast<uint16_t *>(lut + LUT_HI)[m] = (uint16_t)(hi < 0 ? 0 : hi);
        if (bad) atomicAnd(lut + LUT_FLAG, 0u);
    }
}

// ---- edges straight into the packed planes ---------------------------------------------------
// The whole-algorithm and batch paths never need the byte edge maps: this kernel detects the edges of BOTH
// images of a pair over the PADDED band (rows [row0-half, row1+half), columns [-PADL, WPR*32-PADL)) and writes
// the three 1-bit planes LA / LB / RB of sm_common.cuh directly, with the border policy of the variant applied
// to the coordinates (a padding pixel of the WRAP variant IS the wrapped image pixel; GHOST padding is zero and
// invalid).  It stands in for a byte-map detector followed by k_pack: one launch and 4 B per pixel of traffic
// less.  Thread = 4 consecutive pixels of one image over EP_ROWS rows, a sliding window of three rows (three aligned
// words per new row, asked for one step early); eight threads' nibbles are OR-reduced into a 32-pixel word by
// shuffles.
// WRITE_U8: also store the byte maps (in-image pixels only), for sm_download(SM_EDGES*) and the debug planes.
// Padded rows per block and resident blocks per SM of k_edges_planes.  Measured on the fixtures, wrap / ghost
// (tools/edges_time.py): 8 rows and 56 registers (9 blocks per SM: a 1080p pair is 1.04 waves) 28.4 / 31.8 us at 1080p,
// 12.3 / 14.4 us at 480x270; 4 rows and 48 registers (10 blocks per SM, shorter serial chains) 24.6 / 30.4 and 8.2 / 12.3 us, 4K
// unchanged (63 / 75 us); 2 rows or fewer lose the sliding window at 4K, 12 blocks per SM spill.  With the frame's
// borders on the word path as well (no gather in the regular kernels): 21.6 / 20.4 us at 1080p, 61.5 / 57.4 at 4K,
// 7.2 / 8.2 at 480x270.
constexpr int EP_ROWS = 4;
constexpr int EP_BLOCKS_PER_SM = 10;

// detector decisions of 4 consecutive pixels from their 3 x 6 neighbourhood p[row][x4-1 .. x4+4]
template <typename F>
__device__ __forceinline__ uint32_t edge_nibble(const int (&p)[3][6], F &&edge)
{
    uint32_t e = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int tl = p[0][k], tc = p[0][k + 1], tr = p[0][k + 2];
        const int ml = p[1][k], mr = p[1][k + 2];
        const int bl = p[2][k], bc = p[2][k + 1], br = p[2][k + 2];
        const int b = edge(tl + ml + bl, tr + mr + br) | edge(tl + tc + tr, bl + bc + br) |
                      edge(tl + tc + ml, mr + bc + br) | edge(bl + bc + ml, tc + tr + mr);
        e |= (uint32_t)b << k;
    }
    return e;
}

// pixels x4-1 .. x4+4 of a row as three aligned words (x4 a multiple of 4, 4 <= x4 <= W - 8)
struct RowWords {
    uint32_t a, b, c;
};

// The thread's own word and the words left and right of it, at byte columns xl, x4, xr of the row.  Where the words
// beside come from is decided once per thread: the neighbouring word, or at the frame's border the row's last / first
// word (WRAP: the torus) or any in-bounds word (GHOST: the pixel next to the border is decided without it).
// sh = 8 * (first pixel - x4): a thread whose four pixels start 1..3 bytes into its word (the second image of a range
// whose minimum shift is no multiple of 4) takes its 3 x 6 bytes from the same three words, funnel-shifted.
__device__ __forceinline__ RowWords load_row(const uint8_t *__restrict__ row, int xl, int x4, int xr, int sh)
{
    const uint32_t a = __ldg(reinterpret_cast<const uint32_t *>(row + xl)), b = __ldg(reinterpret_cast<const uint32_t *>(row + x4)),
                   c = __ldg(reinterpret_cast<const uint32_t *>(row + xr));
    return RowWords{__funnelshift_r(a, b, sh), __funnelshift_r(b, c, sh), c >> sh};
}

__device__ __forceinline__ void unpack_row(const RowWords &r, int (&p)[6])
{
    p[0] = r.a >> 24;
    p[1] = r.b & 255, p[2] = (r.b >> 8) & 255, p[3] = (r.b >> 16) & 255, p[4] = r.b >> 24;
    p[5] = r.c & 255;
}

// GHOST's rare path: widths that are no multiple of 4, unaligned images, frames of one row (its borders are on the
// word path).  The 3 x 6 neighbourhood of the thread's four pixels byte by byte, every load independent, the cells
// outside the frame marked -1; then per pixel the integer detector where its stencil is inside, else the border
// rule or -- one-pixel-wide / one-pixel-high frames -- the FP64 detector with the 128.0 ghost cells
// (stereo-ghost.c:384-385).  A real call, so that the FP64 fallback does not cost the word path its registers.
__device__ __noinline__ void edge_gather_ghost(const uint8_t *__restrict__ img, int W, int FH, int x4, int ym, int y, int yp,
                                               double thr, const uint32_t *__restrict__ lut, const uint16_t *hi_s,
                                               bool thresholds_exact, uint32_t &e, uint32_t &v)
{
    auto edge = [&](int L, int R) {
        return thresholds_exact ? (int)(max(L, R) > (int)hi_s[min(L, R)]) : lut_bit(lut, L, R);
    };
    int p[3][6];
    const int ys[3] = {ym, y, yp};
#pragma unroll
    for (int k = 0; k < 6; k++) {
        const int x = x4 - 1 + k;
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const bool in = x >= 0 && x < W && ys[j] >= 0 && ys[j] < FH;
            p[j][k] = in ? (int)__ldg(img + (size_t)ys[j] * W + x) : -1;
        }
    }
    e = v = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int x = x4 + k;
        if (x < 0 || x >= W) continue;  // ghost padding: zero and invalid
        int b;
        if ((p[0][k] | p[0][k + 1] | p[0][k + 2] | p[1][k] | p[1][k + 2] | p[2][k] | p[2][k + 1] | p[2][k + 2]) >= 0) {
            const int tl = p[0][k], tc = p[0][k + 1], tr = p[0][k + 2];
            const int ml = p[1][k], mr = p[1][k + 2];
            const int bl = p[2][k], bc = p[2][k + 1], br = p[2][k + 2];
            b = edge(tl + ml + bl, tr + mr + br) | edge(tl + tc + tr, bl + bc + br) | edge(tl + tc + ml, mr + bc + br) |
                edge(bl + bc + ml, tc + tr + mr);
        } else if (W >= 2 && FH >= 2) {
            b = 1;  // the border rule (k_edges_planes)
        } else {
            auto B = [&](int dx, int dy) {
                const int q = p[dy + 1][k + 1 + dx];
                return q < 0 ? 128.0 : to_bright<uint8_t>((uint8_t)q);
            };
            b = detect(B(-1, -1), B(-1, 0), B(-1, 1), B(1, -1), B(1, 0), B(1, 1), thr) |
                detect(B(-1, -1), B(0, -1), B(1, -1), B(-1, 1), B(0, 1), B(1, 1), thr) |
                detect(B(-1, -1), B(0, -1), B(-1, 0), B(1, 0), B(0, 1), B(1, 1), thr) |
                detect(B(-1, 1), B(0, 1), B(-1, 0), B(0, -1), B(1, -1), B(1, 0), thr);
        }
        e |= (uint32_t)b << k;
        v |= 1u << k;
    }
}

// GENERIC = false: the host has checked that the width is a multiple of 4, the images are word-aligned and the frame
// has at least two rows, so every thread with pixels is on the word path and the gather (GHOST: with its FP64
// fallback and the registers it costs around the call) is not even compiled in.
template <int VARIANT, bool WRITE_U8, bool GENERIC>
__global__ void __launch_bounds__(128, EP_BLOCKS_PER_SM)
k_edges_planes(const uint8_t *__restrict__ img1, const uint8_t *__restrict__ img2, int FH, int row0, PackedGeom g,
               int M, double thr, const uint32_t *__restrict__ lut, uint32_t *__restrict__ LA, uint32_t *__restrict__ LB,
               uint32_t *__restrict__ RB, uint8_t *__restrict__ edges1, uint8_t *__restrict__ edges2, size_t image_stride,
               size_t plane_stride)
{
    // the hot kernel may be scheduled as this grid's programmatic dependent (it waits for completion before
    // it reads the planes)
    asm volatile("griddepcontrol.launch_dependents;");
    __shared__ uint16_t hi_s[2 * HI_WORDS];
    {
        const uint32_t *src = lut + LUT_HI;
        uint32_t *dst = reinterpret_cast<uint32_t *>(hi_s);
        for (int k = threadIdx.x; k < HI_WORDS; k += blockDim.x) dst[k] = __ldg(src + k);
    }
    const bool thresholds_exact = __ldg(lut + LUT_FLAG) != 0u;
    __syncthreads();
    const int pair = blockIdx.z >> 1, side = blockIdx.z & 1;
    const uint8_t *img = (side ? img2 : img1) + (size_t)pair * image_stride;
    // (the second image's byte map when its planes are offset: the host writes it, launch_edges_planes)
    uint8_t *edges = WRITE_U8 && (side == 0 || M == 0) ? (side ? edges2 : edges1) + (size_t)pair * image_stride : nullptr;
    const int W = g.W;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;  // thread <-> 4 pixels; 8 threads <-> one word
    const int wd = t >> 3;
    const int lane = threadIdx.x & 31;
    const int x4 = t * 4 - PADL;
    // the thread's first pixel: the second image's planes start M columns further (the search range [M, M + D))
    const int xc = side ? x4 + M : x4;
    const int pr0 = blockIdx.y * EP_ROWS, pr1 = min(g.ER, pr0 + EP_ROWS);
    // WRAP: a padding pixel IS the wrapped image pixel, so the thread works at its wrapped column xs (when the
    // width is a multiple of 4 its four pixels stay contiguous there).  Word path (widths that are a multiple of 4,
    // word-aligned images, frames of at least two rows): the thread's four pixels are inside the image; the words
    // beside them come through the torus (WRAP) and, GHOST, a pixel whose stencil touches the ghost area is an edge
    // without any arithmetic (below).  Everything else (GENERIC kernels only) is gathered byte by byte.
    // An offset of the second image that is no multiple of 4 (M) puts the four pixels 1..3 bytes into the aligned
    // word xs: the same three loads, funnel-shifted by fsh.  GHOST: such a thread at the frame's border has one to
    // three of its pixels inside (vmask) and stays on the word path; its words outside the frame are replaced by an
    // in-bounds one, whose bytes only reach pixels outside the frame or on its border.
    int xw = xc;
    if (VARIANT == SM_WRAP) {
        xw %= W;
        if (xw < 0) xw += W;
    }
    const int fsh = 8 * (xw & 3), xs = xw - (xw & 3);
    const bool xfast = wd < g.WPR && (W & 3) == 0 && (reinterpret_cast<uintptr_t>(img) & 3) == 0 && FH >= 2 &&
                       xw + 4 > 0 && xw < W;
    const int xb = VARIANT == SM_WRAP ? xs : min(max(xs, 0), W - 4);
    const int xl = xs >= 4 ? xs - 4 : (VARIANT == SM_WRAP ? W - 4 : xb);
    const int xr = xs + 8 <= W ? xs + 4 : (VARIANT == SM_WRAP ? 0 : xb);
    // GHOST: this thread's pixels inside the frame, and those at its left / right border
    const uint32_t vmask = VARIANT == SM_GHOST ? (0xFu << min(4, max(0, -xw))) & (0xFu >> min(4, max(0, xw + 4 - W))) & 0xFu : 0xFu;
    const uint32_t xborder = VARIANT == SM_GHOST ? ((xw <= 0 && xw > -4 ? 1u << -xw : 0u) |
                                                    (xw + 4 >= W && xw < W ? 1u << (W - 1 - xw) : 0u))
                                                 : 0u;
    auto frame_row = [&](int pr, bool &valid) {
        int y = row0 - g.half + pr;
        valid = true;
        if (VARIANT == SM_WRAP) {
            y %= FH;
            if (y < 0) y += FH;
        } else {
            valid = y >= 0 && y < FH;
        }
        return y;
    };
    auto edge_hi = [&](int L, int R) { return (int)(max(L, R) > (int)hi_s[min(L, R)]); };
    auto edge_lut = [&](int L, int R) { return lut_bit(lut, L, R); };

    int p[3][6];       // rows y-1, y, y+1 of the sliding window (xfast threads only)
    int have_y = -2;   // p[1], p[2] hold rows have_y, have_y + 1 (unwrapped successor) when have_y >= 0
    RowWords ahead = {0u, 0u, 0u};  // the row the NEXT step will need, asked for one step early
    int ahead_y = -2;
    bool rowvalid;
    int y = frame_row(pr0, rowvalid);
    for (int pr = pr0; pr < pr1; pr++) {
        uint32_t e = 0, v = 0;
        // frame row of the next padded row: one step further (mod FH for WRAP), no division in the loop
        int yn = y + 1;
        bool nvalid = true;
        if (VARIANT == SM_WRAP) {
            yn = yn >= FH ? yn - FH : yn;
        } else {
            nvalid = yn >= 0 && yn < FH;
        }
        if (wd < g.WPR && rowvalid) {
            int ym = y - 1, yp = y + 1;
            if (VARIANT == SM_WRAP) {
                ym = ym < 0 ? ym + FH : ym;
                yp = yp >= FH ? yp - FH : yp;
            }
            if (VARIANT == SM_GHOST && xfast && (ym < 0 || yp >= FH)) {
                // GHOST, first or last row of the frame: every stencil touches the ghost area and fires (see the
                // border rule below); nothing to load
                have_y = -2;
                e = v = vmask;
            } else if (xfast && ym >= 0 && yp < FH) {
                // consecutive padded rows are consecutive frame rows (mod FH): the window slides, one new row
                // of three words per step, and that row was asked for during the previous step
                RowWords top;
                if (ahead_y == yp) {
                    top = ahead;
                } else {
                    top = load_row(img + (size_t)yp * W, xl, xb, xr, fsh);
                }
                if (have_y == ym) {
#pragma unroll
                    for (int k = 0; k < 6; k++) p[0][k] = p[1][k], p[1][k] = p[2][k];
                } else {
                    unpack_row(load_row(img + (size_t)ym * W, xl, xb, xr, fsh), p[0]);
                    unpack_row(load_row(img + (size_t)y * W, xl, xb, xr, fsh), p[1]);
                }
                {
                    // the row below the next step's row (its `yp`), if that step slides on from this one
                    int y2 = yn + 1;
                    if (VARIANT == SM_WRAP) y2 = y2 >= FH ? y2 - FH : y2;
                    ahead_y = -2;
                    if (pr + 1 < pr1 && nvalid && yn == yp && y2 < FH) {
                        ahead = load_row(img + (size_t)y2 * W, xl, xb, xr, fsh);
                        ahead_y = y2;
                    }
                }
                unpack_row(top, p[2]);
                have_y = y;
                e = thresholds_exact ? edge_nibble(p, edge_hi) : edge_nibble(p, edge_lut);
                // GHOST border rule: a stencil that touches the ghost area always fires.  Towards the border one
                // detector sees three 128.0 cells (l = 128 exactly) or, in a corner, one (r > 42) against image cells
                // below 1 on the other side: a difference above 41, and the limit is clamped to at most 1
                // (stereo-ghost.c: CLAMP, util.h:24-26).  It needs frames of at least 2 x 2: a one-pixel-wide or
                // one-pixel-high frame has ghost cells on BOTH sides of a detector (those take the gather path).
                e |= xborder;
                v = vmask;
            } else {
                have_y = -2;
                if (VARIANT == SM_WRAP && GENERIC) {
                    // widths that are no multiple of 4, unaligned images, one-row frames: every byte through the
                    // wrap, all 18 loads independent (one memory round trip per row, not one per pixel)
                    int xk[6];
#pragma unroll
                    for (int k = 0; k < 6; k++) xk[k] = (xw - 1 + k + W) % W;  // (xw is in [0, W))
                    const int ys[3] = {ym, y, yp};
#pragma unroll
                    for (int j = 0; j < 3; j++)
#pragma unroll
                        for (int k = 0; k < 6; k++) p[j][k] = __ldg(img + (size_t)ys[j] * W + xk[k]);
                    e = thresholds_exact ? edge_nibble(p, edge_hi) : edge_nibble(p, edge_lut);
                    v = 0xFu;
                } else if (VARIANT == SM_GHOST && GENERIC) {
                    edge_gather_ghost(img, W, FH, xc, ym, y, yp, thr, lut, hi_s, thresholds_exact, e, v);
                }  // else: GHOST padding beside the frame, zero and invalid
            }
            if (WRITE_U8 && edges) {
                // the byte maps hold the frame itself: only the unwrapped in-image pixels of this word
                if (x4 >= 0 && x4 + 4 <= W && (W & 3) == 0 && (reinterpret_cast<uintptr_t>(edges) & 3) == 0) {
                    *reinterpret_cast<uint32_t *>(edges + (size_t)y * W + x4) =
                        (e & 1u) | ((e & 2u) << 7) | ((e & 4u) << 14) | ((e & 8u) << 21);
                } else {
                    for (int k = 0; k < 4; k++)
                        if (x4 + k >= 0 && x4 + k < W) edges[(size_t)y * W + x4 + k] = (uint8_t)((e >> k) & 1u);
                }
            }
        } else {
            have_y = -2;
        }
        // eight threads' nibbles -> one 32-pixel word (all 32 lanes take part)
        const int nsh = 4 * (lane & 7);
        uint32_t ew = e << nsh, vw = v << nsh;
#pragma unroll
        for (int m = 1; m <= 4; m <<= 1) {
            ew |= __shfl_xor_sync(0xFFFFFFFFu, ew, m);
            vw |= __shfl_xor_sync(0xFFFFFFFFu, vw, m);
        }
        if ((lane & 7) == 0 && wd < g.WPR) {
            const size_t o = (size_t)pair * plane_stride + (size_t)pr * g.WPR + wd;
            if (side == 0) {
                LA[o] = ew & vw;
                LB[o] = ~ew & vw;
            } else {
                RB[o] = ew & vw;
            }
        }
        y = yn;
        rowvalid = nvalid;
    }
}

int launch_edges_planes(const uint8_t *img1, const uint8_t *img2, int FH, int row0, int variant, const PackedGeom &g,
                        int M, double threshold, const uint32_t *lut, uint32_t *LA, uint32_t *LB, uint32_t *RB, uint8_t *edges1,
                        uint8_t *edges2, cudaStream_t s, int npairs, size_t image_stride, size_t plane_stride)
{
    dim3 block(128);
    dim3 grid((g.WPR * 8 + block.x - 1) / block.x, (g.ER + EP_ROWS - 1) / EP_ROWS, 2 * npairs);
    const bool u8 = edges1 != nullptr && edges2 != nullptr;
    // every image of the launch word-aligned, width a multiple of 4, at least two rows: no gather needed (GHOST)
    const bool regular = (g.W & 3) == 0 && FH >= 2 && ((reinterpret_cast<uintptr_t>(img1) | reinterpret_cast<uintptr_t>(img2)) & 3) == 0 &&
                         (npairs == 1 || (image_stride & 3) == 0);
#define SM_EP(V, U, G) \
    k_edges_planes<V, U, G><<<grid, block, 0, s>>>(img1, img2, FH, row0, g, M, threshold, lut, LA, LB, RB, edges1, edges2, \
                                                   image_stride, plane_stride)
    if (variant == SM_WRAP && regular) {
        if (u8) SM_EP(SM_WRAP, true, false); else SM_EP(SM_WRAP, false, false);
    } else if (variant == SM_WRAP) {
        if (u8) SM_EP(SM_WRAP, true, true); else SM_EP(SM_WRAP, false, true);
    } else if (regular) {
        if (u8) SM_EP(SM_GHOST, true, false); else SM_EP(SM_GHOST, false, false);
    } else {
        if (u8) SM_EP(SM_GHOST, true, true); else SM_EP(SM_GHOST, false, true);
    }
#undef SM_EP
    SM_CUDA(cudaGetLastError());
    return 1;
}

int launch_edge_lut(double threshold, uint32_t *lut, cudaStream_t s)
{
    k_edge_lut<<<LUT_N, 32, 0, s>>>(threshold, lut);
    k_edge_thresholds_init<<<1, 1, 0, s>>>(lut);
    k_edge_thresholds<<<LUT_N, 256, 0, s>>>(lut);
    SM_CUDA(cudaGetLastError());
    return 3;
}

size_t edge_lut_words() { return (size_t)LUT_FLAG + 1; }

void warm_edges(int variant)
{
    warm_kernel(k_edge_lut);
    warm_kernel(k_edge_thresholds_init);
    warm_kernel(k_edge_thresholds);
    if (variant == SM_WRAP) {
        warm_kernel(k_edges<uint8_t, SM_WRAP>);
        warm_kernel(k_edges<double, SM_WRAP>);
        warm_kernel(k_edges_planes<SM_WRAP, true, false>);
        warm_kernel(k_edges_planes<SM_WRAP, false, false>);
        warm_kernel(k_edges_planes<SM_WRAP, true, true>);
        warm_kernel(k_edges_planes<SM_WRAP, false, true>);
    } else {
        warm_kernel(k_edges_planes<SM_GHOST, true, false>);
        warm_kernel(k_edges_planes<SM_GHOST, false, false>);
        warm_kernel(k_edges_planes<SM_GHOST, true, true>);
        warm_kernel(k_edges_planes<SM_GHOST, false, true>);
        warm_kernel(k_edges<uint8_t, SM_GHOST>);
        warm_kernel(k_edges<double, SM_GHOST>);
    }
}

}  // namespace smb
