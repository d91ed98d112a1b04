// k_direct.cu -- the simple hot-path kernel (SM_KERNEL_DIRECT) and the debug planes.
//
// One thread per output pixel.  For every shift the (2*half+1)^2 window of the match
// image is evaluated row by row on the packed planes: a window row is at most 63 bits,
// so it is one 64-bit extract of LA, LB and RB, one LOP3-able combine and one popcount.
// This is the literal sum of addup_pixels_in_square (stereo.cu:142-155) followed by
// record_score (stereo.cu:185-192) and find_highest_scoring_shifts (stereo.cu:211-225),
// fused so that matches[] and scores[] never exist.  It is the slow, obviously-correct
// device path: the bit-sliced kernel (k_bitslice.cu) is checked against it as well as
// against the CPU oracle, and it serves geometries the fast kernel does not cover.
#include "sm_common.cuh"

namespace smb {

// 64 consecutive bits of a packed row starting at bit c (LSB first).
__device__ __forceinline__ unsigned long long extract64(const uint32_t *__restrict__ row, int c)
{
    int k = c >> 5, s = c & 31;
    uint32_t w0 = __ldg(row + k), w1 = __ldg(row + k + 1), w2 = __ldg(row + k + 2);
    uint32_t lo = __funnelshift_r(w0, w1, s);
    uint32_t hi = __funnelshift_r(w1, w2, s);
    return ((unsigned long long)hi << 32) | lo;
}

// box sum and centre match of shift i at pixel (x, band row j)
__device__ __forceinline__ void window(const HotArgs &a, int x, int j, int i, int &box, int &centre)
{
    const int half = a.g.half, n = 2 * half + 1;
    const unsigned long long mask = n >= 64 ? ~0ull : ((1ull << n) - 1ull);
    const int c0 = PADL + x - half;
    box = 0;
    centre = 0;
    for (int r = 0; r < n; r++) {
        size_t o = (size_t)(j + r) * a.g.WPR;
        unsigned long long A = extract64(a.LA + o, c0);
        unsigned long long B = extract64(a.LB + o, c0);
        unsigned long long R = extract64(a.RB + o, c0 + i);
        unsigned long long m = ((R & A) | (~R & B)) & mask;
        box += __popcll(m);
        if (r == half) centre = (int)((m >> half) & 1ull);
    }
}

// best / web of pixel x of band row j, stored as T; best may be NULL (16-bit outputs: web only).  RU: also the
// runner-up score (the second largest of the pixel's scores, best again where two shifts tie for it).  SUB: also
// web_sub, the web in sixteenths of a shift (k_bitslice.cuh, sub_frac), from the scores next to the winner: the shift
// before it, kept when it wins, and the one after it, captured when no new winner takes it
template <typename T, bool RU = false, bool SUB = false>
__device__ __forceinline__ void direct_pixel(const HotArgs &a, T *best_out, T *web_out, uint16_t *ru_out = nullptr,
                                             uint16_t *sub_out = nullptr)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int j = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= a.g.W || j >= a.g.BH) return;
    int best = 0, web = 0, ru = 0;
    int sm = 0, sp = 0, last = 0;  // SUB: s(w - 1), s(w + 1), the previous shift's score
    for (int i = 0; i < a.g.D; i++) {
        int box, centre;
        window(a, x, j, i, box, centre);
        int score = centre ? box : 0;  // record_score: only where the centre matched
        if (score >= best) {           // last equal maximum wins -> highest shift
            if (RU) ru = best;
            best = score;
            web = i + 1;
            if (SUB) sm = last;
        } else {
            if (RU) ru = max(ru, score);
            if (SUB && i == web) sp = score;  // the shift after the winner (web = winner + 1)
        }
        if (SUB) last = score;
    }
    size_t p = (size_t)(a.row0 + j) * a.g.W + x;
    if (sizeof(T) == 4 || best_out) best_out[p] = (T)best;  // (the int32 kernel always has a best)
    web_out[p] = (T)(a.M + web);  // shift i of the planes is M + i
    if (RU) ru_out[p] = (uint16_t)ru;
    if (SUB) {
        // frac = min(7, floor((16 * (s+ - s-) + den) / (2 * den))), den = 2 * best - s- - s+ >= 1; 0 at the range ends
        int frac = 0;
        if (web > 1 && web < a.g.D) {
            const int den = 2 * best - sm - sp, num = 16 * (sp - sm) + den;
            const int q = num >= 0 ? num / (2 * den) : -((-num + 2 * den - 1) / (2 * den));
            frac = min(7, q);
        }
        sub_out[p] = (uint16_t)(16 * (a.M + web) + frac);
    }
}

__global__ void __launch_bounds__(256) k_direct(HotArgs a)
{
    direct_pixel(a, static_cast<int32_t *>(a.best), static_cast<int32_t *>(a.web));
}

// the 16-bit twin (a.best may be NULL)
__global__ void __launch_bounds__(256) k_direct16(HotArgs a)
{
    direct_pixel(a, static_cast<uint16_t *>(a.best), static_cast<uint16_t *>(a.web));
}

// the 16-bit twin with the runner-up score (a.best may be NULL; runner_up may not)
__global__ void __launch_bounds__(256) k_direct16_ru(HotArgs a, uint16_t *runner_up)
{
    direct_pixel<uint16_t, true>(a, static_cast<uint16_t *>(a.best), static_cast<uint16_t *>(a.web), runner_up);
}

// the 16-bit twin with web_sub (a.best may be NULL; web_sub may not)
__global__ void __launch_bounds__(256) k_direct16_sub(HotArgs a, uint16_t *web_sub)
{
    direct_pixel<uint16_t, false, true>(a, static_cast<uint16_t *>(a.best), static_cast<uint16_t *>(a.web), nullptr,
                                        web_sub);
}

// the 16-bit twin with the runner-up and web_sub (a.best may be NULL; the other two may not)
__global__ void __launch_bounds__(256) k_direct16_ru_sub(HotArgs a, uint16_t *runner_up, uint16_t *web_sub)
{
    direct_pixel<uint16_t, true, true>(a, static_cast<uint16_t *>(a.best), static_cast<uint16_t *>(a.web), runner_up,
                                       web_sub);
}

int launch_direct(const HotArgs &a, cudaStream_t s, bool out16, uint16_t *runner_up, uint16_t *web_sub)
{
    dim3 block(32, 8);
    dim3 grid((a.g.W + block.x - 1) / block.x, (a.g.BH + block.y - 1) / block.y);
    if (runner_up && web_sub)
        k_direct16_ru_sub<<<grid, block, 0, s>>>(a, runner_up, web_sub);
    else if (web_sub)
        k_direct16_sub<<<grid, block, 0, s>>>(a, web_sub);
    else if (runner_up)
        k_direct16_ru<<<grid, block, 0, s>>>(a, runner_up);
    else if (out16)
        k_direct16<<<grid, block, 0, s>>>(a);
    else
        k_direct<<<grid, block, 0, s>>>(a);
    SM_CUDA(cudaGetLastError());
    return 1;
}

// matches[i], the unmasked box sum ("score_all-i") and scores[i] for one shift: the
// planes the reference dumps under -DDEBUG (stereo.cu:108-114,167-173,201-203).
__global__ void __launch_bounds__(256)
k_planes(HotArgs a, int shift, uint8_t *__restrict__ match, int32_t *__restrict__ score_all,
         int32_t *__restrict__ score)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int j = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= a.g.W || j >= a.g.BH) return;
    int box, centre;
    window(a, x, j, shift, box, centre);
    size_t p = (size_t)(a.row0 + j) * a.g.W + x;
    if (match) match[p] = (uint8_t)centre;
    if (score_all) score_all[p] = box;
    if (score) score[p] = centre ? box : 0;
}

int launch_planes(const HotArgs &a, int shift, uint8_t *match, int32_t *score_all, int32_t *score,
                  cudaStream_t s)
{
    dim3 block(32, 8);
    dim3 grid((a.g.W + block.x - 1) / block.x, (a.g.BH + block.y - 1) / block.y);
    k_planes<<<grid, block, 0, s>>>(a, shift, match, score_all, score);
    SM_CUDA(cudaGetLastError());
    return 1;
}

void warm_direct()
{
    warm_kernel(k_direct);
    warm_kernel(k_direct16);
    warm_kernel(k_direct16_ru);
    warm_kernel(k_direct16_sub);
    warm_kernel(k_direct16_ru_sub);
    warm_kernel(k_planes);
}

}  // namespace smb
