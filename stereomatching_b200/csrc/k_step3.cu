// k_step3.cu -- step 3 of the reference (SURVEY 8f n3) and small utilities.
//
//   fill_web_holes_step  stereo.cu:235-245   (32 launches from fill_web_holes :247-259)
//   array_min/max_gpu    util.cu:15-45       (two launches + malloc/H2D/D2H each)
//   draw_contour_map     stereo.cu:261-274
// Here: one hole-filling kernel per iteration, ONE fused min+max reduction (warp
// shuffles, one atomic pair per block) and the contour kernel.
#include <limits.h>

#include "sm_common.cuh"

namespace smb {

// web is never 0 after step 2 (every pixel gets some i+1), so the branch body never
// runs on real data (SURVEY 3.4).  The reference reads the four neighbours with the unwrapped
// IDX(x+-1, y) and without bounds checks (stereo.cu:240-243): at a row end the right neighbour is the
// first pixel of the next row (and vice versa).  That is kept; only reads that leave the array
// altogether (undefined in the reference) count as 0.
__global__ void __launch_bounds__(256)
k_fill_holes(const int32_t *__restrict__ src, int32_t *__restrict__ dst, int W, int H)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x;
    int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= W || y >= H) return;
    size_t p = (size_t)y * W + x;
    if (src[p] == 0) {
        int32_t r = p + 1 < (size_t)W * H ? src[p + 1] : 0, l = p > 0 ? src[p - 1] : 0;
        int32_t u = y + 1 < H ? src[p + W] : 0, d = y > 0 ? src[p - W] : 0;
        dst[p] = (r + u + l + d) / 4;
    }
    // cells that are not holes keep what the destination buffer already holds, exactly
    // like the reference's ping-pong between web and tmp (stereo.cu:247-259)
}

int launch_fill_web_holes_step(const int32_t *src, int32_t *dst, int W, int H, cudaStream_t s)
{
    dim3 block(64, 4);
    dim3 grid((W + block.x - 1) / block.x, (H + block.y - 1) / block.y);
    k_fill_holes<<<grid, block, 0, s>>>(src, dst, W, H);
    SM_CUDA(cudaGetLastError());
    return 1;
}

// min and max of the web in ONE launch and without a host round trip before the contour kernel:
// mm holds two (min, max) slots.  A call accumulates into slot `cur` with atomics and re-arms the OTHER slot
// for the next call; that slot's last readers (the previous call's contour kernel and device-to-host copy) are
// earlier in the stream.  Both slots are armed once at sm_create (launch_minmax_arm).
__global__ void k_minmax_arm(int32_t *mm)
{
    mm[0] = mm[2] = INT_MAX;
    mm[1] = mm[3] = INT_MIN;
}

__global__ void __launch_bounds__(256) k_minmax(const int32_t *__restrict__ a, size_t n, int32_t *mm, int cur)
{
    int32_t mn = INT_MAX, mx = INT_MIN;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
    if ((reinterpret_cast<uintptr_t>(a) & 15) == 0) {
        const int4 *a4 = reinterpret_cast<const int4 *>(a);
        for (size_t i = tid; i < n / 4; i += nth) {
            const int4 v = a4[i];
            mn = min(min(mn, v.x), min(min(v.y, v.z), v.w));
            mx = max(max(mx, v.x), max(max(v.y, v.z), v.w));
        }
        for (size_t i = (n & ~(size_t)3) + tid; i < n; i += nth) mn = min(mn, a[i]), mx = max(mx, a[i]);
    } else {
        for (size_t i = tid; i < n; i += nth) mn = min(mn, a[i]), mx = max(mx, a[i]);
    }
    mn = __reduce_min_sync(0xFFFFFFFFu, mn);
    mx = __reduce_max_sync(0xFFFFFFFFu, mx);
    __shared__ int32_t smn[8], smx[8];
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) {
        smn[w] = mn;
        smx[w] = mx;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < (int)(blockDim.x >> 5); k++) {
            mn = min(mn, smn[k]);
            mx = max(mx, smx[k]);
        }
        atomicMin(mm + 2 * cur, mn);
        atomicMax(mm + 2 * cur + 1, mx);
        if (blockIdx.x == 0) {
            mm[2 * (cur ^ 1)] = INT_MAX;
            mm[2 * (cur ^ 1) + 1] = INT_MIN;
        }
    }
}

int launch_minmax_arm(int32_t *d_minmax, cudaStream_t s)
{
    k_minmax_arm<<<1, 1, 0, s>>>(d_minmax);
    SM_CUDA(cudaGetLastError());
    return 1;
}

int launch_minmax(const int32_t *a, size_t n, int32_t *d_minmax, int cur, cudaStream_t s)
{
    int blocks = (int)((n / 4 + 255) / 256);
    if (blocks > 148 * 4) blocks = 148 * 4;
    if (blocks < 1) blocks = 1;
    k_minmax<<<blocks, 256, 0, s>>>(a, n, d_minmax, cur);
    SM_CUDA(cudaGetLastError());
    return 1;
}

// out = ((web - min) % interval) == 0 with interval = (max - min) / lines   (stereo.cu:261-285), min and max
// read from the device slot the min/max kernel filled.  A zero interval (the reference divides by zero there,
// stereo.c:265-272) writes nothing; the host sees the same min/max and reports it.
__global__ void __launch_bounds__(256)
k_contour(const int32_t *__restrict__ web, size_t n, const int32_t *__restrict__ mm, int lines,
          uint8_t *__restrict__ out)
{
    const int32_t mn = mm[0], interval = (mm[1] - mn) / lines;
    if (interval == 0) return;
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n && ((reinterpret_cast<uintptr_t>(web) & 15) | (reinterpret_cast<uintptr_t>(out) & 3)) == 0) {
        const int4 v = *reinterpret_cast<const int4 *>(web + i);
        *reinterpret_cast<uchar4 *>(out + i) =
            make_uchar4(((v.x - mn) % interval) == 0, ((v.y - mn) % interval) == 0, ((v.z - mn) % interval) == 0,
                        ((v.w - mn) % interval) == 0);
    } else {
        for (size_t k = i; k < n && k < i + 4; k++) out[k] = ((web[k] - mn) % interval) == 0;
    }
}

int launch_contour(const int32_t *web, size_t n, const int32_t *d_minmax_slot, int lines, uint8_t *out,
                   cudaStream_t s)
{
    k_contour<<<(unsigned)(((n + 3) / 4 + 255) / 256), 256, 0, s>>>(web, n, d_minmax_slot, lines, out);
    SM_CUDA(cudaGetLastError());
    return 1;
}

// four elements per thread: one 16-byte load, one 4- (uint8_t) or 8-byte (uint16_t) store
template <typename T> struct Narrow4;
template <> struct Narrow4<uint8_t> {
    using V = uchar4;
};
template <> struct Narrow4<uint16_t> {
    using V = ushort4;
};

template <typename T>
__global__ void __launch_bounds__(256)
k_narrow(const int32_t *__restrict__ src, T *__restrict__ dst, size_t n)
{
    using V = typename Narrow4<T>::V;
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n) {
        int4 v = *reinterpret_cast<const int4 *>(src + i);
        V o;
        o.x = (T)v.x, o.y = (T)v.y, o.z = (T)v.z, o.w = (T)v.w;
        *reinterpret_cast<V *>(dst + i) = o;
    } else {
        for (; i < n; i++) dst[i] = (T)src[i];
    }
}

template <typename T>
int launch_narrow(const int32_t *src, T *dst, size_t n, cudaStream_t s)
{
    size_t q = (n + 3) / 4;
    k_narrow<T><<<(unsigned)((q + 255) / 256), 256, 0, s>>>(src, dst, n);
    SM_CUDA(cudaGetLastError());
    return 1;
}
template int launch_narrow<uint8_t>(const int32_t *, uint8_t *, size_t, cudaStream_t);
template int launch_narrow<uint16_t>(const int32_t *, uint16_t *, size_t, cudaStream_t);

void warm_step3()
{
    warm_kernel(k_fill_holes);
    warm_kernel(k_minmax_arm);
    warm_kernel(k_minmax);
    warm_kernel(k_contour);
    warm_kernel(k_narrow<uint8_t>);
    warm_kernel(k_narrow<uint16_t>);
}

}  // namespace smb
