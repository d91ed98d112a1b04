// k_pack.cu -- u8 edge maps -> padded 1-bit planes LA / LB / RB (see sm_common.cuh).
//
// This is the "image upload and layout path" of the hot path: the two W*H byte maps
// become three bit planes over the band plus its halo, with the border policy of the
// variant (toroidal wrap, util.h:42-47, or zero ghost cells, ghost.h / stereo-ghost.c:
// 93-97,286-287) baked into the padding, so the main kernels carry no border logic.
// It stands in for fillup_matches' index arithmetic (stereo.cu:127-137) and for
// ghost_alloc_gpu / ghost_add_gpu (ghost.h:61-98).
//
// One thread produces one 32-bit word of each plane (32 pixels).  Interior words of
// 16-byte aligned rows take the fast path: two 128-bit loads per map and a multiply
// that gathers the low bit of 4 bytes into a nibble.  A search range that starts above zero
// (min_shift M > 0) takes k_pack_range, which reads the second map M columns further.
#include "sm_common.cuh"

namespace smb {

__device__ __forceinline__ uint32_t gather4(uint32_t v)
{
    // bytes b0..b3 in {0,1}  ->  bits 0..3
    return ((v & 0x01010101u) * 0x01020408u) >> 24;
}

__device__ __forceinline__ uint32_t gather32(const uint4 &a, const uint4 &b)
{
    return gather4(a.x) | (gather4(a.y) << 4) | (gather4(a.z) << 8) | (gather4(a.w) << 12) |
           (gather4(b.x) << 16) | (gather4(b.y) << 20) | (gather4(b.z) << 24) | (gather4(b.w) << 28);
}

template <int VARIANT>
__global__ void __launch_bounds__(128)
k_pack(const uint8_t *__restrict__ e1, const uint8_t *__restrict__ e2, int FH, int row0,
       PackedGeom g, uint32_t *__restrict__ LA, uint32_t *__restrict__ LB, uint32_t *__restrict__ RB,
       size_t edge_stride, size_t plane_stride)
{
    // Let the programmatic dependent (the main kernel, HotArgs::after_pack) be scheduled right away: it
    // waits (griddepcontrol.wait) for this grid's completion before it reads the planes, and its launch
    // latency hides behind this grid's loads.  Measured on config 2, calls back to back: 29.9 us per call
    // with the edge maps in L2 and 30.4 us with cache-cold edge maps.  Triggering at the END of this
    // kernel instead gives 29.4 / 38.4 us (and 48 instead of 52 us on config 4 with warm maps): faster
    // only as long as every call finds its inputs in L2, so the trigger stays here (a dependent under one
    // wave of CTAs is placed around this grid's still-resident CTAs; the one-pair launch shapes of the
    // main kernel were calibrated under this regime, tools/sweep_runs.py).
    asm volatile("griddepcontrol.launch_dependents;");
    e1 += blockIdx.z * edge_stride;  // one pair per grid z-slice
    e2 += blockIdx.z * edge_stride;
    LA += blockIdx.z * plane_stride;
    LB += blockIdx.z * plane_stride;
    RB += blockIdx.z * plane_stride;
    const int wd = blockIdx.x * blockDim.x + threadIdx.x;  // lane <-> word, a warp covers 32 words
    const int lane = threadIdx.x & 31;
    const int pr = blockIdx.y;
    int y = row0 - g.half + pr;
    bool rowvalid = true;
    if (VARIANT == SM_WRAP) {
        y %= FH;
        if (y < 0) y += FH;
    } else {
        rowvalid = y >= 0 && y < FH;
    }
    const uint8_t *p1 = e1 + (size_t)(rowvalid ? y : 0) * g.W;
    const uint8_t *p2 = e2 + (size_t)(rowvalid ? y : 0) * g.W;
    const int x0 = wd * 32 - PADL;
    const bool inrow = wd < g.WPR && rowvalid;
    // where the word's 32 pixels come from: in WRAP mode a padding word is an image word again
    // whenever it lands on whole in-row pixels after wrapping (always so when W is a multiple of
    // 32); in GHOST mode a word wholly outside the image is zero and needs no loads at all
    int xs = x0;
    if (VARIANT == SM_WRAP) {
        xs %= g.W;
        if (xs < 0) xs += g.W;
    }
    const bool outside = VARIANT == SM_GHOST && (x0 + 32 <= 0 || x0 >= g.W);
    const bool fast = inrow && !outside && xs >= 0 && xs + 32 <= g.W && (g.W & 15) == 0 && (xs & 15) == 0 &&
                      ((reinterpret_cast<uintptr_t>(e1) | reinterpret_cast<uintptr_t>(e2)) & 15) == 0;
    uint32_t l = 0, r = 0, v = 0;
    if (fast) {
        const uint4 *q1 = reinterpret_cast<const uint4 *>(p1 + xs);
        const uint4 *q2 = reinterpret_cast<const uint4 *>(p2 + xs);
        uint4 a0 = __ldg(q1), a1 = __ldg(q1 + 1), b0 = __ldg(q2), b1 = __ldg(q2 + 1);
        l = gather32(a0, a1);
        r = gather32(b0, b1);
        v = 0xFFFFFFFFu;
    }
    // padding / ragged / unaligned words: the whole warp builds each one with ballots,
    // lane b supplying pixel b of the word (wrapped or masked per the variant)
    uint32_t slow = __ballot_sync(0xFFFFFFFFu, inrow && !fast && !outside);
    while (slow) {
        const int k = __ffs(slow) - 1;
        slow &= slow - 1;
        int x = (wd - lane + k) * 32 - PADL + lane;
        bool ok = true;
        if (VARIANT == SM_WRAP) {
            x %= g.W;
            if (x < 0) x += g.W;
        } else {
            ok = x >= 0 && x < g.W;
        }
        const uint32_t lw = __ballot_sync(0xFFFFFFFFu, ok && (p1[ok ? x : 0] & 1));
        const uint32_t rw = __ballot_sync(0xFFFFFFFFu, ok && (p2[ok ? x : 0] & 1));
        const uint32_t vw = __ballot_sync(0xFFFFFFFFu, ok);
        if (lane == k) {
            l = lw;
            r = rw;
            v = vw;
        }
    }
    if (wd < g.WPR) {
        size_t o = (size_t)pr * g.WPR + wd;
        LA[o] = l & v;
        LB[o] = ~l & v;
        RB[o] = r & v;
    }
}

// k_pack for a search range that starts above zero (min_shift > 0): the second map is read M columns further, so
// its words have their own fast-path test, their own loads (a third 16-byte chunk and a funnel shift where the column
// is no multiple of 16) and their own ballots.  (A kernel of its own, so that k_pack -- which
// runs beside the main kernels of every min_shift 0 batch -- stays the kernel it was, instruction for instruction.)
template <int VARIANT>
__global__ void __launch_bounds__(128)
k_pack_range(const uint8_t *__restrict__ e1, const uint8_t *__restrict__ e2, int FH, int row0, PackedGeom g,
             int min_shift, uint32_t *__restrict__ LA, uint32_t *__restrict__ LB, uint32_t *__restrict__ RB,
             size_t edge_stride, size_t plane_stride)
{
    // (the programmatic dependent as in k_pack)
    asm volatile("griddepcontrol.launch_dependents;");
    e1 += blockIdx.z * edge_stride;  // one pair per grid z-slice
    e2 += blockIdx.z * edge_stride;
    LA += blockIdx.z * plane_stride;
    LB += blockIdx.z * plane_stride;
    RB += blockIdx.z * plane_stride;
    const int wd = blockIdx.x * blockDim.x + threadIdx.x;  // lane <-> word, a warp covers 32 words
    const int lane = threadIdx.x & 31;
    const int pr = blockIdx.y;
    int y = row0 - g.half + pr;
    bool rowvalid = true;
    if (VARIANT == SM_WRAP) {
        y %= FH;
        if (y < 0) y += FH;
    } else {
        rowvalid = y >= 0 && y < FH;
    }
    const uint8_t *p1 = e1 + (size_t)(rowvalid ? y : 0) * g.W;
    const uint8_t *p2 = e2 + (size_t)(rowvalid ? y : 0) * g.W;
    const int x0 = wd * 32 - PADL;
    const bool inrow = wd < g.WPR && rowvalid;
    // where the word's 32 pixels come from: in WRAP mode a padding word is an image word again
    // whenever it lands on whole in-row pixels after wrapping (always so when W is a multiple of
    // 32); in GHOST mode a word wholly outside the image is zero and needs no loads at all.
    // The second map's word starts M columns further (the search range [M, M + D)).
    const int M = min_shift;
    const int xr0 = x0 + M;
    int xs = x0, xsr = xr0;
    if (VARIANT == SM_WRAP) {
        xs %= g.W;
        if (xs < 0) xs += g.W;
        xsr %= g.W;
        if (xsr < 0) xsr += g.W;
    }
    const bool outside = VARIANT == SM_GHOST && (x0 + 32 <= 0 || x0 >= g.W);
    const bool outside_r = VARIANT == SM_GHOST && (xr0 + 32 <= 0 || xr0 >= g.W);
    const bool aligned = (g.W & 15) == 0 && ((reinterpret_cast<uintptr_t>(e1) | reinterpret_cast<uintptr_t>(e2)) & 15) == 0;
    const bool fast = inrow && !outside && xs >= 0 && xs + 32 <= g.W && (xs & 15) == 0 && aligned;
    // the second map at any column: the 16-byte chunks around it, shifted (xsr + 32 <= W and W % 16 == 0 put the
    // third chunk inside the row whenever xsr is not a multiple of 16)
    const bool fast_r = inrow && !outside_r && xsr >= 0 && xsr + 32 <= g.W && aligned;
    uint32_t l = 0, r = 0, v = 0, vr = 0;
    if (fast) {
        const uint4 *q1 = reinterpret_cast<const uint4 *>(p1 + xs);
        uint4 a0 = __ldg(q1), a1 = __ldg(q1 + 1);
        l = gather32(a0, a1);
        v = 0xFFFFFFFFu;
    }
    if (fast_r) {
        const int sh = xsr & 15;
        const uint4 *q2 = reinterpret_cast<const uint4 *>(p2 + (xsr - sh));
        uint4 b0 = __ldg(q2), b1 = __ldg(q2 + 1);
        const uint32_t lo = gather32(b0, b1);
        uint32_t hi = 0;
        if (sh) {
            const uint4 b2 = __ldg(q2 + 2);
            hi = gather4(b2.x) | (gather4(b2.y) << 4) | (gather4(b2.z) << 8) | (gather4(b2.w) << 12);
        }
        r = __funnelshift_r(lo, hi, sh);
        vr = 0xFFFFFFFFu;
    }
    // padding / ragged / unaligned words: the whole warp builds each one with ballots,
    // lane b supplying pixel b of the word (wrapped or masked per the variant)
    const bool slow_l = !fast && !outside, slow_r = !fast_r && !outside_r;
    uint32_t slow = __ballot_sync(0xFFFFFFFFu, inrow && (slow_l || slow_r));
    while (slow) {
        const int k = __ffs(slow) - 1;
        slow &= slow - 1;
        int x = (wd - lane + k) * 32 - PADL + lane, xr = x + M;
        bool ok = true, okr = true;
        if (VARIANT == SM_WRAP) {
            x %= g.W;
            if (x < 0) x += g.W;
            xr %= g.W;
            if (xr < 0) xr += g.W;
        } else {
            ok = x >= 0 && x < g.W;
            okr = xr >= 0 && xr < g.W;
        }
        const uint32_t lw = __ballot_sync(0xFFFFFFFFu, ok && (p1[ok ? x : 0] & 1));
        const uint32_t rw = __ballot_sync(0xFFFFFFFFu, okr && (p2[okr ? xr : 0] & 1));
        const uint32_t vw = __ballot_sync(0xFFFFFFFFu, ok);
        const uint32_t vrw = __ballot_sync(0xFFFFFFFFu, okr);
        if (lane == k) {
            if (slow_l) l = lw, v = vw;
            if (slow_r) r = rw, vr = vrw;
        }
    }
    if (wd < g.WPR) {
        size_t o = (size_t)pr * g.WPR + wd;
        LA[o] = l & v;
        LB[o] = ~l & v;
        RB[o] = r & vr;
    }
}

int launch_pack(const uint8_t *e1, const uint8_t *e2, int FH, int row0, int variant,
                const PackedGeom &g, int M, uint32_t *LA, uint32_t *LB, uint32_t *RB, cudaStream_t s,
                int npairs, size_t edge_stride, size_t plane_stride)
{
    // whole warps of words, no idle warps: the main kernel is scheduled as this grid's programmatic dependent
    // while these CTAs are still resident, and every warp here takes registers its CTAs would otherwise get
    const int warps = (g.WPR + 31) / 32;
    dim3 block(32 * (warps < 4 ? warps : 4));
    dim3 grid((g.WPR + block.x - 1) / block.x, g.ER, npairs);
    if (M != 0 && variant == SM_WRAP)
        k_pack_range<SM_WRAP><<<grid, block, 0, s>>>(e1, e2, FH, row0, g, M, LA, LB, RB, edge_stride, plane_stride);
    else if (M != 0)
        k_pack_range<SM_GHOST><<<grid, block, 0, s>>>(e1, e2, FH, row0, g, M, LA, LB, RB, edge_stride, plane_stride);
    else if (variant == SM_WRAP)
        k_pack<SM_WRAP><<<grid, block, 0, s>>>(e1, e2, FH, row0, g, LA, LB, RB, edge_stride, plane_stride);
    else
        k_pack<SM_GHOST><<<grid, block, 0, s>>>(e1, e2, FH, row0, g, LA, LB, RB, edge_stride, plane_stride);
    SM_CUDA(cudaGetLastError());
    return 1;
}

void warm_pack(int variant)
{
    if (variant == SM_WRAP) {
        warm_kernel(k_pack<SM_WRAP>);
        warm_kernel(k_pack_range<SM_WRAP>);
    } else {
        warm_kernel(k_pack<SM_GHOST>);
        warm_kernel(k_pack_range<SM_GHOST>);
    }
}

}  // namespace smb
