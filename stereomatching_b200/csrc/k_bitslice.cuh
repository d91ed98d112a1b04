// k_bitslice.cuh -- the fast hot-path kernel (SM_KERNEL_BITSLICE), shared by its four output families:
// k_bitslice (int32 best / web, k_bitslice.cu), k_bitslice16 (uint16_t, k_bitslice16.cu), k_bitslice_ru (uint16_t
// and the runner-up score, k_bitslice_ru.cu) and k_bitslice_sub (uint16_t and the web in sixteenths of a shift,
// k_bitslice_sub.cu).  Each translation unit instantiates one family through dispatch, so that the four compile in
// parallel.
//
// What it replaces: fillup_matches + 30x{memset, addup_pixels_in_square, record_score} +
// find_highest_scoring_shifts of the reference (stereo.cu:127-225), i.e. per pixel and per
// shift a (2*half+1)^2 box sum of the 0/1 match image, masked by the centre match, then the
// arg-max over shifts with ties to the highest shift.
//
// Formulation.  Shifts are the SIMD axis: one 32-bit word holds, for one pixel, the 1-bit
// match flags of 32 consecutive shifts ("lanes").  Counts are bit-sliced: a k-bit count for
// 32 shifts is k words (planes).  For pixel u of a row the match word is
//        M(u) = valid(u) ? (L(u) ? R[u..u+31] : ~R[u..u+31]) : 0
// where R[..] is a 32-bit funnel-shifted window of the packed right-edge row, L = LA and
// valid = LA | LB (sm_common.cuh).  The box sum is built incrementally, exactly as an
// integer running sum would be, so the counts equal the reference's direct sums:
//   pass A (horizontal): a walker slides along x keeping H(x) = sum_{|sx|<=half} M(x+sx) as a
//           KH-plane up/down counter: one word enters, one leaves, 2*KH-1 LOP3 per step.
//   pass B (vertical):   one lane per pixel column keeps V(x,y) = sum_{|sy|<=half} H(x,y+sy)
//           in PV planes; per row it ripple-adds the entering H row and ripple-subtracts
//           the leaving one.
//   WTA: bit-serial max over the 32*NW shift lanes, from the top plane down:
//           t = cand & V_p & M; if (t != 0) { cand = t; best |= 1 << p; }
//        The survivors are the shifts whose masked score equals the maximum; the highest
//        surviving lane is the reference's tie rule (last i with scores[i] == best,
//        stereo.c:212-219), and with no surviving plane at all (every score 0) cand is still
//        "all shifts", giving web = num_shifts as the reference does.
//
// Decomposition.  ONE WARP owns a strip of 32 pixel columns and a run of output rows and is
// fully autonomous (only __syncwarp while it works): it streams down its rows in blocks of RB
// rows.  Per block: pass A with the 32 lanes as walkers (lane -> segment, row, shift word; every
// walker reads its own windows of the packed rows straight from global memory, prefetched one
// block ahead; the first 2*half words of a walk are summed by a carry-save tree, csa_planes),
// the block's H rows and centre match words through shared memory (the walker -> column
// transposition), then pass B with the 32 lanes as pixel columns.
//
// The vertical window lives in TENSOR MEMORY.  Pass B needs, 2*half+1 rows later, the H planes
// of the row that leaves the window.  A lane only ever re-reads what IT stored, which is exactly
// the access pattern of tcgen05.ld/st.32x32b (thread i <-> TMEM lane i): every warp keeps a ring
// of 2*half+1 rows x NW*KH columns in its own 32 TMEM lanes, reads the leaving row back from it
// and writes the entering row over it.  Shared memory then holds one block of rows instead of a
// ring of RB + 2*half + 1 (43 KB per warp at window 21, 5 warps per SM; now 15.6 KB and 8 warps,
// bounded by the 512 TMEM columns).  A warp reaches only TMEM lanes 32*(warp%4)..+31, hence FOUR
// warps (four adjacent strips) per CTA and one allocation per CTA; the warps share nothing else.
//
// More than 32*NW shifts are processed as successive chunks over the same rows, merging (best,
// web) in place (a later chunk holds higher shifts, so it wins ties; the earlier chunks' best of
// a block's rows is prefetched before pass A).  With 32 shifts or fewer the two words of a lane
// are two pixels instead (C2, 64-column strips); with 16 or fewer every word serves two pixels, u and
// u + 16, one per half (HP).
//
// A run's first 2*half rows only fill the vertical window: a short block and then whole blocks that add
// into the sums and the ring and nothing else, in front of the whole, branch-free steady blocks.
//
// The ALU pipe binds this kernel (LOP3), so what is not bit-plane logic is kept off it: the walker's complement and
// the selects of the winner-take-all are predicated multiply-adds, the winning lane's index is a multiply-add on
// shift amounts, store addresses are one widening multiply-add on a per-lane base (FMA pipe), ring slots advance by
// compare-and-subtract (uniform datapath).  The bit-plane logic itself is written one LOP3 per term
// (tools/sass_budget.py counts what ptxas made of it).
//
// Launching.  Several pairs per launch (grid z) run in the throughput shape: runs of about 32
// windows, several waves deep.  One pair per launch takes the number of row runs a small cost
// model picks (launch_one), as the programmatic dependent of the pack kernel
// (griddepcontrol.wait below).  DESIGN.md 4.1 has the numbers.
//
// Outputs.  The winner-take-all epilogue stores best and web as OutT: int32_t, or uint16_t (web <= 512 and
// best <= 31^2 always fit), half the store bytes.  Both families always store both arrays: several 64-shift chunks
// merge through best, and a per-store "best wanted" predicate costs the 16-bit kernels registers (up to 144 bytes of
// spills at the 128 registers of the C2 + HP kernels).  A caller of the 16-bit entries who wants no best gets a scratch
// array of the context's.  Both families take the same argument (HotArgs::best / web point at OutT arrays).
#pragma once

#include <stdlib.h>

#include <type_traits>

#include "sm_common.cuh"

namespace smb {

namespace {

__host__ __device__ constexpr int bits_for(int v)
{
    int b = 0;
    while ((1 << b) <= v) b++;
    return b;
}

__host__ __device__ constexpr int pow2_at_least(int v)
{
    int p = 32;
    while (p < v) p *= 2;
    return p;
}

template <int HALF, int NW, int SEG>
constexpr bool ring_aligns();

// ALIGNED_M (the runner-up family): the centre-match ring holds a whole number of blocks, so that the RB centre rows a
// steady block reads are consecutive ring rows (see bitslice_body) -- where the larger ring costs no CTA per SM
template <int HALF, int NW, int SEG, bool ALIGNED_M = false>
struct WS {
    static constexpr int N = 2 * HALF + 1;       // window side
    static constexpr int KH = bits_for(N);       // planes of a horizontal count (<= N)
    static constexpr int PV = bits_for(N * N);   // planes of a box count (<= N*N)
    static constexpr int TW = 32;                // pixel columns per warp
    static constexpr int NSEG = TW / SEG;        // walkers per (row, word)
    static constexpr int RB = 32 / (NW * NSEG);  // rows per block: 32 walkers
    static constexpr int NR = RB;                // H rows in shared memory: one block
    static constexpr bool M_ALIGNED = [] {
        if constexpr (ALIGNED_M)
            return ring_aligns<HALF, NW, SEG>();
        else
            return false;
    }();
    static constexpr int NRM = M_ALIGNED ? (RB + HALF + 1 + RB - 1) / RB * RB : RB + HALF + 1;  // centre-match ring rows
    static constexpr int HROW = TW + 1;          // uint4 per (ring row, word); +1 staggers banks
    // words per M ring row, +stagger; two words per lane: even, so that the LDS.64 stays aligned
    static constexpr int MROW = NW == 1 ? TW + 1 : TW * NW + 2;
    static constexpr int STEPS = SEG + 2 * HALF;
    static constexpr int H5N = KH > 4 ? ((NR * NW * HROW + 3) & ~3) : 0;  // words, 16-byte multiple
    static constexpr int MQN = (NRM * MROW + 3) & ~3;                     // words, 16-byte multiple
    static constexpr size_t SMEM = (size_t)NR * NW * HROW * 16 + (size_t)H5N * 4 + (size_t)MQN * 4;  // per warp
    static constexpr int WPC = 4;                                         // warps per CTA (TMEM lane quarters)
    static constexpr size_t SMEM_CTA = WPC * SMEM + 16;                   // + the TMEM base address slot
    static constexpr int EC = NW * KH;                                    // TMEM columns per ring row
    static constexpr int TCOLS = pow2_at_least(N * EC);                   // allocation: a power of two >= 32
    static constexpr int CTAS_SMEM = (int)((227 * 1024) / (SMEM_CTA + 1024));
    static constexpr int CTAS_TMEM = 512 / TCOLS;
    // 16 warps per SM at most (measured: 12 and 16 run alike, and 16 x 128 registers is where ptxas stops spilling)
    static constexpr int CTAS_PER_SM_ = CTAS_SMEM < CTAS_TMEM ? CTAS_SMEM : CTAS_TMEM;
    static constexpr int CTAS_PER_SM = CTAS_PER_SM_ > 4 ? 4 : (CTAS_PER_SM_ < 1 ? 1 : CTAS_PER_SM_);
    // dynamic shared memory to ask for: never more co-resident CTAs than TMEM allocations fit (a CTA that cannot
    // allocate would sit on its shared memory and registers, spinning in tcgen05.alloc)
    static constexpr size_t SMEM_REQ =
        SMEM_CTA > (size_t)(227 * 1024) / (CTAS_PER_SM + 1) ? SMEM_CTA : (size_t)(227 * 1024) / (CTAS_PER_SM + 1) + 16;
    static_assert(RB >= 1 && RB * NW * NSEG == 32, "walkers must fill the warp");
    static_assert(STEPS + 32 <= 96 && STEPS < 64, "walker windows: 96 bits of RB, 64 bits of LA/LB");
    static_assert(N * EC <= 512, "the vertical window must fit one TMEM allocation");
};

// whether the centre-match ring rounded up to whole blocks leaves the CTAs per SM as they are
template <int HALF, int NW, int SEG>
constexpr bool ring_aligns()
{
    using P = WS<HALF, NW, SEG>;
    constexpr int nrm = (P::NRM + P::RB - 1) / P::RB * P::RB;
    constexpr size_t smem_cta = P::SMEM_CTA + (size_t)P::WPC * 4 * (size_t)(((nrm * P::MROW + 3) & ~3) - P::MQN);
    return (int)((227 * 1024) / (smem_cta + 1024)) >= P::CTAS_PER_SM;
}

enum { MODE_LAUNCH = 0, MODE_PREPARE = 1, MODE_TMEM_COLUMNS = 2 };

// throughput mode (several pairs per launch): a warp's run of rows, in windows
inline int throughput_run_windows()
{
#ifdef SMB_DEV
    if (getenv("SMB_TR")) return atoi(getenv("SMB_TR"));
#endif
    return 32;
}

struct BitsliceArgs {
    HotArgs h;
    int rows_per_seg;  // output rows per warp
};


// ---- tensor memory as a lane-private ring (tcgen05.ld/st.32x32b: thread i <-> TMEM lane i) ---------------------
__device__ __forceinline__ void tm_ld(uint32_t a, uint32_t &r0)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r0) : "r"(a));
}
__device__ __forceinline__ void tm_ld(uint32_t a, uint32_t &r0, uint32_t &r1)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(a));
}
__device__ __forceinline__ void tm_ld(uint32_t a, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(a));
}
__device__ __forceinline__ void tm_ld(uint32_t a, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3, uint32_t &r4,
                                      uint32_t &r5, uint32_t &r6, uint32_t &r7)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7) : "r"(a));
}
__device__ __forceinline__ void tm_st(uint32_t a, uint32_t r0)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(a), "r"(r0) : "memory");
}
__device__ __forceinline__ void tm_st(uint32_t a, uint32_t r0, uint32_t r1)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(a), "r"(r0), "r"(r1) : "memory");
}
__device__ __forceinline__ void tm_st(uint32_t a, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(r0), "r"(r1), "r"(r2), "r"(r3)
                 : "memory");
}
__device__ __forceinline__ void tm_st(uint32_t a, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3, uint32_t r4,
                                      uint32_t r5, uint32_t r6, uint32_t r7)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(a), "r"(r0),
                 "r"(r1), "r"(r2), "r"(r3), "r"(r4), "r"(r5), "r"(r6), "r"(r7)
                 : "memory");
}

// EC consecutive columns of the lane, as the power-of-two pieces the instruction offers (10 = 8 + 2, 5 = 4 + 1, ...)
template <int EC>
__device__ __forceinline__ void tm_load(uint32_t a, uint32_t (&v)[EC])
{
    static_assert(EC >= 1 && EC <= 15, "ring row of at most 15 columns");
    constexpr int o4 = EC & 8, o2 = o4 + (EC & 4), o1 = o2 + (EC & 2);
    if constexpr ((EC & 8) != 0) tm_ld(a, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
    if constexpr ((EC & 4) != 0) tm_ld(a + o4, v[o4], v[o4 + 1], v[o4 + 2], v[o4 + 3]);
    if constexpr ((EC & 2) != 0) tm_ld(a + o2, v[o2], v[o2 + 1]);
    if constexpr ((EC & 1) != 0) tm_ld(a + o1, v[o1]);
}

template <int EC>
__device__ __forceinline__ void tm_store(uint32_t a, const uint32_t (&v)[EC])
{
    constexpr int o4 = EC & 8, o2 = o4 + (EC & 4), o1 = o2 + (EC & 2);
    if constexpr ((EC & 8) != 0) tm_st(a, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
    if constexpr ((EC & 4) != 0) tm_st(a + o4, v[o4], v[o4 + 1], v[o4 + 2], v[o4 + 3]);
    if constexpr ((EC & 2) != 0) tm_st(a + o2, v[o2], v[o2 + 1]);
    if constexpr ((EC & 1) != 0) tm_st(a + o1, v[o1]);
}

// the loads are asynchronous: the registers may be used only after the wait.  The empty asm statements tie
// every loaded register to a point after the wait (volatile asm statements keep their order), so that the
// compiler cannot schedule a use above it.
template <int EC>
__device__ __forceinline__ void tm_pin(uint32_t (&v)[EC])
{
#pragma unroll
    for (int k = 0; k < EC; k++) asm volatile("" : "+r"(v[k]));
}
__device__ __forceinline__ void tm_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// x, y, z -> the 3-input function whose truth table is LUT (x = 0xF0, y = 0xCC, z = 0xAA): one LOP3
template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t x, uint32_t y, uint32_t z)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(x), "r"(y), "r"(z), "n"(LUT));
    return r;
}

// V (PV planes) += H (KH planes), ripple carry; the sum always fits PV planes.
template <int PV, int KH>
__device__ __forceinline__ void planes_add(uint32_t (&V)[PV], const uint32_t (&H)[5])
{
    uint32_t c = V[0] & H[0];
    V[0] ^= H[0];
#pragma unroll
    for (int k = 1; k < PV; k++) {
        if (k < KH) {
            uint32_t s = V[k] ^ H[k] ^ c;
            c = (V[k] & H[k]) | (c & (V[k] ^ H[k]));
            V[k] = s;
        } else {
            uint32_t s = V[k] ^ c;
            c = V[k] & c;
            V[k] = s;
        }
    }
}

// V -= H, ripple borrow; the caller guarantees V >= H lane-wise (H was added before).
template <int PV, int KH>
__device__ __forceinline__ void planes_sub(uint32_t (&V)[PV], const uint32_t (&H)[5])
{
    uint32_t b = ~V[0] & H[0];
    V[0] ^= H[0];
#pragma unroll
    for (int k = 1; k < PV; k++) {
        if (k < KH) {
            uint32_t d = V[k] ^ H[k] ^ b;
            b = (~V[k] & (H[k] | b)) | (H[k] & b);
            V[k] = d;
        } else {
            uint32_t d = V[k] ^ b;
            b = ~V[k] & b;
            V[k] = d;
        }
    }
}

// V += Hn - Ho in one ripple: d = Hn - Ho as KH planes plus a sign plane, then V += sext(d).
// 2*KH + 2*PV - 1 LOP3 instead of 2 * (2*PV - 1).  AS_WRITTEN: one LOP3 per term (left to the compiler, the terms
// are re-associated into about 23 instead of 21 per plane pair at window 9).  The kernels with several 64-shift
// chunks (MULTI) keep the compiler's form: at their 128 registers the explicit one makes them spill.
template <int PV, int KH, bool AS_WRITTEN>
__device__ __forceinline__ void planes_addsub(uint32_t (&V)[PV], const uint32_t (&Hn)[5], const uint32_t (&Ho)[5])
{
    if constexpr (AS_WRITTEN) {
        // plane k of d is added as soon as it is known (fewer live registers than all of d first)
        const uint32_t d0 = lop3<0x3C>(Hn[0], Ho[0], Ho[0]);  // Hn ^ Ho
        uint32_t b = lop3<0x0C>(Hn[0], Ho[0], Ho[0]);         // borrow: ~Hn & Ho
        uint32_t c = lop3<0xC0>(V[0], d0, d0);                // carry: V & d
        V[0] = lop3<0x3C>(V[0], d0, d0);
#pragma unroll
        for (int k = 1; k < PV; k++) {
            uint32_t x = b;  // k >= KH: lanes where Hn < Ho, d is negative and its upper planes are all ones
            if (k < KH) {
                x = lop3<0x96>(Hn[k], Ho[k], b);
                b = lop3<0x8E>(Hn[k], Ho[k], b);  // borrow: majority of ~Hn, Ho, b
            }
            const uint32_t sum = lop3<0x96>(V[k], x, c);
            if (k + 1 < PV) c = lop3<0xE8>(V[k], x, c);  // carry: majority
            V[k] = sum;
        }
    } else {
        uint32_t d[KH];
        uint32_t b = ~Hn[0] & Ho[0];
        d[0] = Hn[0] ^ Ho[0];
#pragma unroll
        for (int k = 1; k < KH; k++) {
            d[k] = Hn[k] ^ Ho[k] ^ b;
            b = (~Hn[k] & (Ho[k] | b)) | (Ho[k] & b);
        }
        const uint32_t sgn = b;  // lanes where Hn < Ho: d is negative, its upper planes are all ones
        uint32_t c = V[0] & d[0];
        V[0] ^= d[0];
#pragma unroll
        for (int k = 1; k < PV; k++) {
            const uint32_t x = k < KH ? d[k] : sgn;
            uint32_t sum = V[k] ^ x ^ c;
            c = (V[k] & x) | (c & (V[k] ^ x));
            V[k] = sum;
        }
    }
}

// What a walker needs from the packed planes of its row, as raw words: 96 bits of RB starting
// at its first pixel's first shift and 64 bits each of LA / LB starting at its first pixel
// (plus the alignment slack).  Kept raw across pass B so that the loads stay in flight; the
// funnel shifts that align them run only when the walk starts.
struct WalkRaw {
    uint32_t r[4], a[3], b[3];
};

__device__ __forceinline__ void load_walk_raw(WalkRaw &o, const HotArgs &h, int pr, int rbit, int lbit)
{
    const size_t row = (size_t)pr * h.g.WPR;
    const uint32_t *pq = h.RB + row + (rbit >> 5);
    const uint32_t *pa = h.LA + row + (lbit >> 5), *pb = h.LB + row + (lbit >> 5);
#pragma unroll
    for (int k = 0; k < 4; k++) o.r[k] = __ldg(pq + k);
#pragma unroll
    for (int k = 0; k < 3; k++) o.a[k] = __ldg(pa + k), o.b[k] = __ldg(pb + k);
}

// Sum of N one-bit words as bit planes, by carry-save adders: plane K is the parity of the N
// words of weight 2^K, reduced three at a time (a full adder is two LOP3: sum and majority),
// and every adder's carry is a word of weight 2^(K+1).  About 2 * (N - planes) LOP3 in all.
template <int N, int K>
__device__ __forceinline__ void csa_planes(const uint32_t (&a)[N], uint32_t (&P)[5])
{
    constexpr int NC = N / 2;  // carries this level produces
    uint32_t c[NC > 0 ? NC : 1];
    uint32_t acc = a[0];
#pragma unroll
    for (int i = 1; i + 1 < N; i += 2) {
        c[(i - 1) / 2] = lop3<0xE8>(acc, a[i], a[i + 1]);  // majority
        acc = lop3<0x96>(acc, a[i], a[i + 1]);             // parity
    }
    if ((N & 1) == 0) {  // one word left over: half adder
        c[NC - 1] = acc & a[N - 1];
        acc ^= a[N - 1];
    }
    P[K] = acc;
    if constexpr (NC > 0) csa_planes<NC, K + 1>(c, P);
}

// One walk of pass A.  VALID_ALL: every pixel of the walk is inside the image (always so in
// WRAP mode and away from the borders in GHOST mode), so the validity select drops out.
// The first 2*HALF match words only fill the window: they are summed by a carry-save tree
// instead of 2*HALF counter steps; from then on one word enters and one leaves per step.
template <int HALF, int NW, int SEG, bool VALID_ALL, bool HP>
__device__ __forceinline__ void walk(const uint32_t (&q)[3], const uint32_t (&lw)[2], const uint32_t (&vw)[2],
                                     uint32_t ones, uint4 *hq, uint32_t *h5, uint32_t *mq)
{
    using C = WS<HALF, NW, SEG>;
    constexpr int N = C::N, KH = C::KH, STEPS = C::STEPS;
    uint32_t P[5] = {0, 0, 0, 0, 0};
    uint32_t m[STEPS];
    const uint32_t nl[2] = {~lw[0], ~lw[1]};
    // HP: flags of pixels u (bit t of a 64-bit window) and u + 16 (bit t + 16) land on bits 0 and 16 of one
    // word; times 0xFFFF they are the two half-word masks (the multiply runs on the FMA pipe)
    auto halves = [&](const uint32_t (&x)[2], int t) {
        const uint32_t f = (t < 32 ? __funnelshift_r(x[0], x[1], t) : (x[1] >> (t - 32))) & 0x00010001u;
        return f * 0xFFFFu;
    };
    auto match_word = [&](int t) {
        const int qi = t >> 5;
        uint32_t mm = __funnelshift_r(q[qi], q[qi + 1 > 2 ? 2 : qi + 1], t & 31);
        if constexpr (HP) {
            mm ^= halves(nl, t);                      // per half: L(u) ? R : ~R
            if (!VALID_ALL) mm &= halves(vw, t);      // per half: taps outside the image count nothing
        } else {
            // L(u) ? R : ~R, the complement as a predicated multiply-add (~x == x * 0xFFFFFFFF + 0xFFFFFFFF) on the
            // FMA pipe.  `ones` is 0xFFFFFFFF that ptxas cannot see, or it turns the multiply-add into an IADD3.
            asm("{ .reg .pred p; setp.eq.u32 p, %1, 0; @p mad.lo.u32 %0, %0, %2, %2; }"
                : "+r"(mm) : "r"(lw[t >> 5] & (1u << (t & 31))), "r"(ones));
            if (!VALID_ALL && !(vw[t >> 5] & (1u << (t & 31)))) mm = 0u;  // taps outside the image count nothing
        }
        if (t >= HALF && t < HALF + SEG) mq[(t - HALF) * NW] = mm;    // centre word of pixel ws*SEG + t - HALF
        return mm;
    };
    if constexpr (HALF > 0) {
        uint32_t fill[2 * HALF];
#pragma unroll
        for (int t = 0; t < 2 * HALF; t++) fill[t] = m[t] = match_word(t);
        csa_planes<2 * HALF, 0>(fill, P);
    }
#pragma unroll
    for (int t = 2 * HALF; t < STEPS; t++) {
        const uint32_t mm = m[t] = match_word(t);
        const uint32_t mout = t >= N ? m[t - N] : 0u;
        // up/down counter: +1 where mm & ~mout, -1 where mout & ~mm; one LOP3 per term, as written (left to the
        // compiler, the terms are re-associated into more instructions)
        uint32_t c = lop3<0x24>(mm, mout, P[0]);  // (mm ^ mout) & (P[0] ^ mout)
        P[0] = lop3<0x96>(P[0], mm, mout);
#pragma unroll
        for (int k = 1; k < KH; k++) {
            const uint32_t cn = lop3<0x60>(c, P[k], mout);  // c & (P[k] ^ mout)
            P[k] ^= c;
            c = cn;
        }
        hq[t - 2 * HALF] = make_uint4(P[0], P[1], P[2], P[3]);
        if (KH > 4) h5[t - 2 * HALF] = P[4];
    }
}

// Winner-take-all of NR_ output rows at once.  The rows are independent, so interleaving
// their bit-serial chains (AND -> test -> select, PV times) gives the scheduler NR_ chains
// to overlap.  The selects are predicated multiply-adds on purpose: ptxas puts them on the
// FMA pipe, which is otherwise idle, instead of the ALU pipe that carries all the LOP3 work.
//
// AS_WRITTEN (all but the MULTI kernels, which would spill at their 128 registers): the first plane's select and
// the winning lane's index are kept off the ALU pipe too (below); otherwise ptxas makes the former three SELs per
// row and the latter two FLO, a LOP3, a max and an add.
//
// One plane of a bit-serial max: t = cand & V_p & M; if (t != 0) { cand = t; acc |= 1 << p }.  The "any lane left"
// test is folded into the same LOP3s: the predicate output of one feeds the next (lop3.or d|p), so a plane costs NW
// ALU instructions instead of NW + 1 (a separate OR-and-test); the selects are predicated multiply-adds.
template <int NW>
__device__ __forceinline__ void wta_plane(uint32_t (&cand)[NW], int &acc, const uint32_t (&Vp)[NW],
                                          const uint32_t (&M)[NW], int one, int p)
{
    if (NW == 2) {
        asm("{ .reg .pred q0, q; .reg .b32 t0, t1;\n\t"
            "lop3.or.b32 t0|q0, %0, %3, %4, 0x80, 0;\n\t"
            "lop3.or.b32 t1|q, %1, %5, %6, 0x80, q0;\n\t"
            "@q mad.lo.u32 %0, t0, %7, 0;\n\t@q mad.lo.u32 %1, t1, %7, 0;\n\t@q mad.lo.s32 %2, %7, %8, %2; }"
            : "+r"(cand[0]), "+r"(cand[NW - 1]), "+r"(acc)
            : "r"(Vp[0]), "r"(M[0]), "r"(Vp[NW - 1]), "r"(M[NW - 1]), "r"(one), "r"(1 << p));
    } else {
        asm("{ .reg .pred q; .reg .b32 t0;\n\t"
            "lop3.or.b32 t0|q, %0, %2, %3, 0x80, 0;\n\t"
            "@q mad.lo.u32 %0, t0, %4, 0;\n\t@q mad.lo.s32 %1, %4, %5, %1; }"
            : "+r"(cand[0]), "+r"(acc)
            : "r"(Vp[0]), "r"(M[0]), "r"(one), "r"(1 << p));
    }
}

// PTX shifts clamp the amount (to 32: the result is 0), which C++ shifts do not promise
__device__ __forceinline__ uint32_t shr_clamp(uint32_t x, uint32_t n)
{
    uint32_t r;
    asm("shr.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n));
    return r;
}

// The valid lanes but one of those that tie for best (cand, the survivors of the first chain, never empty): the lowest,
// c & -c over the 32*NW lanes of the row.  The negation is a multiply by all ones (`ones`, opaque to ptxas), with two
// words one 64-bit multiply: both run on the FMA pipe, and what is left is one LOP3 per word, valid ^ (c & -c).
template <int NW>
__device__ __forceinline__ void drop_one_tied(const uint32_t (&valid)[NW], const uint32_t (&cand)[NW], uint32_t ones,
                                              uint32_t (&cand2)[NW])
{
    uint32_t n[NW];
    if constexpr (NW == 2) {
        asm("{ .reg .u64 c, o, n; mov.b64 c, {%2, %3}; mov.b64 o, {%4, %4}; mul.lo.u64 n, c, o; mov.b64 {%0, %1}, n; }"
            : "=r"(n[0]), "=r"(n[1]) : "r"(cand[0]), "r"(cand[1]), "r"(ones));
    } else {
        asm("mad.lo.u32 %0, %1, %2, 0;" : "=r"(n[0]) : "r"(cand[0]), "r"(ones));
    }
#pragma unroll
    for (int w = 0; w < NW; w++) cand2[w] = lop3<0x78>(valid[w], cand[w], n[w]);  // x ^ (y & z)
}

// SUB (the sub-pixel family, k_bitslice_sub): the masked score of the lane set in nb (one lane of the NW words, or
// none), NEGATED: -sum_p [V_p & M & nb != 0] << p.  One lop3.or per word and plane, the words chained through its
// predicate output as in wta_plane; the sum is a predicated multiply-add (FMA pipe).
template <int NW, int PV>
__device__ __forceinline__ int sub_gather(const uint32_t (&V)[NW][PV], const uint32_t (&M)[NW], const uint32_t (&nb)[NW],
                                          int one)
{
    int acc = 0;
#pragma unroll
    for (int p = PV - 1; p >= 0; p--) {
        if (NW == 2) {
            asm("{ .reg .pred q0, q; .reg .b32 t0, t1;\n\t"
                "lop3.or.b32 t0|q0, %1, %2, %3, 0x80, 0;\n\t"
                "lop3.or.b32 t1|q, %4, %5, %6, 0x80, q0;\n\t"
                "@q mad.lo.s32 %0, %7, %8, %0; }"
                : "+r"(acc)
                : "r"(V[0][p]), "r"(M[0]), "r"(nb[0]), "r"(V[NW - 1][p]), "r"(M[NW - 1]), "r"(nb[NW - 1]), "r"(one),
                  "r"(-(1 << p)));
        } else {
            asm("{ .reg .pred q; .reg .b32 t0;\n\t"
                "lop3.or.b32 t0|q, %1, %2, %3, 0x80, 0;\n\t"
                "@q mad.lo.s32 %0, %4, %5, %0; }"
                : "+r"(acc) : "r"(V[0][p]), "r"(M[0]), "r"(nb[0]), "r"(one), "r"(-(1 << p)));
        }
    }
    return acc;
}

// SUB: the lanes next to the winner, from its shift amount m (31 - its bit in the word, or with two words 63 - its
// lane): nbm = lane - 1, nbp = lane + 1, empty past either end of the words.  With two words the winner's bit of each
// word is one shift each (an empty word's amount is clamped out); the rest are multiply-adds on the FMA pipe (x * 2 is
// x * one + x; x >> 1 and x >> 31 are the high words of x * 2^31 and x * 2).
template <int NW>
__device__ __forceinline__ void sub_neighbours(uint32_t m, int one, uint32_t (&nbm)[NW], uint32_t (&nbp)[NW])
{
    if constexpr (NW == 2) {
        uint32_t m32;  // m - 32, a multiply-add (an immediate add is a VIADD on the ALU pipe)
        asm("mad.lo.u32 %0, %1, %2, -32;" : "=r"(m32) : "r"(m), "r"(one));
        const uint32_t b1 = shr_clamp(0x80000000u, m), b0 = shr_clamp(0x80000000u, m32);
        // (the multipliers 2 and 2^31 come from `one`, opaque to ptxas: as immediates the high-word multiply-adds
        // become LEA.HI on the ALU pipe)
        asm("{ .reg .b32 t;\n\t"
            "mad.lo.u32 %0, %4, %6, %4;\n\t"                 // nbp0 = b0 * 2
            "mad.hi.u32 t, %4, %7, %5;\n\t"                  // b1 + (b0 >> 31)
            "mad.lo.u32 %1, %5, %6, t;\n\t"                  // nbp1 = b1 * 2 + (b0 >> 31)
            "mul.hi.u32 %3, %5, %8;\n\t"                     // nbm1 = b1 >> 1
            "mad.lo.u32 t, %5, %8, 0;\n\t"                   // b1 << 31
            "mad.hi.u32 %2, %4, %8, t; }"                    // nbm0 = (b0 >> 1) + (b1 << 31)
            : "=r"(nbp[0]), "=r"(nbp[NW - 1]), "=r"(nbm[0]), "=r"(nbm[NW - 1])
            : "r"(b0), "r"(b1), "r"(one), "r"(2 * one), "r"((uint32_t)one << 31));
    } else {
        const uint32_t b = shr_clamp(0x80000000u, m);
        asm("mad.lo.u32 %0, %2, %3, %2;\n\tmul.hi.u32 %1, %2, %4;"
            : "=r"(nbp[0]), "=r"(nbm[0]) : "r"(b), "r"(one), "r"((uint32_t)one << 31));
    }
}

// SUB: web_sub = 16 * web + frac from the winner's masked score s0 and its neighbours' NEGATED scores nsm = -s(w - 1),
// nsp = -s(w + 1).  frac is the largest f in [-8, 7] with (2f - 1) * den <= 16 * (s+ - s-), den = 2 * s0 - s- - s+,
// i.e. min(7, floor((16 * (s+ - s-) + den) / (2 * den))): a 4-step search on g = (2f - 1) * den - 16 * (s+ - s-),
// one compare per step (ISETP), everything else multiply-adds.  Where the winner is the range's first or last shift
// (web == M + 1: c1 = -(M + 2); web == M + D: c2 = M + D - 1) den gains 2^20 - 1 (the high word of 2^20 * (2^32 - 1)),
// far above 16 * |s+ - s-| <= 16 * 63^2, so f == 0 whatever the missing neighbour's lane held.  den >= 1 everywhere
// else (ties go to the highest shift: s+ < s0, s- <= s0), and f >= -8 always (|s+ - s-| <= den).
__device__ __forceinline__ int sub_frac(int s0, int nsm, int nsp, int web, int c1, int c2, int one)
{
    // (multipliers that are powers of two come from `one`, opaque to ptxas: with immediates it makes them LEAs, which
    // run on the ALU pipe)
    int ws;
    asm("{ .reg .pred p; .reg .s32 den, d2, d4, d8, d16, g, t, y;\n\t"
        "mad.lo.s32 den, %1, %7, %2;\n\t"           // s0 - s-
        "mad.lo.s32 den, %1, %7, den;\n\t"          // 2 s0 - s-
        "mad.lo.s32 den, %3, %7, den;\n\t"          // - s+
        "mad.lo.s32 y, %4, %7, %5;\n\t"             // web - (M + 2): -1 where w == M (no s-)
        "mad.hi.u32 den, y, %10, den;\n\t"          // + 2^20 - 1 there
        "mad.lo.s32 y, %4, %8, %6;\n\t"             // (M + D - 1) - web: -1 where w == M + D - 1 (no s+)
        "mad.hi.u32 den, y, %10, den;\n\t"
        "mad.lo.s32 d2, den, %7, den;\n\t"
        "mad.lo.s32 d4, d2, %7, d2;\n\t"
        "mad.lo.s32 d8, d4, %7, d4;\n\t"
        "mad.lo.s32 d16, d8, %7, d8;\n\t"
        "mad.lo.s32 y, %2, %8, %3;\n\t"             // s- - s+
        "mad.lo.s32 g, den, -17, 0;\n\t"
        "mad.lo.s32 g, y, %9, g;\n\t"               // g = -17 den - 16 (s+ - s-)
        "mad.lo.s32 %0, %4, %9, -8;\n\t"            // 16 web - 8
        "mad.lo.s32 t, d16, %7, g;\n\tsetp.le.s32 p, t, 0;\n\t@p mad.lo.s32 g, t, %7, 0;\n\t@p mad.lo.s32 %0, %7, 8, %0;\n\t"
        "mad.lo.s32 t, d8, %7, g;\n\tsetp.le.s32 p, t, 0;\n\t@p mad.lo.s32 g, t, %7, 0;\n\t@p mad.lo.s32 %0, %7, 4, %0;\n\t"
        "mad.lo.s32 t, d4, %7, g;\n\tsetp.le.s32 p, t, 0;\n\t@p mad.lo.s32 g, t, %7, 0;\n\t@p mad.lo.s32 %0, %7, 2, %0;\n\t"
        "mad.lo.s32 t, d2, %7, g;\n\tsetp.le.s32 p, t, 0;\n\t@p mad.lo.s32 %0, %7, 1, %0; }"
        : "=r"(ws)
        : "r"(s0), "r"(nsm), "r"(nsp), "r"(web), "r"(c1), "r"(c2), "r"(one), "r"(-one), "r"(16 * one), "r"(one << 20));
    return ws;
}

// What the sub-pixel family's winner-take-all hands on per row (SUB).  One chunk: ws = web_sub.  MULTI: the chunk's
// own neighbour scores of its winner (nsm / nsp, negated; 0 past the chunk's lanes) and the scores of its first and
// last lane (f / l), for the merge in bitslice_body.
struct SubOut {
    int *ws, *nsm, *nsp, *f, *l;
    int c1, c2;  // sub_frac's range ends
};

// RU (the runner-up family, k_bitslice_ru): ru[k] = the second-largest masked score of row k's lanes, i.e. the maximum
// over every valid lane but the winner's.  A second bit-serial max from the top plane down runs over the valid lanes
// but one of those that tie for best (drop_one_tied; which one does not change the value): where several lanes tie,
// one of the others survives every plane best has, so ru == best there; with one lane, ru == 0.
// SUB (the sub-pixel family): the winner's neighbours' scores gathered from V & M after the first chain (SubOut).
template <int NR_, int NW, int PV, bool AS_WRITTEN, bool RU = false, bool SUB = false>
__device__ __forceinline__ void wta(const uint32_t (&V)[NR_][NW][PV], const uint32_t (&M)[NR_][NW],
                                    const uint32_t (&valid)[NW], int one, int base, int (&best)[NR_], int (&web)[NR_],
                                    int *ru = nullptr, const SubOut *so = nullptr)
{
    uint32_t cand[NR_][NW];
#pragma unroll
    for (int k = 0; k < NR_; k++) {
        best[k] = 0;
        if (!AS_WRITTEN) {
#pragma unroll
            for (int w = 0; w < NW; w++)
                asm("mad.lo.u32 %0, %1, %2, 0;" : "=r"(cand[k][w]) : "r"(valid[w]), "r"(one));
        }
    }
#pragma unroll
    for (int p = PV - 1; p >= 0; p--) {
#pragma unroll
        for (int k = 0; k < NR_; k++) {
            // t = cand & V_p & M with the "any lane left" test folded into the same LOP3s: the
            // predicate output of one feeds the next (lop3.or d|p), so a plane costs NW ALU
            // instructions instead of NW + 1 (a separate OR-and-test)
            if (AS_WRITTEN && p == PV - 1) {
                // first plane, cand = valid: cand = q ? t : valid.  Without a lane left t is 0, so that is t, plus
                // valid where !q: a predicated multiply-add on t's own register.  (A copy of valid overwritten where
                // q is what ptxas turns into a SEL on the ALU pipe.)
                if (NW == 2) {
                    asm("{ .reg .pred q0, q;\n\t"
                        "lop3.or.b32 %0|q0, %3, %4, %5, 0x80, 0;\n\t"
                        "lop3.or.b32 %1|q, %6, %7, %8, 0x80, q0;\n\t"
                        "@!q mad.lo.u32 %0, %3, %9, %0;\n\t@!q mad.lo.u32 %1, %6, %9, %1;\n\t"
                        "@q mad.lo.s32 %2, %9, %10, %2; }"
                        : "=r"(cand[k][0]), "=r"(cand[k][NW - 1]), "+r"(best[k])
                        : "r"(valid[0]), "r"(V[k][0][p]), "r"(M[k][0]), "r"(valid[NW - 1]), "r"(V[k][NW - 1][p]),
                          "r"(M[k][NW - 1]), "r"(one), "r"(1 << p));
                } else {
                    asm("{ .reg .pred q;\n\t"
                        "lop3.or.b32 %0|q, %2, %3, %4, 0x80, 0;\n\t"
                        "@!q mad.lo.u32 %0, %2, %5, %0;\n\t@q mad.lo.s32 %1, %5, %6, %1; }"
                        : "=r"(cand[k][0]), "+r"(best[k])
                        : "r"(valid[0]), "r"(V[k][0][p]), "r"(M[k][0]), "r"(one), "r"(1 << p));
                }
            } else {
                uint32_t Vp[NW];
#pragma unroll
                for (int w = 0; w < NW; w++) Vp[w] = V[k][w][p];
                wta_plane<NW>(cand[k], best[k], Vp, M[k], one, p);
            }
        }
    }
    uint32_t cand2[NR_][NW];  // RU: the valid lanes but one of those that tie for best
#pragma unroll
    for (int k = 0; k < NR_; k++) {
        // web = base + the highest surviving lane; a later word holds higher shifts.  m = 32 * NW - 1 - lane, from
        // the shift amounts (31 - highest bit) of the words: with two words, that of word 1 if it has a lane, else
        // 32 + that of word 0, which is one unsigned min, since an empty word's shift amount is 0xFFFFFFFF (and if
        // word 0 is empty, word 1 is not: 0xFFFFFFFF + 32 wraps to 31, not below word 1's).  base + 32 * NW - 1 - m
        // is a multiply-add by -one: the FMA pipe.
        if (!AS_WRITTEN) {
            // the bit index of an empty word is -1, and -1 ^ 32 stays negative, so one signed max picks the word
            int idx = 31 - __clz(cand[k][0]);
            if (NW == 2) idx = max(idx, (31 - __clz(cand[k][NW - 1])) ^ 32);
            web[k] = base + idx;
            if constexpr (RU) drop_one_tied<NW>(valid, cand[k], (uint32_t)-one, cand2[k]);
            if constexpr (SUB) {
                // the chunk merge (MULTI) resolves what lies outside this chunk's lanes
                uint32_t nbm[NW], nbp[NW];
                sub_neighbours<NW>((uint32_t)(32 * NW - 1 - idx), one, nbm, nbp);
                so->nsm[k] = sub_gather<NW, PV>(V[k], M[k], nbm, one);
                so->nsp[k] = sub_gather<NW, PV>(V[k], M[k], nbp, one);
                const uint32_t first[1] = {(uint32_t)one}, last[1] = {0x80000000u};
                const uint32_t m0[1] = {M[k][0]}, m1[1] = {M[k][NW - 1]};
                so->f[k] = -sub_gather<1, PV>(reinterpret_cast<const uint32_t(&)[1][PV]>(V[k][0]), m0, first, one);
                so->l[k] = -sub_gather<1, PV>(reinterpret_cast<const uint32_t(&)[1][PV]>(V[k][NW - 1]), m1, last, one);
            }
            continue;
        }
        uint32_t m, m1;
        asm("bfind.shiftamt.u32 %0, %1;" : "=r"(m) : "r"(cand[k][0]));
        if (NW == 2) {
            asm("bfind.shiftamt.u32 %0, %1;" : "=r"(m1) : "r"(cand[k][NW - 1]));
            m = min(m1, m + 32u);
        }
        asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(web[k]) : "r"(m), "r"(-one), "r"(base + 32 * NW - 1));
        if constexpr (RU) {
            if constexpr (NW == 2) {
                drop_one_tied<NW>(valid, cand[k], (uint32_t)-one, cand2[k]);
            } else {
                // one word (also the chains of C2 and HP): the winner's own bit, from its shift amount m (fewer
                // registers there than the negation, which at 128 registers made some of those kernels spill)
                cand2[k][0] = lop3<0x30>(valid[0], shr_clamp(0x80000000u, m), 0u);  // valid & ~bit
            }
        }
        if constexpr (SUB) {
            uint32_t nbm[NW], nbp[NW];
            sub_neighbours<NW>(m, one, nbm, nbp);
            const int nsm = sub_gather<NW, PV>(V[k], M[k], nbm, one), nsp = sub_gather<NW, PV>(V[k], M[k], nbp, one);
            so->ws[k] = sub_frac(best[k], nsm, nsp, web[k], so->c1, so->c2, one);
        }
    }
    if constexpr (RU) {
#pragma unroll
        for (int k = 0; k < NR_; k++) ru[k] = 0;
#pragma unroll
        for (int p = PV - 1; p >= 0; p--) {
#pragma unroll
            for (int k = 0; k < NR_; k++) {
                uint32_t Vp[NW];
#pragma unroll
                for (int w = 0; w < NW; w++) Vp[w] = V[k][w][p];
                wta_plane<NW>(cand2[k], ru[k], Vp, M[k], one, p);
            }
        }
    }
}

// lane_base[row * row_bytes / 4 + OFF] = v where `on`: lane_base is the lane's own column of the output array, so the
// address is ONE widening multiply-add with a per-thread addend (IMAD.WIDE on the FMA pipe, which has room) and the
// column offset rides in the store's immediate field -- no shift / add / add-with-carry on the ALU pipe, which
// binds this kernel.
// (uint16_t: the store takes the low half of v's register.)
template <int OFF>
__device__ __forceinline__ void store_if(int32_t *lane_base, int row, int row_bytes, int v, bool on)
{
    asm volatile(
        "{ .reg .pred q; .reg .u64 ad; setp.ne.s32 q, %4, 0; mad.wide.s32 ad, %1, %2, %0; @q st.global.b32 [ad+%5], %3; }" ::"l"(
            lane_base),
        "r"(row), "r"(row_bytes), "r"(v), "r"((int)on), "n"(4 * OFF)
        : "memory");
}
template <int OFF>
__device__ __forceinline__ void store_if(uint16_t *lane_base, int row, int row_bytes, int v, bool on)
{
    asm volatile(
        "{ .reg .pred q; .reg .u64 ad; setp.ne.s32 q, %4, 0; mad.wide.s32 ad, %1, %2, %0; @q st.global.b16 [ad+%5], %3; }" ::"l"(
            lane_base),
        "r"(row), "r"(row_bytes), "r"(v), "r"((int)on), "n"(2 * OFF)
        : "memory");
}

// C2 ("column pairs", for num_shifts <= 32): the NW = 2 words of a lane are not two shift words of one pixel but
// the one shift word of TWO pixels, columns x and x + 32 of a 64-column strip.  Rings, walkers and adders are the
// two-word machinery unchanged; only the column of word w, the shift base and the winner-take-all (one per word)
// differ.  It runs 32-shift problems at the per-word cost of the two-word kernel (8-row blocks, 17-row rings at
// window 9) instead of the one-word kernel's 16-row blocks.
//
// HP ("half-word pairs", for num_shifts <= 16): a 32-bit match word of pixel u is R[u .. u+31], so its upper half IS
// the 16-shift match word of pixel u + 16.  One word then serves TWO pixels, u and u + 16: walkers, counters, rings
// and adders are unchanged (bit lanes never interact); only the complement / validity masks of a match word are
// per half, the winner-take-all runs one chain per half, and lane l of a strip stands for the pixel columns
// 32*(l/16) + l%16 and that + 16 (so a walker's 16-pixel segment covers 32 columns and a strip is twice as wide).
//
// The body of the kernel families; OutT (int32_t or uint16_t) is the type of the stored best and web.  Pair z's
// outputs are z * best_stride (best) and z * out_stride (web, runner-up, web_sub) elements further.  RU (k_bitslice_ru,
// 16-bit): the runner-up score goes to out_ru as well.  SUB (k_bitslice_sub, 16-bit): web_sub goes to out_ws, and MULTI
// carries one u16 per pixel between chunks in out_carry (see put).
template <typename OutT, int HALF, int NW, int SEG, bool MULTI, bool C2, bool HP, bool RU = false, bool SUB = false>
__device__ __forceinline__ void bitslice_body(BitsliceArgs a, OutT *out_best, OutT *out_web, size_t best_stride,
                                              uint16_t *out_ru = nullptr, uint16_t *out_ws = nullptr,
                                              uint16_t *out_carry = nullptr)
{
    using C = WS<HALF, NW, SEG, (RU || SUB) && !C2 && !HP>;  // (C2 / HP: the aligned ring costs them registers and spills)
    constexpr int N = C::N, KH = C::KH, PV = C::PV, TW = C::TW, RB = C::RB, NR = C::NR, NRM = C::NRM;
    constexpr int HROW = C::HROW, MROW = C::MROW, STEPS = C::STEPS, EC = C::EC, WPC = C::WPC;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = (int)(threadIdx.x >> 5);  // one strip per warp; the warps of a CTA share nothing but
    const int lane = threadIdx.x & 31;         // the TMEM allocation
    unsigned char *smem_w = smem_raw + 16 + (size_t)warp * C::SMEM;
    uint4 *Hq = reinterpret_cast<uint4 *>(smem_w);                     // [NR][NW][HROW]
    uint32_t *H5 = reinterpret_cast<uint32_t *>(Hq + NR * NW * HROW);  // [NR][NW][HROW] (KH == 5)
    uint32_t *Mq = H5 + C::H5N;                                        // [NRM][MROW], word (x, w) at x*NW + w

    // one TMEM allocation per CTA (warp 0 allocates, everybody reads the address after a barrier);
    // this warp's ring row s is columns [s*EC, (s+1)*EC) of its own 32 lanes
    uint32_t tring = 0;
    {
        uint32_t *slot = reinterpret_cast<uint32_t *>(smem_raw);
        if (warp == 0) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                             (uint32_t)__cvta_generic_to_shared(slot)),
                         "r"((uint32_t)C::TCOLS)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tring = *slot + ((uint32_t)(warp * 32) << 16);
    }

    // one pair per grid z-slice
    a.h.LA += blockIdx.z * a.h.plane_stride;
    a.h.LB += blockIdx.z * a.h.plane_stride;
    a.h.RB += blockIdx.z * a.h.plane_stride;
    static_assert(std::is_same<OutT, int32_t>::value || std::is_same<OutT, uint16_t>::value, "int32 or 16-bit outputs");
    out_best += blockIdx.z * best_stride;
    out_web += blockIdx.z * a.h.out_stride;
    static_assert(!RU || std::is_same<OutT, uint16_t>::value, "runner-up: 16-bit outputs only");
    if constexpr (RU) out_ru += blockIdx.z * a.h.out_stride;
    static_assert(!SUB || (std::is_same<OutT, uint16_t>::value && !RU), "sub-pixel: 16-bit outputs, no runner-up");
    if constexpr (SUB) {
        out_ws += blockIdx.z * a.h.out_stride;
        if (MULTI) out_carry += blockIdx.z * a.h.out_stride;
    }
    const PackedGeom &g = a.h.g;
    static_assert(!C2 || (NW == 2 && !MULTI), "column pairs: two words, one 32-shift chunk");
    static_assert(!HP || (!MULTI && SEG == 16 && (C2 || NW == 1)), "half-word pairs: one chunk, 16-pixel segments");
    constexpr int PW = HP ? 2 : 1;                    // pixels per word
    constexpr int WCOLS = TW * PW;                    // pixel columns one word of all 32 lanes covers
    constexpr int SCOLS = WCOLS * (C2 ? NW : 1);      // pixel columns per strip
    const int x0 = (blockIdx.x * WPC + warp) * SCOLS;
    const int ja = blockIdx.y * a.rows_per_seg;
    const int jb = min(g.BH, ja + a.rows_per_seg);
    const int ximg = HP ? x0 + 32 * (lane >> 4) + (lane & 15) : x0 + lane;
    const bool store_ok = ximg < g.W;
    const bool store_ok2 = ximg + TW < g.W;  // C2: the lane's second pixel
    const int nchunks = MULTI ? (g.D + 32 * NW - 1) / (32 * NW) : 1;
    const int last_pr = jb + 2 * HALF;   // padded rows [ja, last_pr) feed this warp
    const int first_out = ja + 2 * HALF; // the padded row that completes output row ja

    // walker role of this lane
    const int ws = lane / (NW * RB), wl = lane - ws * (NW * RB);
    const int wr = wl / NW, ww = wl - wr * NW;
    const int lbit = PADL + x0 + ws * SEG * PW - HALF + (C2 ? WCOLS * ww : 0);  // first pixel of the walk, as a bit of LA / LB

    auto load_h = [&](int slot, int w, uint32_t (&h)[5]) {
        const uint4 qv = Hq[(slot * NW + w) * HROW + lane];
        h[0] = qv.x, h[1] = qv.y, h[2] = qv.z, h[3] = qv.w;
        h[4] = KH > 4 ? H5[(slot * NW + w) * HROW + lane] : 0u;
    };
    // the KH planes of both words of a ring row <-> EC consecutive TMEM columns
    auto to_cols = [&](const uint32_t (&h)[NW][5], uint32_t (&e)[EC]) {
#pragma unroll
        for (int w = 0; w < NW; w++)
#pragma unroll
            for (int k = 0; k < KH; k++) e[w * KH + k] = h[w][k];
    };
    auto from_cols = [&](const uint32_t (&e)[EC], uint32_t (&h)[NW][5]) {
#pragma unroll
        for (int w = 0; w < NW; w++)
#pragma unroll
            for (int k = 0; k < 5; k++) h[w][k] = k < KH ? e[w * KH + k] : 0u;
    };

    // launched as the pack kernel's programmatic dependent (HotArgs::after_pack): everything above
    // overlapped its tail; the packed planes are complete and visible only after this point
    asm volatile("griddepcontrol.wait;" ::: "memory");

    // a warp whose strip lies beyond the frame (the last CTA of a row of strips) or whose run is empty has
    // nothing to do but to take part in the barriers of the TMEM allocation
    const bool has_work = ja < jb && x0 < g.W;
    for (int chunk = 0; has_work && chunk < nchunks; chunk++) {
        const int wg0 = chunk * NW;  // first 32-shift word of this chunk
        const int rbit = lbit + 32 * (wg0 + (C2 ? 0 : ww));
        uint32_t valid[NW];
#pragma unroll
        for (int w = 0; w < NW; w++) {
            int lanes = g.D - 32 * (wg0 + (C2 ? 0 : w));
            valid[w] = lanes >= 32 ? 0xFFFFFFFFu : (lanes <= 0 ? 0u : ((1u << lanes) - 1u));
        }
        // HP: the shift lanes of the lower and of the upper pixel of a word (num_shifts <= 16)
        const uint32_t valid_lo = valid[0] & 0xFFFFu, valid_hi = valid_lo << 16;
        const int one = valid[0] ? 1 : g.W;  // always 1 (word 0 of a chunk has lanes); opaque to ptxas
        uint32_t V[NW][PV];
#pragma unroll
        for (int w = 0; w < NW; w++) {
#pragma unroll
            for (int p = 0; p < PV; p++) V[w][p] = 0;
        }
        {
            // ring row N-1 stands for padded row ja-1: all zero, so that the first output row may subtract it
            // like any other
            uint32_t z[EC];
#pragma unroll
            for (int k = 0; k < EC; k++) z[k] = 0u;
            tm_wait_st();  // (the previous chunk's last rows)
            tm_store<EC>(tring + (N - 1) * EC, z);
        }
        int tslot = 0;  // ring row of padded row p0 (= (p0 - ja) mod N)

        WalkRaw in = {};
        if (ja + wr < last_pr) load_walk_raw(in, a.h, ja + wr, rbit, lbit);
        // centre-match ring slot of padded row p0.  C::M_ALIGNED (RU): started so that the centre rows of every steady block begin at a
        // multiple of RB (p0 - ja is (2*HALF) % RB plus whole blocks there), and with NRM a multiple of RB they never wrap
        // within the block: one ring slot per block instead of a compare-and-select per row (which ptxas keeps on the
        // ALU pipe in this family)
        int mslot0 = C::M_ALIGNED ? ((HALF - (2 * HALF) % RB) % RB + RB) % RB : 0;
        // next output row of the frame, and the lane's own column of the two output arrays
        int orow = a.h.row0 + ja;
        const int row_bytes = (int)sizeof(OutT) * g.W;
        OutT *const lane_best = out_best + ximg, *const lane_web = out_web + ximg;
        uint16_t *const lane_ru = RU ? out_ru + ximg : nullptr;
        uint16_t *const lane_ws = SUB ? out_ws + ximg : nullptr;
        uint16_t *const lane_carry = SUB && MULTI ? out_carry + ximg : nullptr;
        // SUB: sub_frac's range ends, web == M + 1 and web == M + D
        const int sub_c1 = -(a.h.M + 2), sub_c2 = a.h.M + g.D - 1;

        // store a finished row (best, web[, runner-up]) and advance the output pointers.  MULTI: a later chunk holds
        // higher shifts, so it wins ties against what the earlier chunks left in `best` (prev).  The runner-up of the
        // shifts so far is the larger of the loser's best and the winner's runner-up (prev_ru: the earlier chunks')
        //
        // SUB, one chunk: ws is web_sub.  MULTI: between chunks a pixel's winner is SETTLED (web_sub final; the carry
        // holds the score of the previous chunk's last lane) or PENDING (on its chunk's last lane, whose score is then
        // best itself; web_sub holds 0, which no final value is, and the carry the winner's s-).  A winner on this
        // chunk's first lane takes s- from there; a pending one that survives this chunk takes s+ = its first lane (f).
        auto put = [&](int best, int web, int prev, int ru, int prev_ru, int ws, int nsm, int nsp, int f, int l,
                       int prev_ws, int prev_carry) {
            bool st = store_ok;
            const bool wins = !MULTI || chunk == 0 || best >= prev;
            if (MULTI && chunk != 0) st = st && wins;
            store_if<0>(lane_best, orow, row_bytes, best, st);
            store_if<0>(lane_web, orow, row_bytes, web, st);
            if constexpr (RU) {
                if (MULTI) ru = max(min(best, prev), best >= prev ? ru : prev_ru);  // (chunk 0: prev == prev_ru == 0)
                store_if<0>(lane_ru, orow, row_bytes, ru, store_ok);
            }
            if constexpr (SUB) {
                if constexpr (MULTI) {
                    const int cbase = a.h.M + 32 * wg0;  // web of this chunk's first lane is cbase + 1
                    const bool pending_prev = chunk != 0 && prev_ws == 0;
                    const int last_prev = pending_prev ? prev : prev_carry;  // score of the previous chunk's last lane
                    const bool pending = wins && web == cbase + 32 * NW && chunk + 1 < nchunks;
                    const int s0 = wins ? best : prev, w = wins ? web : cbase;
                    const int nm = wins ? (chunk != 0 && web == cbase + 1 ? -last_prev : nsm) : -prev_carry;
                    const int np = wins ? nsp : -f;
                    const int wsn = sub_frac(s0, nm, np, w, sub_c1, sub_c2, one);
                    ws = pending ? 0 : (wins || pending_prev ? wsn : prev_ws);
                    store_if<0>(lane_carry, orow, row_bytes, pending ? -nsm : l, store_ok);
                }
                store_if<0>(lane_ws, orow, row_bytes, ws, store_ok);
            }
            orow++;
        };
        // what the earlier chunks left in `best` for the next output row + k (only read where it is stored)
        auto load_prev = [&](int k) {
            int v = 0;
            if (MULTI && chunk != 0 && store_ok) v = lane_best[(size_t)(orow + k) * g.W];
            return v;
        };
        // ... and in the runner-up
        auto load_prev_ru = [&](int k) {
            int v = 0;
            if (RU && MULTI && chunk != 0 && store_ok) v = lane_ru[(size_t)(orow + k) * g.W];
            return v;
        };
        // ... and (SUB) in web_sub and the carry
        auto load_prev_ws = [&](int k) {
            int v = 0;
            if (SUB && MULTI && chunk != 0 && store_ok) v = lane_ws[(size_t)(orow + k) * g.W];
            return v;
        };
        auto load_prev_carry = [&](int k) {
            int v = 0;
            if (SUB && MULTI && chunk != 0 && store_ok) v = lane_carry[(size_t)(orow + k) * g.W];
            return v;
        };
        // C2: the two pixels of a lane (columns ximg and ximg + 32) of one finished row
        auto put2 = [&](int best0, int web0, int best1, int web1, int ru0, int ru1, int ws0, int ws1) {
            store_if<0>(lane_best, orow, row_bytes, best0, store_ok);
            store_if<0>(lane_web, orow, row_bytes, web0, store_ok);
            store_if<TW>(lane_best, orow, row_bytes, best1, store_ok2);
            store_if<TW>(lane_web, orow, row_bytes, web1, store_ok2);
            if constexpr (RU) {
                store_if<0>(lane_ru, orow, row_bytes, ru0, store_ok);
                store_if<TW>(lane_ru, orow, row_bytes, ru1, store_ok2);
            }
            if constexpr (SUB) {
                store_if<0>(lane_ws, orow, row_bytes, ws0, store_ok);
                store_if<TW>(lane_ws, orow, row_bytes, ws1, store_ok2);
            }
            orow++;
        };
        // HP: the 2 * NW pixels of a lane of one finished row: word w covers columns ximg + w * WCOLS and that + 16
        auto put_hp = [&](const int *bl, const int *wl, const int *bh, const int *wh, const int *rl, const int *rh,
                          const int *sl, const int *sh) {
            store_if<0>(lane_best, orow, row_bytes, bl[0], ximg < g.W);
            store_if<0>(lane_web, orow, row_bytes, wl[0], ximg < g.W);
            store_if<16>(lane_best, orow, row_bytes, bh[0], ximg + 16 < g.W);
            store_if<16>(lane_web, orow, row_bytes, wh[0], ximg + 16 < g.W);
            if constexpr (RU) {
                store_if<0>(lane_ru, orow, row_bytes, rl[0], ximg < g.W);
                store_if<16>(lane_ru, orow, row_bytes, rh[0], ximg + 16 < g.W);
            }
            if constexpr (SUB) {
                store_if<0>(lane_ws, orow, row_bytes, sl[0], ximg < g.W);
                store_if<16>(lane_ws, orow, row_bytes, sh[0], ximg + 16 < g.W);
            }
            if constexpr (NW == 2) {
                store_if<WCOLS>(lane_best, orow, row_bytes, bl[NW - 1], ximg + WCOLS < g.W);
                store_if<WCOLS>(lane_web, orow, row_bytes, wl[NW - 1], ximg + WCOLS < g.W);
                store_if<WCOLS + 16>(lane_best, orow, row_bytes, bh[NW - 1], ximg + WCOLS + 16 < g.W);
                store_if<WCOLS + 16>(lane_web, orow, row_bytes, wh[NW - 1], ximg + WCOLS + 16 < g.W);
                if constexpr (RU) {
                    store_if<WCOLS>(lane_ru, orow, row_bytes, rl[NW - 1], ximg + WCOLS < g.W);
                    store_if<WCOLS + 16>(lane_ru, orow, row_bytes, rh[NW - 1], ximg + WCOLS + 16 < g.W);
                }
                if constexpr (SUB) {
                    store_if<WCOLS>(lane_ws, orow, row_bytes, sl[NW - 1], ximg + WCOLS < g.W);
                    store_if<WCOLS + 16>(lane_ws, orow, row_bytes, sh[NW - 1], ximg + WCOLS + 16 < g.W);
                }
            }
            orow++;
        };
        // winner-take-all of G rows held as Vs[G][NW][PV] / Ms[G][NW], then the stores: one WTA over both words
        // of a pixel, or (C2) one per word, the 2*G single-word chains interleaved like rows, or (HP) one per
        // half word: the lower halves of all words first, then the upper halves
        auto finish_rows = [&](auto gtag, const auto &Vs, const auto &Ms, const int *prev, const int *prev_ru,
                               const int *prev_ws, const int *prev_carry) {
            constexpr int G_ = decltype(gtag)::value;
            if constexpr (HP) {
                constexpr int NCH = G_ * NW;
                uint32_t V1[NCH][1][PV], M1[NCH][1];
#pragma unroll
                for (int k = 0; k < G_; k++)
#pragma unroll
                    for (int w = 0; w < NW; w++) {
                        M1[k * NW + w][0] = Ms[k][w];
#pragma unroll
                        for (int p = 0; p < PV; p++) V1[k * NW + w][0][p] = Vs[k][w][p];
                    }
                const uint32_t vl1[1] = {valid_lo}, vh1[1] = {valid_hi};
                // the upper half's lanes are 16..31 of the word: web = M + lane - 16 + 1
                int bl[NCH], wl[NCH], bh[NCH], wh[NCH], rl[NCH], rh[NCH], sl[NCH], sh[NCH];
                const SubOut sol = {sl, nullptr, nullptr, nullptr, nullptr, sub_c1, sub_c2};
                const SubOut soh = {sh, nullptr, nullptr, nullptr, nullptr, sub_c1, sub_c2};
                wta<NCH, 1, PV, !MULTI, RU, SUB>(V1, M1, vl1, one, a.h.M + 1, bl, wl, rl, &sol);
                wta<NCH, 1, PV, !MULTI, RU, SUB>(V1, M1, vh1, one, a.h.M + 1 - 16, bh, wh, rh, &soh);
#pragma unroll
                for (int k = 0; k < G_; k++)
                    put_hp(bl + k * NW, wl + k * NW, bh + k * NW, wh + k * NW, rl + k * NW, rh + k * NW, sl + k * NW,
                           sh + k * NW);
            } else if constexpr (!C2) {
                int best[G_], web[G_], ru[G_], ws[G_], nsm[G_], nsp[G_], f[G_], l[G_];
                const SubOut so = {ws, nsm, nsp, f, l, sub_c1, sub_c2};
                wta<G_, NW, PV, !MULTI, RU, SUB>(Vs, Ms, valid, one, a.h.M + 32 * wg0 + 1, best, web, ru, &so);
#pragma unroll
                for (int k = 0; k < G_; k++)
                    put(best[k], web[k], prev[k], ru[k], prev_ru[k], ws[k], nsm[k], nsp[k], f[k], l[k], prev_ws[k],
                        prev_carry[k]);
            } else {
                uint32_t V1[2 * G_][1][PV], M1[2 * G_][1];
#pragma unroll
                for (int k = 0; k < G_; k++)
#pragma unroll
                    for (int w = 0; w < 2; w++) {
                        M1[2 * k + w][0] = Ms[k][w];
#pragma unroll
                        for (int p = 0; p < PV; p++) V1[2 * k + w][0][p] = Vs[k][w][p];
                    }
                const uint32_t valid1[1] = {valid[0]};
                int best[2 * G_], web[2 * G_], ru[2 * G_], ws[2 * G_];
                const SubOut so = {ws, nullptr, nullptr, nullptr, nullptr, sub_c1, sub_c2};
                wta<2 * G_, 1, PV, !MULTI, RU, SUB>(V1, M1, valid1, one, a.h.M + 1, best, web, ru, &so);
#pragma unroll
                for (int k = 0; k < G_; k++)
                    put2(best[2 * k], web[2 * k], best[2 * k + 1], web[2 * k + 1], ru[2 * k], ru[2 * k + 1], ws[2 * k],
                         ws[2 * k + 1]);
            }
        };
        auto load_m = [&](int mslot_c, uint32_t (&M)[NW]) {
#pragma unroll
            for (int w = 0; w < NW; w++) M[w] = Mq[mslot_c * MROW + lane * NW + w];
        };
        // ring index helpers: x in [0, 2n) -> x mod n, and x in [-n, n) -> x mod n
        auto wrap_hi = [](int x, int n) { return x >= n ? x - n : x; };
        auto wrap_m = [&](int ms) { return ms < 0 ? ms + NRM : (ms >= NRM ? ms - NRM : ms); };
        // ring row of x = tslot + r, tslot < N, r < RB
        auto wrap_t = [&](int x) { return N >= RB ? wrap_hi(x, N) : x % N; };

        // ---------------- pass A: 32 walkers over the nrows rows of the block at padded row p0 ----------------
        auto pass_a = [&](int p0, int nrows) {
            {
                const bool active = wr < nrows;
                const int slot = wr;
                int mslot = mslot0 + wr;
                mslot = mslot >= NRM ? mslot - NRM : mslot;
                uint4 *hq = Hq + (slot * NW + ww) * HROW + ws * SEG;
                uint32_t *h5 = H5 + (slot * NW + ww) * HROW + ws * SEG;
                uint32_t *mq = Mq + mslot * MROW + (ws * SEG) * NW + ww;
                const int rs = rbit & 31, ls = lbit & 31;
                const uint32_t q[3] = {__funnelshift_r(in.r[0], in.r[1], rs), __funnelshift_r(in.r[1], in.r[2], rs),
                                       __funnelshift_r(in.r[2], in.r[3], rs)};
                const uint32_t lw[2] = {__funnelshift_r(in.a[0], in.a[1], ls), __funnelshift_r(in.a[1], in.a[2], ls)};
                const uint32_t bw[2] = {__funnelshift_r(in.b[0], in.b[1], ls), __funnelshift_r(in.b[1], in.b[2], ls)};
                const uint32_t vw[2] = {lw[0] | bw[0], lw[1] | bw[1]};
                const unsigned long long vl = (((unsigned long long)vw[1]) << 32) | vw[0];
                const bool all_valid = (~vl & ((1ull << (STEPS + (HP ? 16 : 0))) - 1ull)) == 0ull;
                if (__all_sync(0xFFFFFFFFu, all_valid || !active)) {
                    if (active) walk<HALF, NW, SEG, true, HP>(q, lw, vw, -one, hq, h5, mq);
                } else {
                    if (active) walk<HALF, NW, SEG, false, HP>(q, lw, vw, -one, hq, h5, mq);
                }
            }
            __syncwarp();
            // prefetch the next block's walker inputs; they land while pass B runs
            if (p0 + nrows + wr < last_pr) load_walk_raw(in, a.h, p0 + nrows + wr, rbit, lbit);
        };
        // rows that only fill the window: they enter the ring and the sums, nothing leaves, nothing is stored
        auto fill_rows = [&](int nrows) {
#pragma unroll 1
            for (int r = 0; r < nrows; r++) {
                uint32_t hn[NW][5], en[EC];
#pragma unroll
                for (int w = 0; w < NW; w++) load_h(r, w, hn[w]);
                to_cols(hn, en);
                tm_store<EC>(tring + wrap_t(tslot + r) * EC, en);
#pragma unroll
                for (int w = 0; w < NW; w++) planes_add<PV, KH>(V[w], hn[w]);
            }
        };
        auto advance = [&](int nrows) {
            __syncwarp();
            mslot0 += nrows;
            mslot0 = mslot0 >= NRM ? mslot0 - NRM : mslot0;
            // (no remainder by N here: a conditional subtraction stays on the uniform datapath, and with it the ring
            // rows of the next block's loads and stores)
            tslot += nrows;
            if (N >= RB) {
                tslot = tslot >= N ? tslot - N : tslot;
            } else {
                tslot %= N;
            }
        };

        // Blocks of RB padded rows.  The 2*HALF rows that only fill the window come first: a short block of
        // (2*HALF) % RB rows (this prologue), then whole blocks that add and never subtract or output (`filling`),
        // so that every block from the first output row on is a whole, branch-free `steady` block (but the run's
        // ragged end).  A run always has more than 2*HALF padded rows, so the short block is never cut.
        constexpr int FILL0 = (2 * HALF) % RB;
        if constexpr (FILL0 != 0) {
            pass_a(ja, FILL0);
            fill_rows(FILL0);
            advance(FILL0);
        }
        for (int p0 = ja + FILL0; p0 < last_pr; p0 += RB) {
            const int nrows = min(RB, last_pr - p0);
            const bool steady = p0 >= first_out && nrows == RB;
            const bool filling = p0 + RB <= first_out;

            // MULTI: the earlier chunks' `best` of the rows this block finishes, asked for now so that the loads
            // are back long before the stores that depend on them (they used to be one exposed L2 round trip per row)
            int prev[RB], prev_ru[RB], prev_ws[RB], prev_carry[RB];
#pragma unroll
            for (int r = 0; r < RB; r++) prev[r] = steady ? load_prev(r) : 0;
#pragma unroll
            for (int r = 0; r < RB; r++) prev_ru[r] = RU && steady ? load_prev_ru(r) : 0;
#pragma unroll
            for (int r = 0; r < RB; r++) prev_ws[r] = SUB && steady ? load_prev_ws(r) : 0;
#pragma unroll
            for (int r = 0; r < RB; r++) prev_carry[r] = SUB && steady ? load_prev_carry(r) : 0;

            pass_a(p0, nrows);

            // ---------------- pass B: 32 pixel columns ----------------
            if (steady) {
                // steady state, branch-free: every row enters, one leaves, one output row.
                // Rows go in groups of G so that their winner-take-all chains interleave.
                constexpr int G = (RB % 4 == 0) ? 4 : ((RB % 2 == 0) ? 2 : 1);
                constexpr int GT = N < G ? 1 : G;  // a group's rows must be distinct ring rows
                const int mbase = C::M_ALIGNED ? wrap_m(mslot0 - HALF) : 0;  // the ring row of the block's first centre row
#pragma unroll
                for (int r = 0; r < RB; r += G) {
                    uint32_t Vs[G][NW][PV], Ms[G][NW];
                    uint32_t eo[G][EC];  // the leaving rows, as read back from tensor memory
                    int ts[G];
                    {
#pragma unroll
                        for (int k = 0; k < G; k++) ts[k] = wrap_t(tslot + r + k);
                        if (GT == G) {
                            tm_wait_st();  // a ring row written by an earlier group is complete before it is re-read
#pragma unroll
                            for (int k = 0; k < G; k++) tm_load<EC>(tring + ts[k] * EC, eo[k]);
                            tm_wait_ld();
#pragma unroll
                            for (int k = 0; k < G; k++) tm_pin<EC>(eo[k]);
                        }
                    }
#pragma unroll
                    for (int k = 0; k < G; k++) {
                        uint32_t hn[NW][5], ho[NW][5];
                        if (GT != G) {
                            tm_wait_st();
                            tm_load<EC>(tring + ts[k] * EC, eo[k]);
                            tm_wait_ld();
                            tm_pin<EC>(eo[k]);
                        }
                        from_cols(eo[k], ho);
#pragma unroll
                        for (int w = 0; w < NW; w++) load_h(r + k, w, hn[w]);
                        uint32_t en[EC];
                        to_cols(hn, en);
                        tm_store<EC>(tring + ts[k] * EC, en);  // the entering row takes the leaving row's place
#pragma unroll
                        for (int w = 0; w < NW; w++) {
                            planes_addsub<PV, KH, !MULTI>(V[w], hn[w], ho[w]);
#pragma unroll
                            for (int p = 0; p < PV; p++) Vs[k][w][p] = V[w][p];
                        }
                        if constexpr (C::M_ALIGNED)
                            load_m(mbase + r + k, Ms[k]);
                        else
                            load_m(wrap_m(mslot0 + r + k - HALF), Ms[k]);
                    }
                    finish_rows(std::integral_constant<int, G>{}, Vs, Ms, prev + r, prev_ru + r, prev_ws + r,
                                prev_carry + r);
                }
            } else if (filling) {
                fill_rows(RB);
            } else {
                // the ragged last block of a run
                for (int r = 0; r < nrows; r++) {
                    const int pr = p0 + r;
                    uint32_t hn[NW][5], ho[NW][5];
#pragma unroll
                    for (int w = 0; w < NW; w++) load_h(r, w, hn[w]);
                    {
                        const int t = wrap_t(tslot + r);
                        if (pr > first_out) {  // padded row pr - N left the window: it is what ring row t holds
                            uint32_t eo[EC];
                            tm_wait_st();
                            tm_load<EC>(tring + t * EC, eo);
                            tm_wait_ld();
                            tm_pin<EC>(eo);
                            from_cols(eo, ho);
                        }
                        uint32_t en[EC];
                        to_cols(hn, en);
                        tm_store<EC>(tring + t * EC, en);
                    }
#pragma unroll
                    for (int w = 0; w < NW; w++) {
                        planes_add<PV, KH>(V[w], hn[w]);
                        if (pr > first_out) planes_sub<PV, KH>(V[w], ho[w]);
                    }
                    if (pr >= first_out) {
                        uint32_t Vs[1][NW][PV], Ms[1][NW];
#pragma unroll
                        for (int w = 0; w < NW; w++)
#pragma unroll
                            for (int p = 0; p < PV; p++) Vs[0][w][p] = V[w][p];
                        load_m(wrap_m(mslot0 + r - HALF), Ms[0]);  // centre row j + HALF
                        const int pv = load_prev(0), pvr = load_prev_ru(0), pvs = load_prev_ws(0), pvc = load_prev_carry(0);
                        finish_rows(std::integral_constant<int, 1>{}, Vs, Ms, &pv, &pvr, &pvs, &pvc);
                    }
                }
            }
            advance(nrows);
        }
    }

    {
        tm_wait_st();
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (warp == 0)
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tring), "r"((uint32_t)C::TCOLS) : "memory");
    }
}

// int32 best / web (HotArgs::best, web)
template <int HALF, int NW, int SEG, bool MULTI, bool C2, bool HP>
__global__ void __launch_bounds__(32 * WS<HALF, NW, SEG>::WPC, WS<HALF, NW, SEG>::CTAS_PER_SM)
k_bitslice(BitsliceArgs a)
{
    bitslice_body<int32_t, HALF, NW, SEG, MULTI, C2, HP>(a, static_cast<int32_t *>(a.h.best),
                                                         static_cast<int32_t *>(a.h.web), a.h.out_stride);
}

// uint16_t best / web: the same argument, only the type of the arrays differs
template <int HALF, int NW, int SEG, bool MULTI, bool C2, bool HP>
__global__ void __launch_bounds__(32 * WS<HALF, NW, SEG>::WPC, WS<HALF, NW, SEG>::CTAS_PER_SM)
k_bitslice16(BitsliceArgs a)
{
    bitslice_body<uint16_t, HALF, NW, SEG, MULTI, C2, HP>(a, static_cast<uint16_t *>(a.h.best),
                                                          static_cast<uint16_t *>(a.h.web), a.h.out_stride);
}

// uint16_t best / web and the runner-up score: the 16-bit kernels' argument and the runner-up array (HotArgs and
// BitsliceArgs stay as they are: a field there moves the other families' registers)
struct BitsliceRuArgs {
    BitsliceArgs b;
    uint16_t *runner_up;  // [pairs][FH][W], pair z out_stride elements further
};

// CTAs per SM of a runner-up kernel: its 16-bit sibling's, but one fewer for the MULTI kernels of windows 9 to 15.
// At the sibling's 4 CTAs (128 registers) those spill 36 to 128 bytes more than it; 12 and 16 warps per SM run alike.
template <int HALF, int NW, int SEG, bool MULTI>
constexpr int ru_ctas_per_sm()
{
    constexpr int c = WS<HALF, NW, SEG, true>::CTAS_PER_SM;
    return MULTI && HALF >= 4 && HALF <= 7 && c == 4 ? c - 1 : c;
}

template <int HALF, int NW, int SEG, bool MULTI, bool C2, bool HP>
__global__ void __launch_bounds__(32 * WS<HALF, NW, SEG, true>::WPC, (ru_ctas_per_sm<HALF, NW, SEG, MULTI>()))
k_bitslice_ru(BitsliceRuArgs a)
{
    bitslice_body<uint16_t, HALF, NW, SEG, MULTI, C2, HP, true>(a.b, static_cast<uint16_t *>(a.b.h.best),
                                                                static_cast<uint16_t *>(a.b.h.web), a.b.h.out_stride,
                                                                a.runner_up);
}

// uint16_t best / web and web_sub, the web in sixteenths of a shift: the 16-bit kernels' argument, the web_sub array
// and (MULTI) the u16 per pixel that carries a winner's neighbour scores between chunks
struct BitsliceSubArgs {
    BitsliceArgs b;
    uint16_t *web_sub;  // [pairs][FH][W], pair z out_stride elements further
    uint16_t *carry;    // the same layout, MULTI only (scratch of the caller's)
};

// CTAs per SM of a sub-pixel kernel: its 16-bit sibling's, but one fewer for the MULTI kernels of windows 5 to 15.  At
// the sibling's 4 CTAs (128 registers) those spill (windows 5 and 7: 104 and 52 bytes of stores)
template <int HALF, int NW, int SEG, bool MULTI>
constexpr int sub_ctas_per_sm()
{
    constexpr int c = WS<HALF, NW, SEG, true>::CTAS_PER_SM;
    return MULTI && HALF >= 2 && HALF <= 7 && c == 4 ? c - 1 : c;
}

template <int HALF, int NW, int SEG, bool MULTI, bool C2, bool HP>
__global__ void __launch_bounds__(32 * WS<HALF, NW, SEG, true>::WPC, (sub_ctas_per_sm<HALF, NW, SEG, MULTI>()))
k_bitslice_sub(BitsliceSubArgs a)
{
    bitslice_body<uint16_t, HALF, NW, SEG, MULTI, C2, HP, false, true>(a.b, static_cast<uint16_t *>(a.b.h.best),
                                                                       static_cast<uint16_t *>(a.b.h.web),
                                                                       a.b.h.out_stride, nullptr, a.web_sub, a.carry);
}

// which outputs a family stores beyond best / web
enum Extra { EXTRA_NONE = 0, EXTRA_RU = 1, EXTRA_SUB = 2 };

// the family: int32 (k_bitslice), 16-bit (k_bitslice16), 16-bit with the runner-up (RU, k_bitslice_ru) or with web_sub
// (SUB, k_bitslice_sub)
template <typename OutT, int X, int HALF, int NW, int SEG, bool MULTI, bool C2, bool HP>
constexpr auto kernel_of()
{
    static_assert(X == EXTRA_NONE || std::is_same<OutT, uint16_t>::value, "runner-up / sub-pixel: 16-bit outputs only");
    if constexpr (X == EXTRA_SUB)
        return k_bitslice_sub<HALF, NW, SEG, MULTI, C2, HP>;
    else if constexpr (X == EXTRA_RU)
        return k_bitslice_ru<HALF, NW, SEG, MULTI, C2, HP>;
    else if constexpr (std::is_same<OutT, uint16_t>::value)
        return k_bitslice16<HALF, NW, SEG, MULTI, C2, HP>;
    else
        return k_bitslice<HALF, NW, SEG, MULTI, C2, HP>;
}

// extra: the runner-up array (X == EXTRA_RU) or web_sub (EXTRA_SUB); carry: EXTRA_SUB's chunk carry
template <typename OutT, int X, int HALF, int NW, int SEG, bool C2, bool HP>
int launch_one(const HotArgs &h, int num_sms, cudaStream_t s, int mode, LaunchRecord *rec, uint16_t *extra,
               uint16_t *carry)
{
    constexpr bool RU = X == EXTRA_RU, SUB = X == EXTRA_SUB;
    using C = WS<HALF, NW, SEG, (RU || SUB) && !C2 && !HP>;  // (bitslice_body's layout: its centre-match ring, its shared memory)
    if (mode == MODE_TMEM_COLUMNS) return C::TCOLS;
    // MULTI: more than one chunk of 32*NW shifts, i.e. (best, web) are merged across passes
    // (one word per lane is only chosen for 32 shifts or fewer: no MULTI flavour of it is instantiated)
    const bool multi = !C2 && NW == 2 && h.g.D > 32 * NW;
    if (!C2 && !multi && h.g.D > 32 * NW) {
        set_error("bit-sliced kernel: %d shifts need two shift words per lane", h.g.D);
        return SM_ERR_ARG;
    }
    if (HP && h.g.D > 16) {
        set_error("bit-sliced kernel: half-word pairs hold at most 16 shifts, not %d", h.g.D);
        return SM_ERR_ARG;
    }
    auto kern = (C2 || HP) ? kernel_of<OutT, X, HALF, NW, SEG, false, C2, HP>()
                           : (multi ? kernel_of<OutT, X, HALF, NW, SEG, NW == 2 && !HP, false, false>()
                                    : kernel_of<OutT, X, HALF, NW, SEG, false, false, false>());
    // resident warps per SM of this instantiation: what shared memory, the 512 TMEM columns and the register file
    // allow, all known at compile time (WS::CTAS_PER_SM is also the kernel's __launch_bounds__).  (The occupancy
    // API is not asked: it answers 1 CTA per SM for these kernels, whatever carve-out is set, while the
    // hardware runs the 4 that ncu's launch__occupancy_limit_* report.)
    // (the runner-up and sub-pixel families' MULTI kernels may hold fewer: ru_ctas_per_sm, sub_ctas_per_sm)
    const int ctas_per_sm = RU && multi    ? ru_ctas_per_sm<HALF, NW, SEG, NW == 2 && !HP && !C2>()
                            : SUB && multi ? sub_ctas_per_sm<HALF, NW, SEG, NW == 2 && !HP && !C2>()
                                           : C::CTAS_PER_SM;
    const int warps_per_sm = ctas_per_sm * C::WPC;
    if (mode == MODE_PREPARE) {
        SM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_REQ));
        SM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    if (mode == MODE_PREPARE) return warps_per_sm;  // module loaded, attribute set
    BitsliceArgs a;
    a.h = h;
    const int strip_cols = C::TW * (C2 ? NW : 1) * (HP ? 2 : 1);
    const int strips = (h.g.W + strip_cols - 1) / strip_cols;
    // a run is at least one block of rows.  (Short runs pay 2*half warm-up rows each, but they
    // only happen when the frame is too small to fill the machine, where latency is what counts.)
    const int min_rows = C::RB;
    const int max_segs = (h.g.BH + min_rows - 1) / min_rows;
    // a wanted number of runs -> whole blocks of RB rows per run (only the frame's last run has a
    // ragged, slower block) and the number of runs that results
    auto shape = [&](int want_segs, int &rows) {
        int sg = want_segs < 1 ? 1 : (want_segs > max_segs ? max_segs : want_segs);
        rows = (h.g.BH + sg - 1) / sg;
        rows = (rows + C::RB - 1) / C::RB * C::RB;
        return (h.g.BH + rows - 1) / rows;
    };
    // CTA slots of the machine and CTAs per row run of one pair
    const int slots = num_sms * warps_per_sm / C::WPC > 0 ? num_sms * warps_per_sm / C::WPC : 1;
    const int ctas_per_run = (strips + C::WPC - 1) / C::WPC;
    int segs;
    if (h.force_segs > 0) {
        segs = h.force_segs;  // development hook (sm_set_option)
    } else if (h.npairs == 1) {
        // latency mode (one pair per launch).  All CTAs do the same work: a run of R rows costs R rows, the
        // window-filling blocks in front of them (whole blocks of RB rows, about half a row's work per row: pass A and
        // one add, no subtraction, no winner-take-all) and a fixed start-up.  The kernel is bound by the ALU pipe, so
        // an SM takes as long as the work of the CTAs that land on it: ceil(CTAs / SMs) on the fullest while the grid
        // is under about 1.7 waves of CTA slots (everything resident at once or a ragged second round), CTAs / SMs
        // once the block scheduler has several rounds to even things out.  Too few resident warps leave the pipe
        // idle (measured on one-pair launches, tools/sweep_runs.py: 4 warps per SM reach about 0.6 of the rate of
        // 16, 8 about 0.85, 12 about 0.94).  Pick the number of runs that minimises that: a cost model, nothing
        // is timed at sm_create.
        const int start_rows = 4;
        const int fill_rows = (2 * HALF + C::RB - 1) / C::RB * C::RB;
        auto eff_of = [](int warps) {
            if (warps >= 16) return 1.0;
            if (warps >= 12) return 0.94 + (warps - 12) * (0.06 / 4);
            if (warps >= 8) return 0.85 + (warps - 8) * (0.09 / 4);
            return 0.6 + (warps > 4 ? warps - 4 : 0) * (0.25 / 4);
        };
        double best_cost = -1.0;
        segs = 1;
        for (int sg = 1; sg <= max_segs; sg++) {
            int rows, got = shape(sg, rows);
            if (got != sg) continue;
            const int ctas = ctas_per_run * got;
            const int per_sm_max = (ctas + num_sms - 1) / num_sms;
            const double per_sm = 10 * ctas < 17 * slots ? (double)per_sm_max : (double)ctas / num_sms + 0.05;
            const int resident = (per_sm_max < ctas_per_sm ? per_sm_max : ctas_per_sm) * C::WPC;
            const double cost = per_sm * (rows + 0.5 * fill_rows + start_rows) / eff_of(resident);
            if (best_cost < 0 || cost < best_cost) best_cost = cost, segs = got;
            if (ctas > 6 * slots) break;
        }
    } else {
        // throughput mode (several pairs per launch): runs of about 32 windows -- the launch may be several waves
        // deep, the block scheduler keeps the slots full and the next launch (other stream) covers the tail --
        // but never so few CTAs that one launch cannot fill the machine once
        const int want = throughput_run_windows() * C::N;
        segs = (h.g.BH + want - 1) / want;
        const int fill = (slots + ctas_per_run * h.npairs - 1) / (ctas_per_run * h.npairs);
        if (segs < fill) segs = fill;
    }
    segs = shape(segs, a.rows_per_seg);
    dim3 grid((strips + C::WPC - 1) / C::WPC, segs, h.npairs);
    // the kernel's argument: BitsliceArgs, or with RU that and the runner-up array, with SUB web_sub and the carry
    typename std::conditional<RU, BitsliceRuArgs, typename std::conditional<SUB, BitsliceSubArgs, BitsliceArgs>::type>::type arg;
    if constexpr (RU)
        arg = BitsliceRuArgs{a, extra};
    else if constexpr (SUB)
        arg = BitsliceSubArgs{a, extra, carry};
    else
        arg = a;
    if (h.after_pack) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid;
        cfg.blockDim = dim3(32 * C::WPC);
        cfg.dynamicSmemBytes = C::SMEM_REQ;
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        SM_CUDA(cudaLaunchKernelEx(&cfg, kern, arg));
    } else {
        kern<<<grid, 32 * C::WPC, C::SMEM_REQ, s>>>(arg);
    }
    SM_CUDA(cudaGetLastError());
    if (rec) {
        rec->shape = SM_SHAPE_BITSLICE | HALF | (NW == 2 ? SM_SHAPE_TWO_WORDS : 0) | (SEG == 8 ? SM_SHAPE_SEG8 : 0) |
                     (C2 ? SM_SHAPE_C2 : 0) | (HP ? SM_SHAPE_HP : 0) | (multi ? SM_SHAPE_MULTI : 0);
        rec->row_runs = (int)grid.y;
    }
    return 1;
}

// How a lane's words are used and how long a walker's segment is.
//   words: two shift words of one pixel (64 shifts per pass); for num_shifts <= 32 the one shift word of two
//          pixels (column pairs, C2) for windows up to 13 and frames at least one 64-column strip wide, else one
//          word of one pixel.  Measured at 1080p, one pair per launch, 32 shifts: window 9: 19.4 vs 22.9 us,
//          window 13: 22.9 vs 23.7, window 17: 25.8 vs 24.6.
//   segment: shorter walks = fewer rows per block = smaller rings, but more window-filling steps per output.
//          Measured on config 2 (us per pair, batched): 8 -> 18.2, 16 -> 18.0, 32 -> 25.2.
struct Shape {
    int nw, seg;
    bool c2, hp;
    int strip_cols() const { return 32 * (c2 ? nw : 1) * (hp ? 2 : 1); }
};

constexpr int C2_MAX_HALF = 6;

static Shape pick_shape(const HotArgs &h, int num_sms)
{
    Shape sh;
    sh.seg = 16;
    sh.hp = false;
    if (h.g.D > 32) {
        sh.nw = 2;
        sh.c2 = false;
    } else {
        sh.c2 = h.g.W >= 64 && h.g.half <= C2_MAX_HALF;
        sh.nw = sh.c2 ? 2 : 1;
        // 16 shifts or fewer: two pixels per word (half-word pairs)
        sh.hp = h.g.D <= 16 && h.g.W >= 64;
        // One small frame per launch cannot fill the machine with 16-row blocks (480x270 at the reference defaults is
        // 68 CTAs): 8-pixel walker segments halve the block to 8 rows and double the CTAs.  They cost a quarter more
        // walker steps per pixel, so batches keep the 16-pixel segments.  Measured, one frame per call: 480x270
        // 15.5 -> 13.5 us, 327x245 15.4 -> 13.4 us (a call costs the host 13.4 us, which is what 240x135 shows either way).
        if (sh.nw == 1 && !sh.hp && h.npairs == 1 && num_sms > 0) {
            const int ctas = ((h.g.W + 31) / 32 + 3) / 4 * ((h.g.BH + 15) / 16);
            if (ctas < num_sms) sh.seg = 8;
        }
    }
#ifdef SMB_DEV  // experiment hooks of the development build only (make DEV=1); never in the shipped library
    if (getenv("SMB_NO_C2") && atoi(getenv("SMB_NO_C2")) && sh.c2) sh.c2 = false, sh.nw = 1;
    if (getenv("SMB_NO_HP") && atoi(getenv("SMB_NO_HP"))) sh.hp = false;
    if (getenv("SMB_NW") && !sh.c2) sh.nw = atoi(getenv("SMB_NW"));
    if (getenv("SMB_SEG")) sh.seg = atoi(getenv("SMB_SEG"));
#endif
    return sh;
}

// the kernel of the geometry, from the family that stores OutT (X: and the runner-up or web_sub, to extra; the
// sub-pixel family's chunk carry to carry)
template <typename OutT, int X = EXTRA_NONE>
int dispatch(const HotArgs &h, int num_sms, cudaStream_t s, int mode, LaunchRecord *rec = nullptr,
             uint16_t *extra = nullptr, uint16_t *carry = nullptr)
{
    if (mode == MODE_PREPARE && h.npairs == 1) {
        // a context launches one pair at a time AND batches: prepare the batch flavour too if it is another kernel
        HotArgs hb = h;
        hb.npairs = 2;
        const Shape a = pick_shape(h, num_sms), b = pick_shape(hb, num_sms);
        if (a.seg != b.seg || a.nw != b.nw || a.c2 != b.c2 || a.hp != b.hp) {
            const int rc = dispatch<OutT, X>(hb, num_sms, s, mode);
            if (rc < 0) return rc;
        }
    }
    const Shape sh = pick_shape(h, num_sms);
    const int half = h.g.half;
#define SM_SHAPE(HF, NW_, SEG_, C2_, HP_) \
    if (half == HF && sh.nw == NW_ && sh.seg == SEG_ && sh.c2 == C2_ && sh.hp == HP_) \
        return launch_one<OutT, X, HF, NW_, SEG_, C2_, HP_>(h, num_sms, s, mode, rec, extra, carry);
#define SM_HALVES(M, ...) \
    M(0, __VA_ARGS__) M(1, __VA_ARGS__) M(2, __VA_ARGS__) M(3, __VA_ARGS__) M(4, __VA_ARGS__) M(5, __VA_ARGS__) \
    M(6, __VA_ARGS__) M(7, __VA_ARGS__) M(8, __VA_ARGS__) M(9, __VA_ARGS__) M(10, __VA_ARGS__) M(11, __VA_ARGS__) \
    M(12, __VA_ARGS__) M(13, __VA_ARGS__) M(14, __VA_ARGS__) M(15, __VA_ARGS__)
    SM_HALVES(SM_SHAPE, 1, 16, false, false)
    SM_HALVES(SM_SHAPE, 2, 16, false, false)
    SM_HALVES(SM_SHAPE, 1, 16, false, true)
    SM_HALVES(SM_SHAPE, 1, 8, false, false)
#define SM_C2(HP_) \
    SM_SHAPE(0, 2, 16, true, HP_) SM_SHAPE(1, 2, 16, true, HP_) SM_SHAPE(2, 2, 16, true, HP_) SM_SHAPE(3, 2, 16, true, HP_) \
    SM_SHAPE(4, 2, 16, true, HP_) SM_SHAPE(5, 2, 16, true, HP_) SM_SHAPE(6, 2, 16, true, HP_)
    SM_C2(false) SM_C2(true)
#undef SM_C2
#undef SM_HALVES
#undef SM_SHAPE
    set_error("bit-sliced kernel: window half %d with %d word(s) per lane and %d-column walks is not instantiated",
              half, sh.nw, sh.seg);
    return SM_ERR_ARG;
}

}  // namespace

}  // namespace smb
