// stereo_b200.cu -- the C ABI of include/stereo_b200.h: context, transfers, orchestration.
//
// Stands in for the host side of the reference's CUDA programs: main()'s
// MAKE_GPU_COPY uploads (stereo.cu:402-403), algorithm()'s allocations, launch
// sequence and frees (stereo.cu:296-347), write_gpu_image's D2H (image.cu:15-23) and
// the min/max helpers (util.cu:34-42).  No kernel lives here (k_*.cu).
#include <stdarg.h>
#include <stdlib.h>

#include <condition_variable>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "sm_common.cuh"

namespace smb {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

}  // namespace smb

using namespace smb;

struct sm_ctx {
    int device = 0;
    int W = 0, FH = 0;         // frame geometry
    int row0 = 0, row1 = 0;    // output rows owned by this context
    int D = 0, sw = 0, half = 0, variant = 0;
    int M = 0;  // min_shift: the context searches shifts [M, M + D)
    int kernel = SM_KERNEL_AUTO;
    int num_sms = 148;
    PackedGeom g{};

    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    // sm_profile_*: one event triple per hot-path call
    cudaEvent_t *prof_ev = nullptr;
    int prof_cap = 0, prof_n = 0;
    int last_launches = 0;
    int tuned_segs = 0;  // SM_OPT_ROW_RUNS: row runs per strip of a one-pair launch (0: the kernel's cost model)
    int occ = 0;         // resident warps per SM of the bit-sliced kernel of this geometry (prepare_bitslice)
    LaunchRecord last_launch;  // the most recent hot-path launch (SM_INFO_KERNEL_SHAPE, SM_INFO_ROW_RUNS)

    // frame-sized device arrays (a band context touches only the rows it needs)
    uint8_t *img_u8[2] = {nullptr, nullptr};
    double *img_f64[2] = {nullptr, nullptr};
    int img_kind = 0;  // 0 none, 1 u8, 2 f64
    uint8_t *edges[2] = {nullptr, nullptr};
    bool have_edges = false;
    bool planes_valid = false;  // LA/LB/RB already hold the packed planes of edges[] (sm_edges wrote them itself)
    uint32_t *edge_lut = nullptr;  // detector decisions for all (L, R) sum pairs at lut_threshold
    double lut_threshold = -1.0;
    bool edges_fp64_only = false;  // SM_OPT_EDGES_FP64: always take the FP64 kernel (cross-check)
    int pipe_group_opt = 0;        // SM_OPT_PIPE_GROUP: pairs per sm_run_batch stage (0: by frame size)
    int32_t *best = nullptr, *web = nullptr;
    bool have_web = false;
    // frame-sized 16-bit arrays: sm_bands_run16's results, sm_download_web_u16's narrowed web
    uint16_t *best16 = nullptr, *web16 = nullptr;
    uint16_t *ru16 = nullptr;  // sm_bands_run_ru16's runner-up scores
    uint16_t *sub16 = nullptr;    // sm_bands_run_sub16's web_sub
    uint16_t *carry16 = nullptr;  // the sub-pixel kernels' chunk carry of one-pair launches (more than 64 shifts)
    bool prepared16 = false;  // the 16-bit bit-sliced kernels of this geometry are loaded (prepare_bitslice16)
    int occ_ru = 0;           // ... the runner-up kernels (prepare_bitslice_ru; 0: not yet): their resident warps per SM
    int occ_sub = 0;          // ... the sub-pixel kernels (prepare_bitslice_sub; 0: not yet)
    int32_t *web2 = nullptr, *tmp = nullptr;  // step 3 ping-pong
    const int32_t *web_filled = nullptr;      // result of fill_web_holes (may alias web)
    bool have_web2 = false;
    bool web_may_have_holes = false;          // only a web from sm_set_web can contain zeros
    uint8_t *out = nullptr;
    bool have_out = false;
    int32_t *minmax = nullptr;       // two (min, max) slots, used alternately (k_step3.cu)
    int32_t *minmax_host = nullptr;  // pinned landing place of a slot
    int minmax_cur = 0;
    // band-sized packed planes
    uint32_t *LA = nullptr, *LB = nullptr, *RB = nullptr;
    // sm_match_wta_dev_batch: a second stream packs pair k+1.. while the main kernel of
    // pair k runs; NPB packed-plane sets rotate between the two
    static constexpr int NPB = 3;
    cudaStream_t pack_stream = nullptr, main2_stream = nullptr;  // main kernels alternate stream / main2_stream
    cudaEvent_t ev_join = nullptr;
    int batch_group = 1;      // pairs per launch in sm_match_wta_dev_batch (1 for the literal kernel)
    int batch_group_cap = 0;  // ... of the bit-sliced kernel; the plane sets are sized for it
    bool batch_ready = false;
    uint32_t *pLA[NPB] = {nullptr, nullptr, nullptr}, *pLB[NPB] = {nullptr, nullptr, nullptr},
             *pRB[NPB] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_packed[NPB] = {nullptr, nullptr, nullptr}, ev_used[NPB] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr;
    // the best of 16-bit batches without a caller's best (the bit-sliced kernel always stores it): one scratch per
    // plane set, batch_group_cap frames each (ev_used[b] orders its reuse like that of the plane set)
    // (with the caller's pair stride, out_stride: pbest16_elems elements each)
    uint16_t *pBest16[NPB] = {nullptr, nullptr, nullptr};
    size_t pbest16_elems = 0;
    // the sub-pixel kernels' chunk carry (more than 64 shifts), sized and ordered like pBest16
    uint16_t *pCarry16[NPB] = {nullptr, nullptr, nullptr};
    size_t pcarry16_elems = 0;
    // scratch for on-demand debug planes / u8 web
    uint8_t *scratch_u8 = nullptr;
    int32_t *scratch_i32 = nullptr;

    // sm_run_batch: a three-stage pipeline (H2D | edges + hot path | D2H) over groups of pairs;
    // NPIPE group buffer sets rotate between the stages
    static constexpr int NPIPE = 3;
    struct Pipe {
        int group = 0;  // pairs per stage
        bool ready = false;
        cudaStream_t up = nullptr, down = nullptr;
        uint8_t *img[NPIPE] = {nullptr, nullptr, nullptr};    // [2*group][npix]: first images, then second images
        uint8_t *edg[NPIPE] = {nullptr, nullptr, nullptr};    // same layout
        int32_t *web[NPIPE] = {nullptr, nullptr, nullptr};    // [group][npix]
        int32_t *best[NPIPE] = {nullptr, nullptr, nullptr};   // [group][npix]
        uint8_t *web8[NPIPE] = {nullptr, nullptr, nullptr};   // [group][npix], only for the u8 result
        // the 16-bit results, written by the hot path itself ([group][npix]; best16 only when the caller wants best)
        uint16_t *web16[NPIPE] = {nullptr, nullptr, nullptr}, *best16[NPIPE] = {nullptr, nullptr, nullptr};
        uint16_t *ru16[NPIPE] = {nullptr, nullptr, nullptr};  // the runner-up scores, only when the caller wants them
        uint16_t *sub16[NPIPE] = {nullptr, nullptr, nullptr};  // web_sub, only when the caller wants it
        cudaEvent_t ev_up[NPIPE] = {nullptr, nullptr, nullptr}, ev_comp[NPIPE] = {nullptr, nullptr, nullptr},
                    ev_down[NPIPE] = {nullptr, nullptr, nullptr};
    } pipe;

    size_t npix() const { return (size_t)W * FH; }
};

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

#define SM_ENTER(ctx)                                                   \
    if (!(ctx)) {                                                       \
        set_error("%s: NULL context", __func__);                        \
        return SM_ERR_ARG;                                              \
    }                                                                   \
    DeviceGuard guard__((ctx)->device);                                 \
    if (!guard__.ok) {                                                  \
        set_error("%s: cudaSetDevice(%d) failed", __func__, (ctx)->device); \
        return SM_ERR_CUDA;                                             \
    }

template <typename T>
int dev_alloc(T **p, size_t count)
{
    if (*p) return SM_OK;
    SM_CUDA(cudaMalloc((void **)p, count * sizeof(T)));
    return SM_OK;
}

// Frame rows [lo, hi) as up to a few contiguous [start, start+count) runs inside the
// frame: wrapped mod FH for WRAP (util.h:42-47), clipped for GHOST.
struct RowRuns {
    int n = 0;
    int start[4], count[4];
};

RowRuns row_runs(int lo, int hi, int FH, bool wrap)
{
    RowRuns r;
    if (hi - lo >= FH) {
        r.n = 1;
        r.start[0] = 0;
        r.count[0] = FH;
        return r;
    }
    if (!wrap) {
        lo = lo < 0 ? 0 : lo;
        hi = hi > FH ? FH : hi;
        if (hi > lo) {
            r.n = 1;
            r.start[0] = lo;
            r.count[0] = hi - lo;
        }
        return r;
    }
    int a = ((lo % FH) + FH) % FH, len = hi - lo;
    while (len > 0 && r.n < 4) {
        int c = len < FH - a ? len : FH - a;
        r.start[r.n] = a;
        r.count[r.n] = c;
        r.n++;
        len -= c;
        a = 0;
    }
    return r;
}

template <typename T>
int copy_rows_h2d(sm_ctx *c, T *dst, const T *src, int lo, int hi)
{
    RowRuns rr = row_runs(lo, hi, c->FH, c->variant == SM_WRAP);
    for (int k = 0; k < rr.n; k++) {
        size_t off = (size_t)rr.start[k] * c->W;
        SM_CUDA(cudaMemcpyAsync(dst + off, src + off, (size_t)rr.count[k] * c->W * sizeof(T),
                                cudaMemcpyHostToDevice, c->stream));
    }
    return SM_OK;
}

template <typename T>
int copy_band_d2h(sm_ctx *c, T *host, const T *dev)
{
    size_t off = (size_t)c->row0 * c->W;
    SM_CUDA(cudaMemcpyAsync(host + off, dev + off, (size_t)(c->row1 - c->row0) * c->W * sizeof(T),
                            cudaMemcpyDeviceToHost, c->stream));
    return SM_OK;
}

// Where a hot-path call writes best / web: int32 arrays, or (web16 set) 16-bit ones, best16 possibly NULL.  With
// 16-bit ones, runner_up (if set) receives the runner-up scores (the runner-up kernels), or web_sub (if set) the web in
// sixteenths of a shift (the sub-pixel kernels; past 64 shifts they need a carry array of the same layout).
struct Outputs {
    int32_t *best = nullptr, *web = nullptr;
    uint16_t *best16 = nullptr, *web16 = nullptr;
    uint16_t *runner_up = nullptr;
    uint16_t *web_sub = nullptr, *carry = nullptr;
    // pair k of a batch: every array k * stride elements further
    Outputs pair(size_t k, size_t stride) const
    {
        auto at = [&](auto *p) { return p ? p + k * stride : p; };
        return {at(best), at(web), at(best16), at(web16), at(runner_up), at(web_sub), at(carry)};
    }
};

HotArgs hot_args(sm_ctx *c, const Outputs &o)
{
    HotArgs a;
    a.g = c->g;
    a.LA = c->LA;
    a.LB = c->LB;
    a.RB = c->RB;
    a.best = o.web16 ? (void *)o.best16 : (void *)o.best;
    a.web = o.web16 ? (void *)o.web16 : (void *)o.web;
    a.row0 = c->row0;
    a.force_segs = c->tuned_segs;
    a.blocks_per_sm = c->occ;
    a.M = c->M;
    return a;
}

int hot_kernel(const sm_ctx *c)
{
    return c->kernel == SM_KERNEL_AUTO ? (bitslice_supports(c->half, c->D) ? SM_KERNEL_BITSLICE : SM_KERNEL_DIRECT)
                                       : c->kernel;
}

// The bit-sliced kernel always stores best (it merges 64-shift chunks through it, and a per-store predicate would cost
// its 16-bit family registers): a 16-bit call without a best of the caller's gives it a scratch array.
bool stores_best(const sm_ctx *c) { return hot_kernel(c) == SM_KERNEL_BITSLICE; }

// Loads the runner-up kernels of the context's geometry (once); their resident warps per SM go to c->occ_ru.
int prepare_ru(sm_ctx *c)
{
    if (c->occ_ru > 0) return SM_OK;
    int occ = c->occ;
    if (hot_kernel(c) == SM_KERNEL_BITSLICE && bitslice_supports(c->half, c->D)) {
        occ = prepare_bitslice_ru(hot_args(c, Outputs{}), c->num_sms);
        if (occ < 0) return occ;
    }
    c->occ_ru = occ > 0 ? occ : 1;
    return SM_OK;
}

// Loads the sub-pixel kernels of the context's geometry (once); their resident warps per SM go to c->occ_sub.
int prepare_sub(sm_ctx *c)
{
    if (c->occ_sub > 0) return SM_OK;
    int occ = c->occ;
    if (hot_kernel(c) == SM_KERNEL_BITSLICE && bitslice_supports(c->half, c->D)) {
        occ = prepare_bitslice_sub(hot_args(c, Outputs{}), c->num_sms);
        if (occ < 0) return occ;
    }
    c->occ_sub = occ > 0 ? occ : 1;
    return SM_OK;
}

// whether the sub-pixel kernel of the context merges 64-shift chunks (and needs Outputs::carry)
bool sub_needs_carry(const sm_ctx *c) { return hot_kernel(c) == SM_KERNEL_BITSLICE && c->D > 64; }

// The main kernel: of the runner-up family with runner_up, of the sub-pixel one with web_sub, of the 16-bit one with
// out16, else of the int32 one.
int launch_main(sm_ctx *c, const HotArgs &a, bool out16, uint16_t *runner_up, cudaStream_t st, uint16_t *web_sub = nullptr,
                uint16_t *carry = nullptr)
{
    const int k = hot_kernel(c);
    if (k == SM_KERNEL_BITSLICE) {
        if (!bitslice_supports(c->half, c->D)) {
            set_error("bit-sliced kernel does not cover square_width %d / num_shifts %d", c->sw, c->D);
            return SM_ERR_ARG;
        }
        if (out16 && !runner_up && !web_sub && !c->prepared16) {  // (sm_create prepared the int32 family)
            const int rc = prepare_bitslice16(hot_args(c, Outputs{}), c->num_sms);
            if (rc < 0) return rc;
            c->prepared16 = true;
        }
        if (runner_up) {
            const int rc = prepare_ru(c);
            if (rc < 0) return rc;
        }
        if (web_sub) {
            const int rc = prepare_sub(c);
            if (rc < 0) return rc;
        }
        LaunchRecord rec;
        const int rc = runner_up ? launch_bitslice_ru(a, runner_up, c->num_sms, st, &rec)
                       : web_sub ? launch_bitslice_sub(a, web_sub, carry, c->num_sms, st, &rec)
                       : out16   ? launch_bitslice16(a, c->num_sms, st, &rec)
                                 : launch_bitslice(a, c->num_sms, st, &rec);
        if (rc >= 0) c->last_launch = rec;
        return rc;
    }
    const int rc = launch_direct(a, st, out16, runner_up, web_sub);
    if (rc >= 0) {
        c->last_launch.shape = SM_SHAPE_DIRECT;
        c->last_launch.row_runs = 0;
    }
    return rc;
}

int run_hot(sm_ctx *c, const uint8_t *e1, const uint8_t *e2, const Outputs &out)
{
    int launches = 0, rc;
    cudaEvent_t *pe = (c->prof_ev && c->prof_n < c->prof_cap) ? c->prof_ev + 3 * c->prof_n : nullptr;
    SM_CUDA(cudaEventRecord(c->ev0, c->stream));
    if (pe) SM_CUDA(cudaEventRecord(pe[0], c->stream));
    // sm_edges writes the packed planes itself (k_edges_planes): no pack launch then
    const bool packed = c->planes_valid && e1 == c->edges[0] && e2 == c->edges[1];
    if (!packed) {
        rc = launch_pack(e1, e2, c->FH, c->row0, c->variant, c->g, c->M, c->LA, c->LB, c->RB, c->stream);
        if (rc < 0) return rc;
        launches += rc;
    }
    if (pe) SM_CUDA(cudaEventRecord(pe[1], c->stream));
    HotArgs a = hot_args(c, out);
#ifdef SMB_DEV
    static const bool no_pdl = getenv("SMB_NO_PDL") && atoi(getenv("SMB_NO_PDL"));  // experiment hook, development build only
#else
    constexpr bool no_pdl = false;
#endif
    // the producer of the planes (pack or edge kernel) is the launch just before on this stream unless the
    // per-kernel profile put an event in between: the main kernel may start as its programmatic dependent.
    // (It waits for every earlier grid of the stream to complete before it reads anything, whatever that grid is.)
    a.after_pack = pe == nullptr && !no_pdl;
    uint16_t *carry = nullptr;
    if (out.web_sub && sub_needs_carry(c)) {
        if ((rc = dev_alloc(&c->carry16, c->npix()))) return rc;  // (frame-sized: band contexts write their own rows)
        carry = c->carry16;
    }
    rc = launch_main(c, a, out.web16 != nullptr, out.runner_up, c->stream, out.web_sub, carry);
    if (rc < 0) return rc;
    launches += rc;
    SM_CUDA(cudaEventRecord(c->ev1, c->stream));
    if (pe) {
        SM_CUDA(cudaEventRecord(pe[2], c->stream));
        c->prof_n++;
    }
    c->timed = true;
    c->last_launches = launches;
    return SM_OK;
}

void profile_free(sm_ctx *c)
{
    for (int k = 0; k < 3 * c->prof_cap; k++)
        if (c->prof_ev[k]) cudaEventDestroy(c->prof_ev[k]);
    free(c->prof_ev);
    c->prof_ev = nullptr;
    c->prof_cap = c->prof_n = 0;
}

}  // namespace

// ---- library-level ---------------------------------------------------------------

extern "C" const char *sm_last_error(void) { return g_err; }

// 1.1: sm_multi_*, sm_bands_*; 1.2: sm_set_option / sm_get_info, square_width 0, the microbenchmarks moved out;
// 1.3: SM_INFO_KERNEL_SHAPE / SM_INFO_ROW_RUNS; then, additive, the 16-bit result entries (*16, sm_download_web_u16),
// the search-range creators (*_range), the runner-up entries (*_ru16) and the sub-pixel entries (*_sub16)
extern "C" int sm_version(void) { return (1 << 16) | 3; }

extern "C" int sm_device_count(void)
{
    int n = 0;
    SM_CUDA(cudaGetDeviceCount(&n));
    return n;
}

extern "C" int sm_host_alloc(void **ptr, size_t bytes)
{
    SM_REQUIRE(ptr, "sm_host_alloc: NULL ptr");
    SM_CUDA(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return SM_OK;
}

extern "C" int sm_host_free(void *ptr)
{
    if (ptr) SM_CUDA(cudaFreeHost(ptr));
    return SM_OK;
}

extern "C" int sm_band_rows(int height, int n_bands, int band, int *row0, int *row1)
{
    SM_REQUIRE(height > 0 && n_bands > 0 && band >= 0 && band < n_bands && row0 && row1,
               "sm_band_rows: bad arguments");
    // as even as possible: the first (height % n_bands) bands get one extra row
    int q = height / n_bands, r = height % n_bands;
    *row0 = band * q + (band < r ? band : r);
    *row1 = *row0 + q + (band < r ? 1 : 0);
    return SM_OK;
}

// ---- context -----------------------------------------------------------------------

extern "C" int sm_create_band_range(sm_ctx **out, int device, int width, int frame_height, int row0, int row1,
                                    int min_shift, int num_shifts, int square_width, int variant)
{
    SM_REQUIRE(out, "sm_create: NULL ctx pointer");
    *out = nullptr;
    SM_REQUIRE(width > 0 && frame_height > 0, "sm_create: width/height must be positive");
    SM_REQUIRE((size_t)width * frame_height < ((size_t)1 << 31), "sm_create: frame too large");
    SM_REQUIRE(num_shifts >= 1 && num_shifts <= 512, "sm_create: num_shifts must be in [1, 512]");
    // web = 1 + the winning shift <= min_shift + num_shifts must stay exact in 16 bits, and above step 3's hole (0)
    SM_REQUIRE(min_shift >= 0 && min_shift <= 65535 - num_shifts,
               "sm_create: min_shift must be >= 0 with min_shift + num_shifts <= 65535");
    // the reference takes any square_width up to the frame size (stereo.cu:395-398); its window is
    // half = square_width / 2 either side, so 0 (and -1) mean the 1x1 window.  Wider than 63 is not built here.
    SM_REQUIRE(square_width >= -1 && square_width <= 63, "sm_create: square_width must be in [0, 63]");
    // same check as the reference driver (stereo.cu:395-398)
    SM_REQUIRE(square_width <= width && square_width <= frame_height,
               "sm_create: square width must not be higher than image width/height");
    SM_REQUIRE(variant == SM_WRAP || variant == SM_GHOST, "sm_create: unknown variant");
    SM_REQUIRE(row0 >= 0 && row1 > row0 && row1 <= frame_height, "sm_create: bad row band");
    int ndev = 0;
    SM_CUDA(cudaGetDeviceCount(&ndev));
    SM_REQUIRE(device >= 0 && device < ndev, "sm_create: device %d of %d", device, ndev);

    sm_ctx *c = new (std::nothrow) sm_ctx;
    if (!c) {
        set_error("sm_create: out of memory");
        return SM_ERR_NOMEM;
    }
    c->device = device;
    DeviceGuard guard(device);
    c->W = width;
    c->FH = frame_height;
    c->row0 = row0;
    c->row1 = row1;
    c->D = num_shifts;
    c->M = min_shift;
    c->sw = square_width;
    c->half = square_width / 2;
    c->variant = variant;
    c->g.W = width;
    c->g.BH = row1 - row0;
    c->g.half = c->half;
    c->g.ER = c->g.BH + 2 * c->half;
    c->g.D = num_shifts;
    c->g.WPR = packed_words_per_row(width, c->half, num_shifts);

    int rc = SM_OK;
    auto fail = [&](int code) {
        sm_destroy(c);
        return code;
    };
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->num_sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
        set_error("sm_create: stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(SM_ERR_CUDA);
    }
    c->own_stream = true;
    size_t n = c->npix(), pw = (size_t)c->g.ER * c->g.WPR;
    // both edge maps (and, in sm_upload_u8, both images) live in ONE allocation each, second right after first,
    // so that sm_edges detects the pair in a single launch (grid z = image)
    if ((rc = dev_alloc(&c->edges[0], 2 * n)) ||
        (rc = dev_alloc(&c->best, n)) || (rc = dev_alloc(&c->web, n)) ||
        (rc = dev_alloc(&c->LA, pw)) || (rc = dev_alloc(&c->LB, pw)) || (rc = dev_alloc(&c->RB, pw)) ||
        (rc = dev_alloc(&c->minmax, 4)))
        return fail(rc);
    if (cudaHostAlloc((void **)&c->minmax_host, 2 * sizeof(int32_t), cudaHostAllocDefault) != cudaSuccess) {
        set_error("sm_create: pinned allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(SM_ERR_NOMEM);
    }
    if ((rc = launch_minmax_arm(c->minmax, c->stream)) < 0) return fail(rc);
    c->edges[1] = c->edges[0] + n;
    // whole-frame contexts run step 3 as well: its buffers belong to the untimed set-up, like
    // the allocations at the top of the reference's algorithm() (stereo.cu:299-306)
    if (row0 == 0 && row1 == frame_height && ((rc = dev_alloc(&c->tmp, n)) || (rc = dev_alloc(&c->out, n))))
        return fail(rc);
    // load the kernels this geometry uses now, not inside the first timed call
    warm_edges(variant);
    warm_pack(variant);
    warm_direct();
    warm_step3();
    if (bitslice_supports(c->half, c->D)) {
        HotArgs a = hot_args(c, {c->best, c->web});
        if ((rc = prepare_bitslice(a, c->num_sms)) < 0) return fail(rc);
        c->occ = rc;
    }
    // the detector's decision table depends on the threshold alone: build it for the reference's default
    // (DEFAULT_THRESHOLD 0.15, stereo.cu:7) here, so that sm_edges at that threshold is one launch; another threshold
    // rebuilds the table on first use
    if ((rc = dev_alloc(&c->edge_lut, edge_lut_words()))) return fail(rc);
    if ((rc = launch_edge_lut(0.15, c->edge_lut, c->stream)) < 0) return fail(rc);
    c->lut_threshold = 0.15;
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) {
        set_error("sm_create: %s", cudaGetErrorString(cudaGetLastError()));
        return fail(SM_ERR_CUDA);
    }
    *out = c;
    return SM_OK;
}

extern "C" int sm_create_band(sm_ctx **ctx, int device, int width, int frame_height, int row0, int row1,
                              int num_shifts, int square_width, int variant)
{
    return sm_create_band_range(ctx, device, width, frame_height, row0, row1, 0, num_shifts, square_width, variant);
}

extern "C" int sm_create_range(sm_ctx **ctx, int device, int width, int height, int min_shift, int num_shifts,
                               int square_width, int variant)
{
    return sm_create_band_range(ctx, device, width, height, 0, height, min_shift, num_shifts, square_width, variant);
}

extern "C" int sm_create(sm_ctx **ctx, int device, int width, int height, int num_shifts,
                         int square_width, int variant)
{
    return sm_create_band_range(ctx, device, width, height, 0, height, 0, num_shifts, square_width, variant);
}

extern "C" int sm_destroy(sm_ctx *c)
{
    if (!c) return SM_OK;
    DeviceGuard guard(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (cudaStream_t st : {c->pipe.up, c->pipe.down})
        if (st) {
            cudaStreamSynchronize(st);
            cudaStreamDestroy(st);
        }
    for (int k = 0; k < sm_ctx::NPIPE; k++) {
        void *pp[] = {c->pipe.img[k], c->pipe.edg[k], c->pipe.web[k], c->pipe.best[k], c->pipe.web8[k],
                      c->pipe.web16[k], c->pipe.best16[k], c->pipe.ru16[k], c->pipe.sub16[k]};
        for (void *p : pp)
            if (p) cudaFree(p);
        for (cudaEvent_t e : {c->pipe.ev_up[k], c->pipe.ev_comp[k], c->pipe.ev_down[k]})
            if (e) cudaEventDestroy(e);
    }
    if (c->edge_lut) cudaFree(c->edge_lut);
    if (c->minmax_host) cudaFreeHost(c->minmax_host);
    void *ptrs[] = {c->img_u8[0], nullptr,      c->img_f64[0], c->img_f64[1], c->edges[0], nullptr,  // [1] = [0] + npix
                    c->best,      c->web,       c->web2,       c->tmp,        c->out,      c->minmax,
                    c->LA,        c->LB,        c->RB,         c->scratch_u8, c->scratch_i32,
                    c->best16,    c->web16,     c->ru16,       c->sub16,      c->carry16};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    if (c->prof_ev) profile_free(c);
    if (c->pack_stream) {
        cudaStreamSynchronize(c->pack_stream);
        cudaStreamDestroy(c->pack_stream);
    }
    if (c->main2_stream) {
        cudaStreamSynchronize(c->main2_stream);
        cudaStreamDestroy(c->main2_stream);
    }
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    for (int k = 0; k < sm_ctx::NPB; k++) {
        if (c->pLA[k]) cudaFree(c->pLA[k]);
        if (c->pLB[k]) cudaFree(c->pLB[k]);
        if (c->pRB[k]) cudaFree(c->pRB[k]);
        if (c->ev_packed[k]) cudaEventDestroy(c->ev_packed[k]);
        if (c->ev_used[k]) cudaEventDestroy(c->ev_used[k]);
        if (c->pBest16[k]) cudaFree(c->pBest16[k]);
        if (c->pCarry16[k]) cudaFree(c->pCarry16[k]);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return SM_OK;
}

extern "C" int sm_set_stream(sm_ctx *c, void *cuda_stream)
{
    SM_ENTER(c);
    if (c->own_stream && c->stream) {
        SM_CUDA(cudaStreamSynchronize(c->stream));
        SM_CUDA(cudaStreamDestroy(c->stream));
    }
    c->stream = (cudaStream_t)cuda_stream;
    c->own_stream = false;
    c->timed = false;
    return SM_OK;
}

extern "C" int sm_set_kernel(sm_ctx *c, int kernel)
{
    SM_ENTER(c);
    SM_REQUIRE(kernel >= SM_KERNEL_AUTO && kernel <= SM_KERNEL_BITSLICE, "sm_set_kernel: unknown kernel");
    c->kernel = kernel;
    return SM_OK;
}

extern "C" int sm_set_option(sm_ctx *c, int option, int value)
{
    SM_ENTER(c);
    switch (option) {
    case SM_OPT_EDGES_FP64: c->edges_fp64_only = value != 0; return SM_OK;
    case SM_OPT_PIPE_GROUP:
        SM_REQUIRE(value >= 0 && value <= 1024, "sm_set_option: pairs per stage must be in [0, 1024]");
        SM_REQUIRE(!c->pipe.ready, "sm_set_option: the batch pipeline of this context is already set up");
        c->pipe_group_opt = value;
        return SM_OK;
    case SM_OPT_ROW_RUNS:
        SM_REQUIRE(value >= 0, "sm_set_option: row runs must be >= 0");
        c->tuned_segs = value;
        return SM_OK;
    default: set_error("sm_set_option: unknown option %d", option); return SM_ERR_ARG;
    }
}

extern "C" int sm_get_info(sm_ctx *c, int what)
{
    SM_ENTER(c);
    switch (what) {
    case SM_INFO_WARPS_PER_SM: return c->occ;
    case SM_INFO_PAIRS_PER_LAUNCH: return c->batch_group_cap;
    case SM_INFO_TMEM_COLUMNS: return bitslice_supports(c->half, c->D) ? bitslice_tmem_columns(hot_args(c, {c->best, c->web})) : 0;
    case SM_INFO_KERNEL_SHAPE: return c->last_launch.shape;
    case SM_INFO_ROW_RUNS: return c->last_launch.row_runs;
    case SM_INFO_EDGE_THRESHOLDS: {
        if (!c->edge_lut || c->lut_threshold < 0.0) return -1;
        uint32_t flag = 0;
        SM_CUDA(cudaMemcpyAsync(&flag, c->edge_lut + edge_lut_words() - 1, sizeof flag, cudaMemcpyDeviceToHost, c->stream));
        SM_CUDA(cudaStreamSynchronize(c->stream));
        return flag != 0u;
    }
    default: set_error("sm_get_info: unknown item %d", what); return SM_ERR_ARG;
    }
}

extern "C" int sm_synchronize(sm_ctx *c)
{
    SM_ENTER(c);
    SM_CUDA(cudaStreamSynchronize(c->stream));
    return SM_OK;
}

// ---- step 0: upload ------------------------------------------------------------------

// rows of the brightness images this context reads: its output rows, the window halo,
// and one more row for the 3x3 edge stencil (SURVEY 8e)
static void image_rows(const sm_ctx *c, int *lo, int *hi)
{
    *lo = c->row0 - c->half - 1;
    *hi = c->row1 + c->half + 1;
}

extern "C" int sm_upload_u8(sm_ctx *c, const uint8_t *first, const uint8_t *second)
{
    SM_ENTER(c);
    SM_REQUIRE(first && second, "sm_upload_u8: NULL image");
    int rc, lo, hi;
    if ((rc = dev_alloc(&c->img_u8[0], 2 * c->npix()))) return rc;
    c->img_u8[1] = c->img_u8[0] + c->npix();
    image_rows(c, &lo, &hi);
    if ((rc = copy_rows_h2d(c, c->img_u8[0], first, lo, hi)) ||
        (rc = copy_rows_h2d(c, c->img_u8[1], second, lo, hi)))
        return rc;
    c->img_kind = 1;
    return SM_OK;
}

extern "C" int sm_upload_f64(sm_ctx *c, const double *first, const double *second)
{
    SM_ENTER(c);
    SM_REQUIRE(first && second, "sm_upload_f64: NULL image");
    int rc, lo, hi;
    if ((rc = dev_alloc(&c->img_f64[0], c->npix())) || (rc = dev_alloc(&c->img_f64[1], c->npix()))) return rc;
    image_rows(c, &lo, &hi);
    if ((rc = copy_rows_h2d(c, c->img_f64[0], first, lo, hi)) ||
        (rc = copy_rows_h2d(c, c->img_f64[1], second, lo, hi)))
        return rc;
    c->img_kind = 2;
    return SM_OK;
}

// ---- step 1: edges -------------------------------------------------------------------

extern "C" int sm_edges(sm_ctx *c, double threshold)
{
    SM_ENTER(c);
    if (c->img_kind == 0) {
        set_error("sm_edges: no image uploaded");
        return SM_ERR_STATE;
    }
    // same range check as the reference driver (stereo.cu:391-394)
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "sm_edges: threshold must be between 0 and 1");
    int ystart = c->row0 - c->half, nrows = c->g.ER;
    if (nrows >= c->FH) {
        ystart = 0;
        nrows = c->FH;
    }
    const bool use_lut = c->img_kind == 1 && !c->edges_fp64_only;
    if (use_lut && c->lut_threshold != threshold) {
        int rc;
        if ((rc = dev_alloc(&c->edge_lut, edge_lut_words()))) return rc;
        if ((rc = launch_edge_lut(threshold, c->edge_lut, c->stream)) < 0) return rc;
        c->lut_threshold = threshold;
    }
    c->planes_valid = false;
    if (use_lut) {
        // both images in one launch, straight into the packed planes of the hot path; the byte maps are written
        // as well (sm_download(SM_EDGES*), debug planes)
        int rc = launch_edges_planes(c->img_u8[0], c->img_u8[1], c->FH, c->row0, c->variant, c->g, c->M, threshold, c->edge_lut,
                                     c->LA, c->LB, c->RB, c->edges[0], c->edges[1], c->stream);
        if (rc < 0) return rc;
        // With a minimum shift the second image's planes start M columns into the frame, so their columns no longer
        // cover the whole second map (columns [0, M - PADL) are in no plane word): that map comes from the byte-map
        // detector, whose decisions are the table path's, bit for bit.
        if (c->M != 0 &&
            (rc = launch_edges<uint8_t>(c->img_u8[1], c->W, c->FH, ystart, nrows, c->variant, threshold, c->edges[1],
                                        c->stream)) < 0)
            return rc;
        c->planes_valid = true;
    } else {
        for (int k = 0; k < 2; k++) {
            int rc;
            if (c->img_kind == 1)
                rc = launch_edges<uint8_t>(c->img_u8[k], c->W, c->FH, ystart, nrows, c->variant, threshold,
                                           c->edges[k], c->stream);
            else
                rc = launch_edges<double>(c->img_f64[k], c->W, c->FH, ystart, nrows, c->variant, threshold,
                                          c->edges[k], c->stream);
            if (rc < 0) return rc;
        }
    }
    c->have_edges = true;
    return SM_OK;
}

extern "C" int sm_set_edges(sm_ctx *c, const uint8_t *first_edges, const uint8_t *second_edges)
{
    SM_ENTER(c);
    SM_REQUIRE(first_edges && second_edges, "sm_set_edges: NULL edge map");
    int rc;
    if ((rc = copy_rows_h2d(c, c->edges[0], first_edges, c->row0 - c->half, c->row1 + c->half)) ||
        (rc = copy_rows_h2d(c, c->edges[1], second_edges, c->row0 - c->half, c->row1 + c->half)))
        return rc;
    c->planes_valid = false;
    c->have_edges = true;
    return SM_OK;
}

// ---- step 2: the hot path --------------------------------------------------------------

extern "C" int sm_match_wta(sm_ctx *c)
{
    SM_ENTER(c);
    if (!c->have_edges) {
        set_error("sm_match_wta: no edges (call sm_edges or sm_set_edges first)");
        return SM_ERR_STATE;
    }
    int rc = run_hot(c, c->edges[0], c->edges[1], {c->best, c->web});
    if (rc) return rc;
    c->have_web = true;
    c->web_may_have_holes = false;
    c->have_web2 = c->have_out = false;
    return SM_OK;
}

extern "C" int sm_match_wta_dev(sm_ctx *c, const uint8_t *d_first_edges, const uint8_t *d_second_edges,
                                int32_t *d_best, int32_t *d_web)
{
    SM_ENTER(c);
    SM_REQUIRE(d_first_edges && d_second_edges && d_best && d_web, "sm_match_wta_dev: NULL pointer");
    return run_hot(c, d_first_edges, d_second_edges, {d_best, d_web});
}

// The batched hot path on device-resident inputs: either byte edge maps (packed by k_pack) or, with
// from_images, the 8-bit images themselves (edges detected straight into the packed planes by k_edges_planes;
// the byte maps never exist).  Producer launches run on a second stream one group ahead of the main kernels.
// Results go to `out` (int32 or 16-bit), pair k's out_stride * k elements further.
static int batch_core(sm_ctx *c, int n_pairs, bool from_images, double threshold, const uint8_t *d_first_edges,
                      const uint8_t *d_second_edges, size_t edge_stride, const Outputs &out, size_t out_stride)
{
    constexpr int NPB = sm_ctx::NPB;
    const size_t pw = (size_t)c->g.ER * c->g.WPR;
    const int kk = hot_kernel(c);
    const bool scratch_best = out.web16 && !out.best16 && stores_best(c);
    if (!c->batch_ready) {
        // Set-up of the batch path.  Every object is created only if it does not exist yet and the ready flag is
        // set last, so that a call that failed half way (out of memory on the plane sets, say) is simply resumed
        // by the next one instead of launching with missing buffers.
        // Pairs per launch: enough that every warp's run of rows is long against its warm-up rows
        if (c->batch_group_cap == 0) {
            c->batch_group_cap = 1;
            if (bitslice_supports(c->half, c->D)) {
                HotArgs a = hot_args(c, out);
                int pmax = 16;
#ifdef SMB_DEV
                if (getenv("SMB_PMAX")) pmax = atoi(getenv("SMB_PMAX"));  // experiment hook, development build only
#endif
                c->batch_group_cap = bitslice_pairs_per_launch(a, c->num_sms, pmax);
            }
        }
        if (!c->pack_stream) SM_CUDA(cudaStreamCreateWithFlags(&c->pack_stream, cudaStreamNonBlocking));
        if (!c->main2_stream) SM_CUDA(cudaStreamCreateWithFlags(&c->main2_stream, cudaStreamNonBlocking));
        if (!c->ev_fork) SM_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        if (!c->ev_join) SM_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
        for (int k = 0; k < NPB; k++) {
            int rc;
            if ((rc = dev_alloc(&c->pLA[k], pw * c->batch_group_cap)) || (rc = dev_alloc(&c->pLB[k], pw * c->batch_group_cap)) ||
                (rc = dev_alloc(&c->pRB[k], pw * c->batch_group_cap)))
                return rc;
            if (!c->ev_packed[k]) SM_CUDA(cudaEventCreateWithFlags(&c->ev_packed[k], cudaEventDisableTiming));
            if (!c->ev_used[k]) SM_CUDA(cudaEventCreateWithFlags(&c->ev_used[k], cudaEventDisableTiming));
        }
        c->batch_ready = true;
    }
    if (scratch_best) {
        // pair k of a launch stores its best k * out_stride elements further, like its web (the 16-bit kernels take
        // the int32 kernels' argument layout: one stride for both arrays)
        const size_t need = out_stride * (size_t)c->batch_group_cap;
        if (need > c->pbest16_elems)
            for (int k = 0; k < NPB; k++)
                if (c->pBest16[k]) {
                    SM_CUDA(cudaFree(c->pBest16[k]));  // (waits for the device: no launch still uses it)
                    c->pBest16[k] = nullptr;
                }
        for (int k = 0; k < NPB; k++) {
            int rc;
            if ((rc = dev_alloc(&c->pBest16[k], need > c->pbest16_elems ? need : c->pbest16_elems))) return rc;
        }
        if (need > c->pbest16_elems) c->pbest16_elems = need;
    }
    const bool with_carry = out.web_sub && sub_needs_carry(c);
    if (with_carry) {
        // as the scratch best: pair k of a launch k * out_stride elements further, one array per plane set
        const size_t need = out_stride * (size_t)c->batch_group_cap;
        if (need > c->pcarry16_elems)
            for (int k = 0; k < NPB; k++)
                if (c->pCarry16[k]) {
                    SM_CUDA(cudaFree(c->pCarry16[k]));  // (waits for the device: no launch still uses it)
                    c->pCarry16[k] = nullptr;
                }
        for (int k = 0; k < NPB; k++) {
            int rc;
            if ((rc = dev_alloc(&c->pCarry16[k], need > c->pcarry16_elems ? need : c->pcarry16_elems))) return rc;
        }
        if (need > c->pcarry16_elems) c->pcarry16_elems = need;
    }
    // the kernel may have been switched since the last call (sm_set_kernel): the literal kernel takes one pair
    // per launch, the bit-sliced one a group
    c->batch_group = kk == SM_KERNEL_BITSLICE ? c->batch_group_cap : 1;
    if (out.runner_up && kk == SM_KERNEL_BITSLICE) {
        // the runner-up kernels may hold fewer warps per SM than the int32 ones the group was sized for: the pairs
        // per launch of their own (never more than the plane sets hold)
        int rc;
        if ((rc = prepare_ru(c)) < 0) return rc;
        if (c->occ_ru != c->occ) {
            HotArgs a = hot_args(c, out);
            a.blocks_per_sm = c->occ_ru;
            const int g = bitslice_pairs_per_launch(a, c->num_sms, c->batch_group_cap);
            c->batch_group = g < c->batch_group_cap ? g : c->batch_group_cap;
        }
    }
    if (out.web_sub && kk == SM_KERNEL_BITSLICE) {
        // the same for the sub-pixel kernels
        int rc;
        if ((rc = prepare_sub(c)) < 0) return rc;
        if (c->occ_sub != c->occ) {
            HotArgs a = hot_args(c, out);
            a.blocks_per_sm = c->occ_sub;
            const int g = bitslice_pairs_per_launch(a, c->num_sms, c->batch_group_cap);
            c->batch_group = g < c->batch_group_cap ? g : c->batch_group_cap;
        }
    }
    const int G = c->batch_group;
    // everything queued on the context's stream so far (the producers of the edge maps) comes first
    SM_CUDA(cudaEventRecord(c->ev0, c->stream));
    SM_CUDA(cudaEventRecord(c->ev_fork, c->stream));
    SM_CUDA(cudaStreamWaitEvent(c->pack_stream, c->ev_fork, 0));
    SM_CUDA(cudaStreamWaitEvent(c->main2_stream, c->ev_fork, 0));
    int launches = 0, group = 0;
    for (int k = 0; k < n_pairs; k += G, group++) {
        const int np = n_pairs - k < G ? n_pairs - k : G;  // pairs in this launch
        const int b = group % NPB;
        int rc;
        if (group >= NPB) SM_CUDA(cudaStreamWaitEvent(c->pack_stream, c->ev_used[b], 0));  // set b is free again
        if (from_images)
            rc = launch_edges_planes(d_first_edges + (size_t)k * edge_stride, d_second_edges + (size_t)k * edge_stride,
                                     c->FH, c->row0, c->variant, c->g, c->M, threshold, c->edge_lut, c->pLA[b], c->pLB[b],
                                     c->pRB[b], nullptr, nullptr, c->pack_stream, np, edge_stride, pw);
        else
            rc = launch_pack(d_first_edges + (size_t)k * edge_stride, d_second_edges + (size_t)k * edge_stride, c->FH,
                             c->row0, c->variant, c->g, c->M, c->pLA[b], c->pLB[b], c->pRB[b], c->pack_stream, np,
                             edge_stride, pw);
        if (rc < 0) return rc;
        launches += rc;
        SM_CUDA(cudaEventRecord(c->ev_packed[b], c->pack_stream));
        // consecutive launches are independent: alternate two streams so that the next main
        // kernel's warps fill the SM slots the previous one frees (no tail / ramp between them)
        cudaStream_t ms = (group & 1) ? c->main2_stream : c->stream;
        SM_CUDA(cudaStreamWaitEvent(ms, c->ev_packed[b], 0));
        cudaEvent_t *pe = (c->prof_ev && c->prof_n < c->prof_cap) ? c->prof_ev + 3 * c->prof_n : nullptr;
        if (pe) {
            SM_CUDA(cudaEventRecord(pe[0], ms));  // pack runs on the other stream: not timed here
            SM_CUDA(cudaEventRecord(pe[1], ms));
        }
        const Outputs o = out.pair((size_t)k, out_stride);
        HotArgs a = hot_args(c, o);
        if (scratch_best) a.best = c->pBest16[b];
        a.LA = c->pLA[b];
        a.LB = c->pLB[b];
        a.RB = c->pRB[b];
        a.npairs = np;
        a.plane_stride = pw;
        a.out_stride = out_stride;
        rc = launch_main(c, a, o.web16 != nullptr, o.runner_up, ms, o.web_sub, with_carry ? c->pCarry16[b] : nullptr);
        if (rc < 0) return rc;
        launches += rc;
        if (pe) {
            SM_CUDA(cudaEventRecord(pe[2], ms));
            c->prof_n++;
        }
        SM_CUDA(cudaEventRecord(c->ev_used[b], ms));
    }
    // join: the context's stream is complete only when both main streams are
    SM_CUDA(cudaEventRecord(c->ev_join, c->main2_stream));
    SM_CUDA(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    SM_CUDA(cudaEventRecord(c->ev1, c->stream));
    c->timed = true;
    c->last_launches = launches;
    return SM_OK;
}

extern "C" int sm_match_wta_dev_batch(sm_ctx *c, int n_pairs, const uint8_t *d_first_edges,
                                      const uint8_t *d_second_edges, size_t edge_stride, int32_t *d_best,
                                      int32_t *d_web, size_t out_stride)
{
    SM_ENTER(c);
    SM_REQUIRE(n_pairs >= 0 && d_first_edges && d_second_edges && d_best && d_web,
               "sm_match_wta_dev_batch: bad arguments");
    SM_REQUIRE(edge_stride >= c->npix() && out_stride >= c->npix(), "sm_match_wta_dev_batch: stride below frame size");
    return batch_core(c, n_pairs, false, 0.0, d_first_edges, d_second_edges, edge_stride, {d_best, d_web}, out_stride);
}

extern "C" int sm_match_wta_dev_batch16(sm_ctx *c, int n_pairs, const uint8_t *d_first_edges,
                                        const uint8_t *d_second_edges, size_t edge_stride, uint16_t *d_best,
                                        uint16_t *d_web, size_t out_stride)
{
    SM_REQUIRE(n_pairs >= 0 && d_first_edges && d_second_edges && d_web, "sm_match_wta_dev_batch16: bad arguments");
    SM_ENTER(c);
    SM_REQUIRE(edge_stride >= c->npix() && out_stride >= c->npix(), "sm_match_wta_dev_batch16: stride below frame size");
    return batch_core(c, n_pairs, false, 0.0, d_first_edges, d_second_edges, edge_stride, {nullptr, nullptr, d_best, d_web},
                      out_stride);
}

extern "C" int sm_match_wta_dev_batch_ru16(sm_ctx *c, int n_pairs, const uint8_t *d_first_edges,
                                           const uint8_t *d_second_edges, size_t edge_stride, uint16_t *d_best,
                                           uint16_t *d_web, uint16_t *d_runner_up, size_t out_stride)
{
    SM_REQUIRE(n_pairs >= 0 && d_first_edges && d_second_edges && d_web && d_runner_up,
               "sm_match_wta_dev_batch_ru16: bad arguments");
    SM_ENTER(c);
    SM_REQUIRE(edge_stride >= c->npix() && out_stride >= c->npix(), "sm_match_wta_dev_batch_ru16: stride below frame size");
    return batch_core(c, n_pairs, false, 0.0, d_first_edges, d_second_edges, edge_stride,
                      {nullptr, nullptr, d_best, d_web, d_runner_up}, out_stride);
}

extern "C" int sm_match_wta_dev_batch_sub16(sm_ctx *c, int n_pairs, const uint8_t *d_first_edges,
                                            const uint8_t *d_second_edges, size_t edge_stride, uint16_t *d_best,
                                            uint16_t *d_web, uint16_t *d_web_sub, size_t out_stride)
{
    SM_REQUIRE(n_pairs >= 0 && d_first_edges && d_second_edges && d_web && d_web_sub,
               "sm_match_wta_dev_batch_sub16: bad arguments");
    SM_REQUIRE(c, "sm_match_wta_dev_batch_sub16: NULL context");
    SM_REQUIRE(c->M + c->D <= SUB_MAX_RANGE, "sm_match_wta_dev_batch_sub16: web_sub needs min_shift + num_shifts <= %d",
               SUB_MAX_RANGE);
    SM_ENTER(c);
    SM_REQUIRE(edge_stride >= c->npix() && out_stride >= c->npix(), "sm_match_wta_dev_batch_sub16: stride below frame size");
    Outputs o;
    o.best16 = d_best;
    o.web16 = d_web;
    o.web_sub = d_web_sub;
    return batch_core(c, n_pairs, false, 0.0, d_first_edges, d_second_edges, edge_stride, o, out_stride);
}

extern "C" int sm_elapsed_ms(sm_ctx *c, float *ms)
{
    SM_ENTER(c);
    SM_REQUIRE(ms, "sm_elapsed_ms: NULL");
    if (!c->timed) {
        set_error("sm_elapsed_ms: no hot-path call has been made on this context");
        return SM_ERR_STATE;
    }
    SM_CUDA(cudaEventSynchronize(c->ev1));
    SM_CUDA(cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return SM_OK;
}

extern "C" int sm_last_launches(sm_ctx *c) { return c ? c->last_launches : SM_ERR_ARG; }

extern "C" int sm_profile_begin(sm_ctx *c, int max_calls)
{
    SM_ENTER(c);
    SM_REQUIRE(max_calls >= 0 && max_calls <= (1 << 20), "sm_profile_begin: bad max_calls");
    SM_CUDA(cudaStreamSynchronize(c->stream));
    if (c->prof_ev) profile_free(c);
    if (max_calls == 0) return SM_OK;
    c->prof_ev = (cudaEvent_t *)calloc((size_t)3 * max_calls, sizeof(cudaEvent_t));
    if (!c->prof_ev) {
        set_error("sm_profile_begin: out of memory");
        return SM_ERR_NOMEM;
    }
    c->prof_cap = max_calls;
    for (int k = 0; k < 3 * max_calls; k++) SM_CUDA(cudaEventCreate(&c->prof_ev[k]));
    return SM_OK;
}

extern "C" int sm_profile_read(sm_ctx *c, int *n_calls, double *pack_ms_total, double *main_ms_total)
{
    SM_ENTER(c);
    SM_REQUIRE(n_calls && pack_ms_total && main_ms_total, "sm_profile_read: NULL");
    SM_CUDA(cudaStreamSynchronize(c->stream));
    double p = 0, m = 0;
    for (int k = 0; k < c->prof_n; k++) {
        float a = 0, b = 0;
        SM_CUDA(cudaEventElapsedTime(&a, c->prof_ev[3 * k], c->prof_ev[3 * k + 1]));
        SM_CUDA(cudaEventElapsedTime(&b, c->prof_ev[3 * k + 1], c->prof_ev[3 * k + 2]));
        p += a;
        m += b;
    }
    *n_calls = c->prof_n;
    *pack_ms_total = p;
    *main_ms_total = m;
    c->prof_n = 0;
    return SM_OK;
}

// ---- step 3 ----------------------------------------------------------------------------

extern "C" int sm_fill_web_holes(sm_ctx *c, int times)
{
    SM_ENTER(c);
    if (!c->have_web) {
        set_error("sm_fill_web_holes: no web (call sm_match_wta first)");
        return SM_ERR_STATE;
    }
    SM_REQUIRE(times >= 0, "sm_fill_web_holes: times must be >= 0");
    SM_REQUIRE(c->row0 == 0 && c->row1 == c->FH, "sm_fill_web_holes: whole-frame contexts only");
    if (!c->web_may_have_holes) {
        // fill_web_holes only ever writes where the web is 0 (stereo.cu:238), and the web that
        // sm_match_wta produces is >= 1 everywhere (some shift always equals the maximum,
        // stereo.c:212-219): every one of the `times` passes is the identity (SURVEY 3.4), so
        // the filled web IS the web.  No kernel, no copy.
        c->web_filled = c->web;
        c->have_web2 = true;
        return SM_OK;
    }
    int rc;
    size_t n = c->npix();
    if ((rc = dev_alloc(&c->web2, n)) || (rc = dev_alloc(&c->tmp, n))) return rc;
    // web2 <- web, tmp <- web (stereo.cu:328), then ping-pong (stereo.cu:247-259)
    SM_CUDA(cudaMemcpyAsync(c->web2, c->web, n * 4, cudaMemcpyDeviceToDevice, c->stream));
    SM_CUDA(cudaMemcpyAsync(c->tmp, c->web, n * 4, cudaMemcpyDeviceToDevice, c->stream));
    int32_t *a = c->web2, *b = c->tmp;
    for (int t = 0; t < times; t++) {
        if ((rc = launch_fill_web_holes_step(b, a, c->W, c->FH, c->stream)) < 0) return rc;
        int32_t *s = a;
        a = b;
        b = s;
    }
    c->web2 = a;  // whichever buffer the reference would return as `web`
    c->tmp = b;
    c->web_filled = c->web2;
    c->have_web2 = true;
    return SM_OK;
}

// Step 3 on a caller-supplied web (host, i32): the only way a web with holes (zeros) can
// enter the library; makes fill_web_holes / draw_contour_map usable and testable on their own.
extern "C" int sm_set_web(sm_ctx *c, const int32_t *web)
{
    SM_ENTER(c);
    SM_REQUIRE(web, "sm_set_web: NULL web");
    SM_REQUIRE(c->row0 == 0 && c->row1 == c->FH, "sm_set_web: whole-frame contexts only");
    SM_CUDA(cudaMemcpyAsync(c->web, web, c->npix() * 4, cudaMemcpyHostToDevice, c->stream));
    SM_CUDA(cudaMemsetAsync(c->best, 0, c->npix() * 4, c->stream));
    c->have_web = true;
    c->web_may_have_holes = true;
    c->have_web2 = c->have_out = false;
    return SM_OK;
}

extern "C" int sm_draw_contour_map(sm_ctx *c, int lines, int32_t *web_min, int32_t *web_max)
{
    SM_ENTER(c);
    if (!c->have_web) {
        set_error("sm_draw_contour_map: no web (call sm_match_wta first)");
        return SM_ERR_STATE;
    }
    SM_REQUIRE(c->row0 == 0 && c->row1 == c->FH, "sm_draw_contour_map: whole-frame contexts only");
    const int32_t *web = c->have_web2 ? c->web_filled : c->web;
    int rc;
    if ((rc = dev_alloc(&c->out, c->npix()))) return rc;
    // min/max, its copy to the host and the contour kernel are queued back to back: the kernel takes min and max
    // from the device slot, the host only needs them for the caller and for the degenerate case
    const int cur = c->minmax_cur;
    c->minmax_cur ^= 1;
    const int32_t *slot = c->minmax + 2 * cur;
    if ((rc = launch_minmax(web, c->npix(), c->minmax, cur, c->stream)) < 0) return rc;
    SM_CUDA(cudaMemcpyAsync(c->minmax_host, slot, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if (lines != 0 && (rc = launch_contour(web, c->npix(), slot, lines, c->out, c->stream)) < 0) return rc;
    SM_CUDA(cudaStreamSynchronize(c->stream));
    const int32_t mm[2] = {c->minmax_host[0], c->minmax_host[1]};
    if (web_min) *web_min = mm[0];
    if (web_max) *web_max = mm[1];
    // interval = (max - min) / num_lines (stereo.cu:276-285 -> stereo.c:265-266)
    if (lines == 0 || (mm[1] - mm[0]) / lines == 0) {
        set_error("sm_draw_contour_map: (max %d - min %d) / lines %d is zero; the reference divides by "
                  "zero here", mm[1], mm[0], lines);
        return SM_ERR_DEGENERATE;
    }
    c->have_out = true;
    return SM_OK;
}

// ---- download ----------------------------------------------------------------------------

extern "C" int sm_download(sm_ctx *c, int which, int shift, void *host)
{
    SM_ENTER(c);
    SM_REQUIRE(host, "sm_download: NULL host pointer");
    int rc = SM_OK;
    switch (which) {
    case SM_EDGES1:
    case SM_EDGES2:
        if (!c->have_edges) goto state;
        rc = copy_band_d2h(c, (uint8_t *)host, c->edges[which - SM_EDGES1]);
        break;
    case SM_MATCH:
    case SM_SCORE_ALL:
    case SM_SCORE: {
        if (!c->have_edges) goto state;
        SM_REQUIRE(shift >= c->M && shift - c->M < c->D, "sm_download: shift %d out of [%d, %d)", shift, c->M,
                   c->M + c->D);
        if ((rc = dev_alloc(&c->scratch_u8, c->npix())) || (rc = dev_alloc(&c->scratch_i32, c->npix())))
            return rc;
        rc = launch_pack(c->edges[0], c->edges[1], c->FH, c->row0, c->variant, c->g, c->M, c->LA, c->LB, c->RB,
                         c->stream);
        if (rc < 0) return rc;
        HotArgs a = hot_args(c, Outputs{});
        rc = launch_planes(a, shift - c->M, which == SM_MATCH ? c->scratch_u8 : nullptr,
                           which == SM_SCORE_ALL ? c->scratch_i32 : nullptr,
                           which == SM_SCORE ? c->scratch_i32 : nullptr, c->stream);
        if (rc < 0) return rc;
        rc = which == SM_MATCH ? copy_band_d2h(c, (uint8_t *)host, c->scratch_u8)
                               : copy_band_d2h(c, (int32_t *)host, c->scratch_i32);
        break;
    }
    case SM_BEST:
        if (!c->have_web) goto state;
        rc = copy_band_d2h(c, (int32_t *)host, c->best);
        break;
    case SM_WEB:
        if (!c->have_web) goto state;
        rc = copy_band_d2h(c, (int32_t *)host, c->web);
        break;
    case SM_WEB_FILLED:
        if (!c->have_web2) goto state;
        rc = copy_band_d2h(c, (int32_t *)host, c->web_filled);
        break;
    case SM_OUTPUT:
        if (!c->have_out) goto state;
        rc = copy_band_d2h(c, (uint8_t *)host, c->out);
        break;
    default:
        set_error("sm_download: unknown plane %d", which);
        return SM_ERR_ARG;
    }
    if (rc) return rc;
    SM_CUDA(cudaStreamSynchronize(c->stream));
    return SM_OK;
state:
    set_error("sm_download: plane %d has not been computed yet", which);
    return SM_ERR_STATE;
}

static int queue_web_u8(sm_ctx *c, uint8_t *host)
{
    int rc;
    if ((rc = dev_alloc(&c->scratch_u8, c->npix()))) return rc;
    size_t off = (size_t)c->row0 * c->W, n = (size_t)(c->row1 - c->row0) * c->W;
    if ((rc = launch_narrow(c->web + off, c->scratch_u8 + off, n, c->stream)) < 0) return rc;
    return copy_band_d2h(c, host, c->scratch_u8);
}

extern "C" int sm_download_web_u8(sm_ctx *c, uint8_t *host)
{
    SM_ENTER(c);
    SM_REQUIRE(host, "sm_download_web_u8: NULL host pointer");
    SM_REQUIRE(c->M + c->D <= 255, "sm_download_web_u8: min_shift + num_shifts = %d does not fit 8 bits", c->M + c->D);
    if (!c->have_web) {
        set_error("sm_download_web_u8: no web (call sm_match_wta first)");
        return SM_ERR_STATE;
    }
    int rc = queue_web_u8(c, host);
    if (rc) return rc;
    SM_CUDA(cudaStreamSynchronize(c->stream));
    return SM_OK;
}

extern "C" int sm_download_web_u16(sm_ctx *c, uint16_t *host)
{
    SM_REQUIRE(host, "sm_download_web_u16: NULL host pointer");
    SM_ENTER(c);
    if (!c->have_web) {
        set_error("sm_download_web_u16: no web (call sm_match_wta first)");
        return SM_ERR_STATE;
    }
    int rc;
    if ((rc = dev_alloc(&c->web16, c->npix()))) return rc;
    size_t off = (size_t)c->row0 * c->W, n = (size_t)(c->row1 - c->row0) * c->W;
    if ((rc = launch_narrow(c->web + off, c->web16 + off, n, c->stream)) < 0) return rc;
    if ((rc = copy_band_d2h(c, host, c->web16))) return rc;
    SM_CUDA(cudaStreamSynchronize(c->stream));
    return SM_OK;
}

// ---- whole pairs, batched ----------------------------------------------------------------

// The result formats of the batch entries: int32 web and best; u8 web (narrowed after the hot path) and int32 best;
// 16-bit web and best, written by the hot path itself.
enum WebFormat { WEB_I32, WEB_U8, WEB_U16 };

static size_t web_bytes(WebFormat f) { return f == WEB_U8 ? 1 : (f == WEB_U16 ? 2 : 4); }
static size_t best_bytes(WebFormat f) { return f == WEB_U16 ? 2 : 4; }

// sm_run_batch / sm_run_batch16 / sm_run_batch_ru16 / sm_run_batch_sub16 (fn: the entry's name, for the messages;
// ru_out: the runner-up scores, sub_out: web_sub, WEB_U16 only, not both)
static int run_batch(const char *fn, sm_ctx *c, int n_pairs, const uint8_t *first, const uint8_t *second,
                     double threshold, WebFormat fmt, void *web_out, void *best_out, uint16_t *ru_out = nullptr,
                     uint16_t *sub_out = nullptr)
{
    SM_ENTER(c);
    SM_REQUIRE(n_pairs >= 0 && first && second && web_out, "%s: bad arguments", fn);
    SM_REQUIRE(!ru_out || fmt == WEB_U16, "%s: the runner-up needs 16-bit results", fn);
    SM_REQUIRE(!sub_out || (fmt == WEB_U16 && !ru_out && c->M + c->D <= SUB_MAX_RANGE),
               "%s: web_sub needs 16-bit results and min_shift + num_shifts <= %d", fn, SUB_MAX_RANGE);
    SM_REQUIRE(c->row0 == 0 && c->row1 == c->FH, "%s: whole-frame contexts only", fn);
    SM_REQUIRE(fmt != WEB_U8 || c->M + c->D <= 255, "%s: u8 web needs min_shift + num_shifts <= 255", fn);
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "%s: threshold must be between 0 and 1", fn);
    constexpr int NP = sm_ctx::NPIPE;
    sm_ctx::Pipe &P = c->pipe;
    const size_t n = c->npix();
    int rc;
    if (!P.ready) {  // resumable set-up, ready flag last (see sm_match_wta_dev_batch)
        // pairs per stage: enough for the batched hot path to run in throughput mode, bounded
        // so that the three buffer sets stay small against HBM (16 B per pixel and pair)
        if (P.group == 0) {
            P.group = n <= ((size_t)1 << 22) ? 16 : (n <= ((size_t)1 << 24) ? 8 : 2);
            if (c->pipe_group_opt > 0) P.group = c->pipe_group_opt;
        }
        if (!P.up) SM_CUDA(cudaStreamCreateWithFlags(&P.up, cudaStreamNonBlocking));
        if (!P.down) SM_CUDA(cudaStreamCreateWithFlags(&P.down, cudaStreamNonBlocking));
        for (int k = 0; k < NP; k++) {
            if ((rc = dev_alloc(&P.img[k], 2 * P.group * n))) return rc;
            if (!P.ev_up[k]) SM_CUDA(cudaEventCreateWithFlags(&P.ev_up[k], cudaEventDisableTiming));
            if (!P.ev_comp[k]) SM_CUDA(cudaEventCreateWithFlags(&P.ev_comp[k], cudaEventDisableTiming));
            if (!P.ev_down[k]) SM_CUDA(cudaEventCreateWithFlags(&P.ev_down[k], cudaEventDisableTiming));
        }
        P.ready = true;
    }
    // the hot path's outputs: int32 web and best (narrowed to u8 after it, for WEB_U8), or 16-bit web and, only when
    // the caller wants it, best
    for (int k = 0; k < NP; k++) {
        if (fmt == WEB_U16) {
            if ((rc = dev_alloc(&P.web16[k], P.group * n)) || (best_out && (rc = dev_alloc(&P.best16[k], P.group * n))) ||
                (ru_out && (rc = dev_alloc(&P.ru16[k], P.group * n))) ||
                (sub_out && (rc = dev_alloc(&P.sub16[k], P.group * n))))
                return rc;
        } else if ((rc = dev_alloc(&P.web[k], P.group * n)) || (rc = dev_alloc(&P.best[k], P.group * n))) {
            return rc;
        }
        if (fmt == WEB_U8 && (rc = dev_alloc(&P.web8[k], P.group * n))) return rc;
    }
    const bool use_lut = !c->edges_fp64_only;
    if (!use_lut)  // byte edge maps exist only on the FP64 cross-check path
        for (int k = 0; k < NP; k++)
            if ((rc = dev_alloc(&P.edg[k], 2 * P.group * n))) return rc;
    if (use_lut && c->lut_threshold != threshold) {
        if ((rc = dev_alloc(&c->edge_lut, edge_lut_words()))) return rc;
        if ((rc = launch_edge_lut(threshold, c->edge_lut, c->stream)) < 0) return rc;
        c->lut_threshold = threshold;
    }
    const int G = P.group;
    int stage = 0, launches = 0;
    for (int k = 0; k < n_pairs; k += G, stage++) {
        const int np = n_pairs - k < G ? n_pairs - k : G;
        const int b = stage % NP;
        // ---- stage 1, upload stream: the group's images (contiguous in the caller's arrays).
        // Buffer set b is free once the download of the group that used it last has finished.
        if (stage >= NP) SM_CUDA(cudaStreamWaitEvent(P.up, P.ev_down[b], 0));
        SM_CUDA(cudaMemcpyAsync(P.img[b], first + (size_t)k * n, (size_t)np * n, cudaMemcpyHostToDevice, P.up));
        SM_CUDA(cudaMemcpyAsync(P.img[b] + (size_t)G * n, second + (size_t)k * n, (size_t)np * n,
                                cudaMemcpyHostToDevice, P.up));
        SM_CUDA(cudaEventRecord(P.ev_up[b], P.up));
        // ---- stage 2, the context's stream: edges of all 2*np images, then the batched hot path
        SM_CUDA(cudaStreamWaitEvent(c->stream, P.ev_up[b], 0));
        const Outputs out = fmt == WEB_U16 ? Outputs{nullptr, nullptr, best_out ? P.best16[b] : nullptr, P.web16[b],
                                                     ru_out ? P.ru16[b] : nullptr, sub_out ? P.sub16[b] : nullptr}
                                           : Outputs{P.best[b], P.web[b]};
        if (use_lut) {
            // edges of all 2*np images straight into the packed planes, then the hot path: two kernels per group
            if ((rc = batch_core(c, np, true, threshold, P.img[b], P.img[b] + (size_t)G * n, n, out, n)))
                return rc;
        } else {
            for (int j = 0; j < 2 * G; j++) {
                if (j % G >= np) continue;
                rc = launch_edges<uint8_t>(P.img[b] + (size_t)j * n, c->W, c->FH, 0, c->FH, c->variant, threshold,
                                           P.edg[b] + (size_t)j * n, c->stream);
                if (rc < 0) return rc;
                launches += rc;
            }
            if ((rc = batch_core(c, np, false, 0.0, P.edg[b], P.edg[b] + (size_t)G * n, n, out, n)))
                return rc;
        }
        launches += c->last_launches;
        if (fmt == WEB_U8) {
            if ((rc = launch_narrow(P.web[b], P.web8[b], (size_t)np * n, c->stream)) < 0) return rc;
            launches += rc;
        }
        SM_CUDA(cudaEventRecord(P.ev_comp[b], c->stream));
        // ---- stage 3, download stream: one copy per array
        SM_CUDA(cudaStreamWaitEvent(P.down, P.ev_comp[b], 0));
        const void *web_dev = fmt == WEB_U8 ? (const void *)P.web8[b]
                                            : (fmt == WEB_U16 ? (const void *)P.web16[b] : (const void *)P.web[b]);
        const void *best_dev = fmt == WEB_U16 ? (const void *)P.best16[b] : (const void *)P.best[b];
        const size_t wb = web_bytes(fmt), bb = best_bytes(fmt);
        SM_CUDA(cudaMemcpyAsync((uint8_t *)web_out + (size_t)k * n * wb, web_dev, (size_t)np * n * wb,
                                cudaMemcpyDeviceToHost, P.down));
        if (best_out)
            SM_CUDA(cudaMemcpyAsync((uint8_t *)best_out + (size_t)k * n * bb, best_dev, (size_t)np * n * bb,
                                    cudaMemcpyDeviceToHost, P.down));
        if (ru_out)
            SM_CUDA(cudaMemcpyAsync(ru_out + (size_t)k * n, P.ru16[b], (size_t)np * n * sizeof(uint16_t),
                                    cudaMemcpyDeviceToHost, P.down));
        if (sub_out)
            SM_CUDA(cudaMemcpyAsync(sub_out + (size_t)k * n, P.sub16[b], (size_t)np * n * sizeof(uint16_t),
                                    cudaMemcpyDeviceToHost, P.down));
        SM_CUDA(cudaEventRecord(P.ev_down[b], P.down));
    }
    SM_CUDA(cudaStreamSynchronize(P.up));
    SM_CUDA(cudaStreamSynchronize(c->stream));
    SM_CUDA(cudaStreamSynchronize(P.down));
    c->last_launches = launches;
    return SM_OK;
}

extern "C" int sm_run_batch(sm_ctx *c, int n_pairs, const uint8_t *first, const uint8_t *second,
                            double threshold, void *web_out, int web_u8, int32_t *best_out)
{
    return run_batch(__func__, c, n_pairs, first, second, threshold, web_u8 ? WEB_U8 : WEB_I32, web_out, best_out);
}

extern "C" int sm_run_batch16(sm_ctx *c, int n_pairs, const uint8_t *first, const uint8_t *second,
                              double threshold, uint16_t *web_out, uint16_t *best_out)
{
    // the checks that need no context first (and no device)
    SM_REQUIRE(n_pairs >= 0 && first && second && web_out, "sm_run_batch16: bad arguments");
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "sm_run_batch16: threshold must be between 0 and 1");
    return run_batch(__func__, c, n_pairs, first, second, threshold, WEB_U16, web_out, best_out);
}

extern "C" int sm_run_batch_ru16(sm_ctx *c, int n_pairs, const uint8_t *first, const uint8_t *second,
                                 double threshold, uint16_t *web_out, uint16_t *best_out, uint16_t *runner_up_out)
{
    // the checks that need no context first (and no device)
    SM_REQUIRE(n_pairs >= 0 && first && second && web_out && runner_up_out, "sm_run_batch_ru16: bad arguments");
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "sm_run_batch_ru16: threshold must be between 0 and 1");
    return run_batch(__func__, c, n_pairs, first, second, threshold, WEB_U16, web_out, best_out, runner_up_out);
}

extern "C" int sm_run_batch_sub16(sm_ctx *c, int n_pairs, const uint8_t *first, const uint8_t *second,
                                  double threshold, uint16_t *web_out, uint16_t *best_out, uint16_t *web_sub_out)
{
    // the checks that need no context first (and no device)
    SM_REQUIRE(n_pairs >= 0 && first && second && web_out && web_sub_out, "sm_run_batch_sub16: bad arguments");
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "sm_run_batch_sub16: threshold must be between 0 and 1");
    SM_REQUIRE(c, "sm_run_batch_sub16: NULL context");
    SM_REQUIRE(c->M + c->D <= SUB_MAX_RANGE, "sm_run_batch_sub16: web_sub needs min_shift + num_shifts <= %d",
               SUB_MAX_RANGE);
    return run_batch(__func__, c, n_pairs, first, second, threshold, WEB_U16, web_out, best_out, nullptr, web_sub_out);
}

// ---- whole pairs over several GPUs of one box ------------------------------------------------
//
// SURVEY 8e: pairs shard with no exchange step.  One context and one host thread per device; device d
// takes a contiguous range of the batch (the caller's arrays are contiguous, so every stage of its
// sm_run_batch pipeline stays a single copy).  No cross-device traffic, no collective.

// One persistent host thread per device slot (sm_multi_*, sm_bands_*): created with the object, parked on a
// condition variable between calls, joined at destroy -- no thread is created or joined inside a run call.
namespace {

class SlotWorkers {
public:
    explicit SlotWorkers(int n) : jobs_((size_t)n), state_((size_t)n, 0)
    {
        for (int k = 0; k < n; k++) {
            try {
                threads_.emplace_back([this, k] { loop(k); });
            } catch (...) {  // no thread to be had: that slot's work runs on the calling thread
                break;
            }
        }
    }
    ~SlotWorkers()
    {
        {
            std::lock_guard<std::mutex> lk(mu_);
            quit_ = true;
        }
        cv_.notify_all();
        for (auto &t : threads_) t.join();
    }
    // run job(k) for every slot k and wait for all of them
    void run_all(const std::function<void(int)> &job)
    {
        const int n = (int)jobs_.size(), nt = (int)threads_.size();
        {
            std::lock_guard<std::mutex> lk(mu_);
            for (int k = 0; k < nt; k++) {
                jobs_[(size_t)k] = job;
                state_[(size_t)k] = 1;
            }
        }
        cv_.notify_all();
        for (int k = nt; k < n; k++) job(k);
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [&] {
            for (int k = 0; k < nt; k++)
                if (state_[(size_t)k] != 0) return false;
            return true;
        });
    }

private:
    void loop(int k)
    {
        for (;;) {
            std::function<void(int)> job;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return quit_ || state_[(size_t)k] == 1; });
                if (quit_) return;
                job = jobs_[(size_t)k];
                state_[(size_t)k] = 2;
            }
            job(k);
            {
                std::lock_guard<std::mutex> lk(mu_);
                state_[(size_t)k] = 0;
            }
            done_.notify_all();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_, done_;
    std::vector<std::function<void(int)>> jobs_;
    std::vector<int> state_;  // 0 idle, 1 job posted, 2 running
    std::vector<std::thread> threads_;
    bool quit_ = false;
};

}  // namespace

struct sm_multi {
    int n = 0;
    sm_ctx **ctx = nullptr;
    SlotWorkers *workers = nullptr;
};

extern "C" int sm_multi_create_range(sm_multi **out, const int *devices, int n_devices, int width, int height,
                                     int min_shift, int num_shifts, int square_width, int variant)
{
    SM_REQUIRE(out && devices && n_devices >= 1 && n_devices <= 64, "sm_multi_create: bad arguments");
    *out = nullptr;
    sm_multi *m = new (std::nothrow) sm_multi;
    if (!m) {
        set_error("sm_multi_create: out of memory");
        return SM_ERR_NOMEM;
    }
    m->ctx = (sm_ctx **)calloc((size_t)n_devices, sizeof(sm_ctx *));
    if (!m->ctx) {
        delete m;
        set_error("sm_multi_create: out of memory");
        return SM_ERR_NOMEM;
    }
    m->n = n_devices;
    for (int d = 0; d < n_devices; d++) {
        int rc = sm_create_range(&m->ctx[d], devices[d], width, height, min_shift, num_shifts, square_width, variant);
        if (rc) {
            for (int k = 0; k < d; k++) sm_destroy(m->ctx[k]);
            free(m->ctx);
            delete m;
            return rc;
        }
    }
    m->workers = new (std::nothrow) SlotWorkers(n_devices);
    *out = m;
    return SM_OK;
}

extern "C" int sm_multi_create(sm_multi **out, const int *devices, int n_devices, int width, int height,
                               int num_shifts, int square_width, int variant)
{
    return sm_multi_create_range(out, devices, n_devices, width, height, 0, num_shifts, square_width, variant);
}

extern "C" int sm_multi_destroy(sm_multi *m)
{
    if (!m) return SM_OK;
    delete m->workers;
    for (int d = 0; d < m->n; d++) sm_destroy(m->ctx[d]);
    free(m->ctx);
    delete m;
    return SM_OK;
}

extern "C" int sm_multi_device_count(const sm_multi *m) { return m ? m->n : SM_ERR_ARG; }

// sm_multi_run_batch / sm_multi_run_batch16 / sm_multi_run_batch_ru16 / sm_multi_run_batch_sub16
static int multi_run_batch(const char *fn, sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second,
                           double threshold, WebFormat fmt, void *web_out, void *best_out, uint16_t *ru_out = nullptr,
                           uint16_t *sub_out = nullptr)
{
    SM_REQUIRE(m && n_pairs >= 0 && first && second && web_out, "%s: bad arguments", fn);
    const int N = m->n;
    std::vector<int> rcs((size_t)N, SM_OK);
    std::vector<std::string> errs((size_t)N);
    const size_t n = m->ctx[0]->npix(), wb = web_bytes(fmt), bb = best_bytes(fmt);
    auto work = [&](int d) {
        const int k0 = (int)((long long)n_pairs * d / N), k1 = (int)((long long)n_pairs * (d + 1) / N);
        if (k1 <= k0) return;
        void *wout = (uint8_t *)web_out + (size_t)k0 * n * wb;
        void *bout = best_out ? (void *)((uint8_t *)best_out + (size_t)k0 * n * bb) : nullptr;
        uint16_t *rout = ru_out ? ru_out + (size_t)k0 * n : nullptr;
        uint16_t *sout = sub_out ? sub_out + (size_t)k0 * n : nullptr;
        rcs[(size_t)d] = run_batch(fn, m->ctx[d], k1 - k0, first + (size_t)k0 * n, second + (size_t)k0 * n, threshold, fmt,
                                   wout, bout, rout, sout);
        if (rcs[(size_t)d]) errs[(size_t)d] = sm_last_error();  // the message is per thread: carry it to the caller's
    };
    if (m->workers)
        m->workers->run_all(work);
    else
        for (int d = 0; d < N; d++) work(d);
    for (int d = 0; d < N; d++)
        if (rcs[d]) {
            set_error("%s: device slot %d: %s", fn, d, errs[d].c_str());
            return rcs[d];
        }
    return SM_OK;
}

extern "C" int sm_multi_run_batch(sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second,
                                  double threshold, void *web_out, int web_u8, int32_t *best_out)
{
    return multi_run_batch(__func__, m, n_pairs, first, second, threshold, web_u8 ? WEB_U8 : WEB_I32, web_out, best_out);
}

extern "C" int sm_multi_run_batch16(sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second,
                                    double threshold, uint16_t *web_out, uint16_t *best_out)
{
    return multi_run_batch(__func__, m, n_pairs, first, second, threshold, WEB_U16, web_out, best_out);
}

extern "C" int sm_multi_run_batch_ru16(sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second,
                                       double threshold, uint16_t *web_out, uint16_t *best_out, uint16_t *runner_up_out)
{
    // the checks that need no handle first (and no device)
    SM_REQUIRE(m && n_pairs >= 0 && first && second && web_out && runner_up_out, "sm_multi_run_batch_ru16: bad arguments");
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "sm_multi_run_batch_ru16: threshold must be between 0 and 1");
    return multi_run_batch(__func__, m, n_pairs, first, second, threshold, WEB_U16, web_out, best_out, runner_up_out);
}

extern "C" int sm_multi_run_batch_sub16(sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second,
                                        double threshold, uint16_t *web_out, uint16_t *best_out, uint16_t *web_sub_out)
{
    // the checks that need no handle first (and no device)
    SM_REQUIRE(m && n_pairs >= 0 && first && second && web_out && web_sub_out, "sm_multi_run_batch_sub16: bad arguments");
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "sm_multi_run_batch_sub16: threshold must be between 0 and 1");
    SM_REQUIRE(m->ctx[0]->M + m->ctx[0]->D <= SUB_MAX_RANGE,
               "sm_multi_run_batch_sub16: web_sub needs min_shift + num_shifts <= %d", SUB_MAX_RANGE);
    return multi_run_batch(__func__, m, n_pairs, first, second, threshold, WEB_U16, web_out, best_out, nullptr,
                           web_sub_out);
}

// ---- one pair, row bands over several GPUs of one box ----------------------------------------------
//
// SURVEY 8e, BASELINE config 3: GPU g owns output rows sm_band_rows(height, N, g); it uploads those rows of
// both images plus half + 1 halo rows per side (wrapped for WRAP, clipped for GHOST), detects the edges of its
// rows plus half, runs the hot path on its band and writes only its own rows of web / best into the caller's
// frame-sized host arrays.  One band context and one host thread per device slot; no exchange step.

struct sm_bands {
    int n = 0;
    sm_ctx **ctx = nullptr;
    SlotWorkers *workers = nullptr;
};

extern "C" int sm_bands_destroy(sm_bands *b)
{
    if (!b) return SM_OK;
    delete b->workers;
    for (int d = 0; d < b->n; d++) sm_destroy(b->ctx[d]);
    free(b->ctx);
    delete b;
    return SM_OK;
}

extern "C" int sm_bands_create_range(sm_bands **out, const int *devices, int n_devices, int width, int height,
                                     int min_shift, int num_shifts, int square_width, int variant)
{
    SM_REQUIRE(out && devices && n_devices >= 1 && n_devices <= 64, "sm_bands_create: bad arguments");
    SM_REQUIRE(height >= n_devices, "sm_bands_create: fewer rows than bands");
    *out = nullptr;
    sm_bands *b = new (std::nothrow) sm_bands;
    if (!b) {
        set_error("sm_bands_create: out of memory");
        return SM_ERR_NOMEM;
    }
    b->ctx = (sm_ctx **)calloc((size_t)n_devices, sizeof(sm_ctx *));
    if (!b->ctx) {
        delete b;
        set_error("sm_bands_create: out of memory");
        return SM_ERR_NOMEM;
    }
    b->n = n_devices;
    for (int d = 0; d < n_devices; d++) {
        int r0 = 0, r1 = 0;
        int rc = sm_band_rows(height, n_devices, d, &r0, &r1);
        if (!rc)
            rc = sm_create_band_range(&b->ctx[d], devices[d], width, height, r0, r1, min_shift, num_shifts, square_width,
                                      variant);
        if (rc) {
            sm_bands_destroy(b);  // sm_destroy(NULL) is a no-op for the slots not created yet
            return rc;
        }
    }
    b->workers = new (std::nothrow) SlotWorkers(n_devices);
    *out = b;
    return SM_OK;
}

extern "C" int sm_bands_create(sm_bands **out, const int *devices, int n_devices, int width, int height,
                               int num_shifts, int square_width, int variant)
{
    return sm_bands_create_range(out, devices, n_devices, width, height, 0, num_shifts, square_width, variant);
}

// One band context's 16-bit run: the hot path writes rows [row0, row1) of the context's frame-sized u16 arrays
// (best16 when the caller wants best or the kernel stores it anyway; ru16 with ru_out); only those rows are downloaded.
// (sub16 with sub_out)
static int band_run16(sm_ctx *c, uint16_t *web_out, uint16_t *best_out, uint16_t *ru_out, uint16_t *sub_out)
{
    SM_ENTER(c);
    int rc;
    const bool with_best = best_out || stores_best(c);
    if ((rc = dev_alloc(&c->web16, c->npix())) || (with_best && (rc = dev_alloc(&c->best16, c->npix()))) ||
        (ru_out && (rc = dev_alloc(&c->ru16, c->npix()))) || (sub_out && (rc = dev_alloc(&c->sub16, c->npix()))))
        return rc;
    if ((rc = run_hot(c, c->edges[0], c->edges[1],
                      {nullptr, nullptr, with_best ? c->best16 : nullptr, c->web16, ru_out ? c->ru16 : nullptr,
                       sub_out ? c->sub16 : nullptr})))
        return rc;
    if ((rc = copy_band_d2h(c, web_out, c->web16)) || (best_out && (rc = copy_band_d2h(c, best_out, c->best16))) ||
        (ru_out && (rc = copy_band_d2h(c, ru_out, c->ru16))) || (sub_out && (rc = copy_band_d2h(c, sub_out, c->sub16))))
        return rc;
    SM_CUDA(cudaStreamSynchronize(c->stream));
    return SM_OK;
}

// sm_bands_run / sm_bands_run16 / sm_bands_run_ru16 / sm_bands_run_sub16
static int bands_run(const char *fn, sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                     WebFormat fmt, void *web_out, void *best_out, uint16_t *ru_out = nullptr, uint16_t *sub_out = nullptr)
{
    SM_REQUIRE(b && first && second && web_out, "%s: bad arguments", fn);
    const int N = b->n;
    std::vector<int> rcs((size_t)N, SM_OK);
    std::vector<std::string> errs((size_t)N);
    auto work = [&](int d) {
        sm_ctx *c = b->ctx[d];
        int rc = sm_upload_u8(c, first, second);  // a band context copies only the rows it needs
        if (!rc) rc = sm_edges(c, threshold);
        if (fmt == WEB_U16) {
            if (!rc) rc = band_run16(c, (uint16_t *)web_out, (uint16_t *)best_out, ru_out, sub_out);
        } else {
            if (!rc) rc = sm_match_wta(c);
            if (!rc) rc = sm_download(c, SM_WEB, 0, web_out);  // ... and writes only its own rows
            if (!rc && best_out) rc = sm_download(c, SM_BEST, 0, best_out);
        }
        rcs[(size_t)d] = rc;
        if (rc) errs[(size_t)d] = sm_last_error();
    };
    if (b->workers)
        b->workers->run_all(work);
    else
        for (int d = 0; d < N; d++) work(d);
    for (int d = 0; d < N; d++)
        if (rcs[d]) {
            set_error("%s: band %d: %s", fn, d, errs[d].c_str());
            return rcs[d];
        }
    return SM_OK;
}

extern "C" int sm_bands_run(sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                            int32_t *web_out, int32_t *best_out)
{
    return bands_run(__func__, b, first, second, threshold, WEB_I32, web_out, best_out);
}

extern "C" int sm_bands_run16(sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                              uint16_t *web_out, uint16_t *best_out)
{
    return bands_run(__func__, b, first, second, threshold, WEB_U16, web_out, best_out);
}

extern "C" int sm_bands_run_ru16(sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                                 uint16_t *web_out, uint16_t *best_out, uint16_t *runner_up_out)
{
    SM_REQUIRE(b && first && second && web_out && runner_up_out, "sm_bands_run_ru16: bad arguments");
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "sm_bands_run_ru16: threshold must be between 0 and 1");
    return bands_run(__func__, b, first, second, threshold, WEB_U16, web_out, best_out, runner_up_out);
}

extern "C" int sm_bands_run_sub16(sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                                  uint16_t *web_out, uint16_t *best_out, uint16_t *web_sub_out)
{
    SM_REQUIRE(b && first && second && web_out && web_sub_out, "sm_bands_run_sub16: bad arguments");
    SM_REQUIRE(threshold >= 0.0 && threshold <= 1.0, "sm_bands_run_sub16: threshold must be between 0 and 1");
    SM_REQUIRE(b->ctx[0]->M + b->ctx[0]->D <= SUB_MAX_RANGE,
               "sm_bands_run_sub16: web_sub needs min_shift + num_shifts <= %d", SUB_MAX_RANGE);
    return bands_run(__func__, b, first, second, threshold, WEB_U16, web_out, best_out, nullptr, web_sub_out);
}
