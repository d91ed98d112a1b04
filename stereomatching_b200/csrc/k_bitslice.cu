// k_bitslice.cu -- the bit-sliced hot-path kernel with int32 outputs (k_bitslice), and the geometry queries.
// The kernel itself is k_bitslice.cuh; k_bitslice16.cu builds its 16-bit family.
#include "k_bitslice.cuh"

namespace smb {

// square_width up to 31 (the reference default is 21, stereo.c:8): 5 planes hold a row count of up to 31 and a
// walk of 16 + 2*15 steps fits the walker's 96-bit window; wider windows take the direct kernel.
bool bitslice_supports(int half, int D) { return half >= 0 && half <= 15 && D >= 1 && D <= 512; }

int launch_bitslice(const HotArgs &h, int num_sms, cudaStream_t s, LaunchRecord *rec)
{
    return dispatch<int32_t>(h, num_sms, s, MODE_LAUNCH, rec);
}

// How many pairs of a batch to put into one launch.  Every warp pays 2*half warm-up rows per
// run, so runs should be as long as the frame allows: pairs are added to the launch until one
// warp per strip walks the whole height (measured on config 2: 24 us per pair with one pair
// per launch, 18.3 us with 12 or more).
int bitslice_pairs_per_launch(const HotArgs &h, int num_sms, int max_pairs)
{
    // enough pairs that one launch is about three waves of the warps the SMs hold (HotArgs::blocks_per_sm)
    const int strip_cols = pick_shape(h, num_sms).strip_cols();
    const int N = 2 * h.g.half + 1, strips = (h.g.W + strip_cols - 1) / strip_cols;
    const int want = throughput_run_windows() * N;
    const int segs = (h.g.BH + want - 1) / want > 0 ? (h.g.BH + want - 1) / want : 1;
    const int warps_per_sm = h.blocks_per_sm > 0 ? h.blocks_per_sm : 8;
    int p = 1;
    while (p < max_pairs && strips * segs * p < 3 * num_sms * warps_per_sm) p++;
    return p;
}

// Loads the kernel this geometry will use and sets its shared-memory attribute, so that the first
// sm_match_wta call pays none of that; returns its resident warps per SM (for HotArgs::blocks_per_sm).
int prepare_bitslice(const HotArgs &h, int num_sms) { return dispatch<int32_t>(h, num_sms, nullptr, MODE_PREPARE); }

int bitslice_tmem_columns(const HotArgs &h) { return dispatch<int32_t>(h, 0, nullptr, MODE_TMEM_COLUMNS); }  // (of the 16-pixel-segment flavour)

}  // namespace smb
