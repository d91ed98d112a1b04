// k_bitslice_ru_sub.cu -- the bit-sliced hot-path kernel with uint16_t best / web, the runner-up score and web_sub from
// one launch (k_bitslice_ru_sub, k_bitslice.cuh): the same instantiations, picked by the same pick_shape, as
// k_bitslice16.cu's 16-bit family.
#include "k_bitslice.cuh"

namespace smb {

int launch_bitslice_ru_sub(const HotArgs &h, uint16_t *runner_up, uint16_t *web_sub, uint16_t *carry, int num_sms,
                           cudaStream_t s, LaunchRecord *rec)
{
    return dispatch<uint16_t, EXTRA_RU_SUB>(h, num_sms, s, MODE_LAUNCH, rec, runner_up, carry, web_sub);
}

// the counterpart of prepare_bitslice_ru / prepare_bitslice_sub: run once per context, before its first launch with
// both extras
int prepare_bitslice_ru_sub(const HotArgs &h, int num_sms)
{
    return dispatch<uint16_t, EXTRA_RU_SUB>(h, num_sms, nullptr, MODE_PREPARE);
}

}  // namespace smb
