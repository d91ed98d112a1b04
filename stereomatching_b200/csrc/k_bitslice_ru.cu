// k_bitslice_ru.cu -- the bit-sliced hot-path kernel with uint16_t best / web and the runner-up score (k_bitslice_ru,
// k_bitslice.cuh): the same instantiations, picked by the same pick_shape, as k_bitslice16.cu's 16-bit family.
#include "k_bitslice.cuh"

namespace smb {

int launch_bitslice_ru(const HotArgs &h, uint16_t *runner_up, int num_sms, cudaStream_t s, LaunchRecord *rec)
{
    return dispatch<uint16_t, EXTRA_RU>(h, num_sms, s, MODE_LAUNCH, rec, runner_up);
}

// the runner-up counterpart of prepare_bitslice16: run once per context, before its first runner-up launch
int prepare_bitslice_ru(const HotArgs &h, int num_sms) { return dispatch<uint16_t, EXTRA_RU>(h, num_sms, nullptr, MODE_PREPARE); }

}  // namespace smb
