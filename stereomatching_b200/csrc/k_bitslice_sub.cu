// k_bitslice_sub.cu -- the bit-sliced hot-path kernel with uint16_t best / web and web_sub, the web in sixteenths of a
// shift (k_bitslice_sub, k_bitslice.cuh): the same instantiations, picked by the same pick_shape, as k_bitslice16.cu's
// 16-bit family.
#include "k_bitslice.cuh"

namespace smb {

int launch_bitslice_sub(const HotArgs &h, uint16_t *web_sub, uint16_t *carry, int num_sms, cudaStream_t s,
                        LaunchRecord *rec)
{
    return dispatch<uint16_t, EXTRA_SUB>(h, num_sms, s, MODE_LAUNCH, rec, web_sub, carry);
}

// the sub-pixel counterpart of prepare_bitslice16: run once per context, before its first sub-pixel launch
int prepare_bitslice_sub(const HotArgs &h, int num_sms)
{
    return dispatch<uint16_t, EXTRA_SUB>(h, num_sms, nullptr, MODE_PREPARE);
}

}  // namespace smb
