// k_bitslice16.cu -- the bit-sliced hot-path kernel with uint16_t outputs (k_bitslice16, k_bitslice.cuh): the same
// instantiations, picked by the same pick_shape, as k_bitslice.cu's int32 family.
#include "k_bitslice.cuh"

namespace smb {

int launch_bitslice16(const HotArgs &h, int num_sms, cudaStream_t s, LaunchRecord *rec)
{
    return dispatch<uint16_t>(h, num_sms, s, MODE_LAUNCH, rec);
}

// the 16-bit counterpart of prepare_bitslice: run once per context, before its first 16-bit launch
int prepare_bitslice16(const HotArgs &h, int num_sms) { return dispatch<uint16_t>(h, num_sms, nullptr, MODE_PREPARE); }

}  // namespace smb
