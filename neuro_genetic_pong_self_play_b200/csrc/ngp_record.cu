// ngp_record.cu -- the recording twins of the fused rollout kernel (ngp_record_matches): every flavour launch_rollout
// (ngp_core.cu) can pick, instantiated with REC = true.  A translation unit of its own so that these five large kernels
// compile in parallel with ngp_core.cu's.
#include "ngp_internal.h"
#include "rollout_kernel.cuh"

RolloutKernel rollout_record_kernel(int flavour)
{
    switch (flavour) {
    case 0: return rollout_kernel<0, false, 384, true>;
    case 1: return rollout_kernel<1, false, 256, true>;
    case 2: return rollout_kernel<1, true, 256, true>;
    case 3: return rollout_kernel<1, true, 384, true>;
    default: return rollout_kernel<1, true, 512, true>;
    }
}
