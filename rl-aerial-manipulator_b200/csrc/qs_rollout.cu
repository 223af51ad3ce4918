// qs_rollout.cu -- the fused rollout step (qs_rollout_step, qs_policy_prepare): the warp-specialised pipeline of
// qs_rollout_impl.cuh in the configuration the fused step wants -- one epilogue warp per (slot, quadrant), one env warp per
// (slot, quadrant): 8 + 8 + 2 warps, registers re-balanced between the roles with setmaxnreg.
#define QS_RO_NS ro_fused
#define QS_RO_EPI_SPLIT 1
#define QS_RO_ENV_SPLIT 2
#define QS_RO_BUILD_FUSED 1
#include "qs_rollout_impl.cuh"
