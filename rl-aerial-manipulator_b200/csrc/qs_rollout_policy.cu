// qs_rollout_policy.cu -- the policy forward alone (QS_POLICY_TENSOR, _PIPELINE and AUTO of qs_policy_forward) on the
// warp-specialised pipeline of qs_rollout_impl.cuh, in the configuration that is fastest without the env step: two epilogue warps
// per (slot, quadrant) taking alternate 32-column chunks, one env warp per quadrant (observation staging, sampling, outputs):
// 16 + 4 + 2 warps.
#define QS_RO_NS ro_policy
#define QS_RO_EPI_SPLIT 2
#define QS_RO_ENV_SPLIT 1
#define QS_RO_BUILD_POLICY 1
#include "qs_rollout_impl.cuh"
