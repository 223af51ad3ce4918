// qs_eval.cuh -- stable_baselines3.common.evaluation.evaluate_policy's episode selection, per env, as __host__ __device__ code
// (compiled by nvcc for qs_eval.cu and by g++ for the host harness, tests/host_harness/harness_eval.cpp).
//
// SB3 2.6.0: env i of n_envs records its first target(i) = (n_eval_episodes + i) // n_envs finished episodes, in completion order
// (within one step, in env index order), and the loop runs while any env is below its target.  With E = n_eval_episodes,
// G = envs over all shards and E = q*G + r (0 <= r < G), the per-env targets and the first output slot of env i are closed forms:
//     target(i) = q + [i >= G - r]          base(i) = q*i + max(0, i - (G - r))      (base = sum of target(j), j < i)
// so a shard of envs [offset, offset + n) owns slots [base(offset), base(offset + n)) and needs no per-env arrays.
#pragma once
#include <stdint.h>

#ifndef QS_HD   // as in qs_model.cuh
#if defined(__CUDACC__)
#define QS_HD __host__ __device__ __forceinline__
#else
#define QS_HD inline
#endif
#endif

namespace qs {

struct EvalSplit {
    int64_t q, r, G;   // E = q*G + r
};

QS_HD EvalSplit eval_split(int64_t n_eval_episodes, int64_t n_global) {
    return EvalSplit{n_eval_episodes / n_global, n_eval_episodes % n_global, n_global};
}

QS_HD int64_t eval_target(const EvalSplit& s, int64_t i) { return s.q + (i >= s.G - s.r ? 1 : 0); }

QS_HD int64_t eval_base(const EvalSplit& s, int64_t i) {
    const int64_t extra = i - (s.G - s.r);
    return s.q * i + (extra > 0 ? extra : 0);
}

// Envs of [offset, offset + n) with a target > 0 (what `remaining` starts at).
QS_HD int64_t eval_active(const EvalSplit& s, int64_t offset, int64_t n) {
    if (s.q > 0) return n;
    const int64_t lo = offset > s.G - s.r ? offset : s.G - s.r;
    return offset + n > lo ? offset + n - lo : 0;
}

// One env after one env step.  Records the episode that just finished if the env is below its target: slot `slot0 + count`
// (slot0 = base(gid) - base(offset), the env's first slot in the shard's output) gets the Monitor return, length, flags byte and
// the completion step, and `count` is advanced.  Returns true when this record brought the env to its target.
template <typename Real>
QS_HD bool eval_record_env(const EvalSplit& s, int64_t gid, int64_t slot0, int32_t step, uint8_t flags,
                      const Real* ep_return, const int32_t* ep_len, int64_t e, int32_t* count, double* ret_out, int32_t* len_out,
                      uint8_t* flags_out, int32_t* step_out) {
    if ((flags & 3u) == 0u) return false;                       // QS_FLAG_TERMINATED | QS_FLAG_TRUNCATED
    const int64_t target = eval_target(s, gid);
    const int32_t k = count[e];
    if (k >= target) return false;                              // reached its target: keeps stepping, ignored
    const int64_t slot = slot0 + k;
    ret_out[slot] = (double)ep_return[e];
    len_out[slot] = ep_len[e];
    flags_out[slot] = flags;
    step_out[slot] = step;
    count[e] = k + 1;
    return k + 1 == target;
}

}  // namespace qs
