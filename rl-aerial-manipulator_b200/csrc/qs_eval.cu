// qs_eval.cu -- episode accounting of stable_baselines3 evaluate_policy on the device, one launch per env step.
//
// Replaces the bookkeeping of stable_baselines3.common.evaluation.evaluate_policy (SB3 2.6.0; reference call site
// initial-implementation-v1/rl_train_vecN.py:42, `evaluate_policy(model, env, 10)`): which finished episodes are recorded, in which
// slot, and when the loop may stop.  The policy forward and the env step stay the shipped kernels (qs_policy_forward /
// qs_policy_forward_philox, qs_step); this kernel runs right after qs_step and reads its flags, ep_return and ep_len.
// The selection rule and its closed form are in qs_eval.cuh.  Traffic: 1 B/env (the flags byte) plus the rows of done envs.
// The completion-step word lives on the device and only the last CTA to finish advances it (ticket, as record_post_kernel in
// qs_gae.cu), so a CUDA graph of many steps can be replayed; `remaining` is what the host polls.
#include "../../include/quadsim.h"
#include "qs_eval.cuh"
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace qs {

constexpr int EVAL_THREADS = 256;
constexpr int64_t EVAL_MAX_BLOCKS = 1184;   // 8 CTAs per SM on 148 SMs; grid-stride beyond

__global__ void __launch_bounds__(EVAL_THREADS) eval_begin_kernel(int64_t n, int32_t* __restrict__ count, int32_t* __restrict__ state,
                                                                  int32_t active) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = tid; e < n; e += stride) count[e] = 0;
    if (tid == 0) {
        state[0] = 0;        // completion step
        state[1] = active;   // remaining
        state[2] = 0;        // ticket
        state[3] = 0;
    }
}

template <typename Real>
__global__ void __launch_bounds__(EVAL_THREADS) eval_record_kernel(EvalSplit s, int64_t n, int64_t offset, int64_t slot_first,
                                                                   const uint8_t* __restrict__ flags, const Real* __restrict__ ep_return,
                                                                   const int32_t* __restrict__ ep_len, int32_t* __restrict__ count,
                                                                   int32_t* __restrict__ state, double* __restrict__ ret_out,
                                                                   int32_t* __restrict__ len_out, uint8_t* __restrict__ flags_out,
                                                                   int32_t* __restrict__ step_out) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    const int32_t step = state[0];                 // advanced only after every CTA has taken its ticket
    int finished = 0;
#pragma unroll 1
    for (int64_t e = tid; e < n; e += stride) {
        const uint8_t f = flags[e];
        if ((f & 3u) == 0u) continue;
        const int64_t gid = offset + e;
        finished += eval_record_env<Real>(s, gid, eval_base(s, gid) - slot_first, step, f, ep_return, ep_len, e, count, ret_out, len_out,
                                          flags_out, step_out);
    }
    // one atomic per warp that brought envs to their target
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) finished += __shfl_down_sync(0xffffffffu, finished, o);
    if ((threadIdx.x & 31) == 0 && finished) atomicSub(state + 1, finished);
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned int* ticket = reinterpret_cast<unsigned int*>(state + 2);
        if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
            *ticket = 0u;
            state[0] = step + 1;
        }
    }
}

thread_local char g_eval_error[256] = "";

static int eval_check(const qs_eval_args* a, const char* what, bool record) {
    const char* why = nullptr;
    if (!a) why = "args is NULL";
    else if (a->n < 1) why = "n must be >= 1";
    else if (a->n_eval_episodes < 1) why = "n_eval_episodes must be >= 1";
    else if (a->env_id_offset < 0 || a->n_global < 1 || a->env_id_offset + a->n > a->n_global) why = "need 0 <= env_id_offset and env_id_offset + n <= n_global";
    else if (a->n > INT32_MAX || a->n_eval_episodes / a->n_global >= INT32_MAX) why = "n and the per-env target must fit in int32";
    else if (!a->count || !a->state) why = "count and state must not be NULL";
    else if (record && (!a->flags || !a->ep_return || !a->ep_len || !a->ret_out || !a->len_out || !a->flags_out || !a->step_out))
        why = "flags, ep_return, ep_len and every output buffer must not be NULL";
    else if (record && a->return_is_f64 != 0 && a->return_is_f64 != 1) why = "return_is_f64 must be 0 or 1";
    if (why) {
        snprintf(g_eval_error, sizeof(g_eval_error), "%s: %s", what, why);
        return QS_EINVAL;
    }
    return QS_OK;
}

static int eval_launched(const char* what) {
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) {
        snprintf(g_eval_error, sizeof(g_eval_error), "%s: %s", what, cudaGetErrorString(err));
        return QS_ECUDA;
    }
    return QS_OK;
}

static unsigned eval_blocks(int64_t n) {
    const int64_t b = (n + EVAL_THREADS - 1) / EVAL_THREADS;
    return (unsigned)(b < EVAL_MAX_BLOCKS ? b : EVAL_MAX_BLOCKS);
}

}  // namespace qs

extern "C" {

const char* qs_eval_last_error(void) { return qs::g_eval_error; }

int qs_eval_begin(const qs_eval_args* a, void* stream) {
    if (int rc = qs::eval_check(a, "qs_eval_begin", false)) return rc;
    const qs::EvalSplit s = qs::eval_split(a->n_eval_episodes, a->n_global);
    qs::eval_begin_kernel<<<qs::eval_blocks(a->n), qs::EVAL_THREADS, 0, (cudaStream_t)stream>>>(
        a->n, a->count, a->state, (int32_t)qs::eval_active(s, a->env_id_offset, a->n));
    return qs::eval_launched("qs_eval_begin");
}

int qs_eval_record(const qs_eval_args* a, void* stream) {
    if (int rc = qs::eval_check(a, "qs_eval_record", true)) return rc;
    const qs::EvalSplit s = qs::eval_split(a->n_eval_episodes, a->n_global);
    const int64_t first = qs::eval_base(s, a->env_id_offset);
    const unsigned blocks = qs::eval_blocks(a->n);
    cudaStream_t st = (cudaStream_t)stream;
    if (a->return_is_f64)
        qs::eval_record_kernel<double><<<blocks, qs::EVAL_THREADS, 0, st>>>(s, a->n, a->env_id_offset, first, a->flags,
                                                                           static_cast<const double*>(a->ep_return), a->ep_len, a->count,
                                                                           a->state, a->ret_out, a->len_out, a->flags_out, a->step_out);
    else
        qs::eval_record_kernel<float><<<blocks, qs::EVAL_THREADS, 0, st>>>(s, a->n, a->env_id_offset, first, a->flags,
                                                                          static_cast<const float*>(a->ep_return), a->ep_len, a->count,
                                                                          a->state, a->ret_out, a->len_out, a->flags_out, a->step_out);
    return qs::eval_launched("qs_eval_record");
}

}  // extern "C"
