// TEST INFRASTRUCTURE ONLY -- the episode accounting of csrc/qs_eval.cuh (what eval_record_kernel runs per env), compiled with g++ so
// that the closed-form targets / slots and the per-step record logic can be checked against SB3's loop on the CPU.
#include "../../rl-aerial-manipulator_b200/csrc/qs_eval.cuh"

using namespace qs;

extern "C" {

int64_t he_target(int64_t E, int64_t G, int64_t i) { return eval_target(eval_split(E, G), i); }
int64_t he_base(int64_t E, int64_t G, int64_t i) { return eval_base(eval_split(E, G), i); }
int64_t he_active(int64_t E, int64_t G, int64_t offset, int64_t n) { return eval_active(eval_split(E, G), offset, n); }

// One qs_eval_record step of a shard, envs in index order; returns how many envs reached their target (what the kernel subtracts
// from `remaining`).
int64_t he_record(int64_t E, int64_t G, int64_t offset, int64_t n, int32_t step, const uint8_t* flags, const void* ep_return,
                  int return_is_f64, const int32_t* ep_len, int32_t* count, double* ret_out, int32_t* len_out, uint8_t* flags_out,
                  int32_t* step_out) {
    const EvalSplit s = eval_split(E, G);
    const int64_t first = eval_base(s, offset);
    int64_t finished = 0;
    for (int64_t e = 0; e < n; ++e) {
        const int64_t gid = offset + e;
        const int64_t slot0 = eval_base(s, gid) - first;
        finished += return_is_f64
            ? eval_record_env<double>(s, gid, slot0, step, flags[e], static_cast<const double*>(ep_return), ep_len, e, count, ret_out,
                                      len_out, flags_out, step_out)
            : eval_record_env<float>(s, gid, slot0, step, flags[e], static_cast<const float*>(ep_return), ep_len, e, count, ret_out,
                                     len_out, flags_out, step_out);
    }
    return finished;
}

}  // extern "C"
