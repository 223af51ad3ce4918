// qs_policy.cu -- SB3 MlpPolicy rollout forward as one fused FP32 kernel (CUDA-core FFMA path).
//
// Replaces stable_baselines3 ActorCriticPolicy.forward for PPO("MlpPolicy", net_arch=[128,64,64], Tanh)
// (reference call sites: initial-implementation-v2/rl_train.py:27-53, initial-implementation-v1/rl_train_vecN.py:13-33;
// parameter shapes pinned by the state_dict of the shipped zips, see tests/golden/policy_*.npz):
//   actor  : Linear(D,128) tanh Linear(128,64) tanh Linear(64,64) tanh -> action_net Linear(64,4)
//   critic : Linear(D,128) tanh Linear(128,64) tanh Linear(64,64) tanh -> value_net  Linear(64,1)
//   a = mu + exp(log_std) * eps ;  log_prob = sum_i -0.5*eps_i^2 - log_std_i - 0.5*log(2*pi)
//
// Structure: persistent CTAs (one per SM, 256 threads), all 30.5k parameters resident in shared memory,
// tiles of 64 envs.  Warps 0-3 run the actor, warps 4-7 the critic (two independent 128-thread halves with
// their own named barrier); each layer is a register-tiled GEMM (8 envs x 8 or 4 outputs per thread) with
// k-major activations in shared memory so every operand fetch is a conflict-free LDS.128.
// Optional VecNormalize fusion: observations are normalised with the running statistics while the tile is
// loaded (stable_baselines3 VecNormalize.normalize_obs), so the rollout needs no separate normalise pass.
#include "../../include/quadsim.h"
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

namespace qs {

constexpr int H1 = 128, H2 = 64, H3 = 64, NACT = 4;
constexpr int TILE = 64;          // envs per tile
constexpr int POLICY_THREADS = 256;

// parameter blob (floats).  Weights are stored input-major, i.e. W^T of torch's [out,in]: W[k][out].
struct PolicyLayout {
    int obs;
    __host__ __device__ int w1(int net) const { return net * per_net(); }
    __host__ __device__ int b1(int net) const { return w1(net) + obs * H1; }
    __host__ __device__ int w2(int net) const { return b1(net) + H1; }
    __host__ __device__ int b2(int net) const { return w2(net) + H1 * H2; }
    __host__ __device__ int w3(int net) const { return b2(net) + H2; }
    __host__ __device__ int b3(int net) const { return w3(net) + H2 * H3; }
    __host__ __device__ int wh(int net) const { return b3(net) + H3; }            // actor: [64][4]; critic: [64][4] (col 0 used)
    __host__ __device__ int bh(int net) const { return wh(net) + H3 * NACT; }      // 4 floats
    __host__ __device__ int per_net() const { return obs * H1 + H1 + H1 * H2 + H2 + H2 * H3 + H3 + H3 * NACT + NACT; }
    __host__ __device__ int log_std() const { return 2 * per_net(); }
    __host__ __device__ int total() const { return 2 * per_net() + NACT; }
};

__device__ __forceinline__ float fast_tanh(float x) {
    // tanh(x) = 1 - 2/(exp(2x)+1); ex2.approx + fast divide: abs error ~1e-7, saturates cleanly at +-1
    const float t = __expf(2.0f * x);
    return 1.0f - __fdividef(2.0f, t + 1.0f);
}

__device__ __forceinline__ void half_barrier(int net) {
    asm volatile("bar.sync %0, 128;" ::"r"(net + 1));
}

struct PolicyArgs {
    const float* params;
    const float* obs;        // [n, OBS]
    const float* noise;      // [n, 4] or null (deterministic)
    const double* norm;      // VecNormalize stats [1 + 2*OBS] (count, mean, var) or null
    float* obs_norm_out;     // [n, OBS] normalised obs (what SB3 stores in the rollout buffer) or null
    float* actions;          // [n, 4] unclipped
    float* actions_clipped;  // [n, 4] clipped to the action box, or null
    float* values;           // [n]
    float* logp;             // [n]
    int64_t n;
    float norm_eps, norm_clip;
    float lo[4], hi[4];
};

// One layer for one half: C[64 envs][NOUT] = tanh(A[K][64]^T . W[K][NOUT] + b), written k-major to Hout[NOUT][RS].
// Thread t (0..127): te = t % 8 -> envs {4te..4te+3} U {32+4te..}; to = t / 8 -> OPT = NOUT/16 outputs per thread.
template <int K, int NOUT, int RS>
__device__ __forceinline__ void layer(const float* __restrict__ A /*[K][RS]*/, const float* __restrict__ W /*[K][NOUT]*/,
                                      const float* __restrict__ b, float* __restrict__ Hout /*[NOUT][RS]*/, int t) {
    constexpr int OPT = NOUT / 16;        // 8 (NOUT=128) or 4 (NOUT=64)
    constexpr int NW = OPT / 4;           // LDS.128 per k for the weights
    const int te = t & 7, to = t >> 3;
    float acc[8][OPT];
#pragma unroll
    for (int j = 0; j < OPT; ++j) {
        const int o = (j >> 2) * (NOUT / 2) + to * 4 + (j & 3);
        const float bj = b[o];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i][j] = bj;
    }
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
        const float4 a0 = *reinterpret_cast<const float4*>(A + k * RS + te * 4);
        const float4 a1 = *reinterpret_cast<const float4*>(A + k * RS + 32 + te * 4);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        float w[OPT];
#pragma unroll
        for (int q = 0; q < NW; ++q) {
            const float4 wv = *reinterpret_cast<const float4*>(W + k * NOUT + q * (NOUT / 2) + to * 4);
            w[4 * q] = wv.x; w[4 * q + 1] = wv.y; w[4 * q + 2] = wv.z; w[4 * q + 3] = wv.w;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < OPT; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
#pragma unroll
    for (int j = 0; j < OPT; ++j) {
        const int o = (j >> 2) * (NOUT / 2) + to * 4 + (j & 3);
        float4 v0 = make_float4(fast_tanh(acc[0][j]), fast_tanh(acc[1][j]), fast_tanh(acc[2][j]), fast_tanh(acc[3][j]));
        float4 v1 = make_float4(fast_tanh(acc[4][j]), fast_tanh(acc[5][j]), fast_tanh(acc[6][j]), fast_tanh(acc[7][j]));
        *reinterpret_cast<float4*>(Hout + o * RS + te * 4) = v0;
        *reinterpret_cast<float4*>(Hout + o * RS + 32 + te * 4) = v1;
    }
}

template <int OBS>
__global__ void __launch_bounds__(POLICY_THREADS, 1) policy_forward_ffma_kernel(const PolicyArgs p) {
#include "qs_policy_ffma_body.cuh"
}

// population: blockIdx.y = agent a, whose blob is params + a * pstride and whose rows are [a*n, (a+1)*n) of every row buffer.
// Rows are independent in the body (a fixed k-order per row), so each row is what policy_forward_ffma_kernel computes for it.
struct PolicyPopArgs {
    PolicyArgs p;                    // agent 0's view; n = rows per agent
    int64_t pstride;                 // floats between consecutive agents' blobs
};

template <int OBS>
__global__ void __launch_bounds__(POLICY_THREADS, 1) policy_forward_pop_kernel(const PolicyPopArgs q) {
    const int64_t a = blockIdx.y, r0 = a * q.p.n;
    PolicyArgs p = q.p;
    p.params += a * q.pstride;
    p.obs += r0 * OBS;
    if (p.noise) p.noise += r0 * NACT;
    p.actions += r0 * NACT;
    if (p.actions_clipped) p.actions_clipped += r0 * NACT;
    p.values += r0;
    p.logp += r0;
#include "qs_policy_ffma_body.cuh"
}

static size_t policy_smem_bytes(int obs) {
    const PolicyLayout L{obs};
    const int ptotal = (L.total() + 3) & ~3;
    return sizeof(float) * (size_t)(ptotal + obs * TILE + 2 * (H1 * TILE + H2 * TILE) + TILE * 8);
}

thread_local char g_policy_error[256] = "";

// tensor-core paths: single float16 (qs_policy_tc.cu), split-float16 with float32 accuracy (qs_rollout_policy.cu)
int launch_policy_tc(const float* params, int obs_dim, const float* obs, const float* noise, int64_t n, const double* norm_stats,
                     float norm_eps, float norm_clip, float* obs_norm_out, float* actions, float* actions_clipped,
                     const float* clip_lo, const float* clip_hi, float* values, float* logp, cudaStream_t stream,
                     const char** err_out);
int launch_policy_pipeline(const float* params, int obs_dim, const float* obs, const float* noise, int64_t n, const double* norm_stats,
                           float norm_eps, float norm_clip, float* obs_norm_out, float* actions, float* actions_clipped,
                           const float* clip_lo, const float* clip_hi, float* values, float* logp, cudaStream_t stream,
                           const char** err_out, uint64_t philox_seed = 0, uint64_t* philox_counter = nullptr, int64_t env_id_offset = 0);

}  // namespace qs

using namespace qs;

extern "C" {

int64_t qs_policy_param_count(int obs_dim) { return PolicyLayout{obs_dim}.total(); }

const char* qs_policy_last_error(void) { return g_policy_error; }

int qs_policy_forward(const float* params, int obs_dim, const float* obs, const float* noise, int64_t n,
                      const double* norm_stats, float norm_eps, float norm_clip, float* obs_norm_out,
                      float* actions, float* actions_clipped, const float* clip_lo, const float* clip_hi,
                      float* values, float* logp, int impl, void* stream) {
    if (!params || !obs || !actions || !values || !logp || n < 0 || (obs_dim != 17 && obs_dim != 20)) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward: bad argument (obs_dim must be 17 or 20)");
        return QS_EINVAL;
    }
    if (n == 0) return QS_OK;
    if ((reinterpret_cast<uintptr_t>(obs) | reinterpret_cast<uintptr_t>(noise) | reinterpret_cast<uintptr_t>(actions) |
         reinterpret_cast<uintptr_t>(actions_clipped) | reinterpret_cast<uintptr_t>(obs_norm_out)) & 15) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward: obs, noise, actions, actions_clipped and obs_norm_out must be 16-byte aligned");
        return QS_EINVAL;
    }
    if (impl < 0 || impl > 4) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward: impl must be one of QS_POLICY_*");
        return QS_EINVAL;
    }
    // QS_POLICY_AUTO: the tcgen05 kernel (float32-accurate split-float16 mode) wins once there are enough 128-env tiles
    // to fill the SMs (profiles/r01/policy_paths.md); below that the FFMA kernel's finer 64-env tiles do
    if (impl >= QS_POLICY_TENSOR || (impl == QS_POLICY_AUTO && n >= 16384)) {
        const char* msg = nullptr;
        // QS_POLICY_TENSOR_FAST: the three-chain kernel (qs_policy_tc.cu); the float32-accurate tensor mode (QS_POLICY_TENSOR,
        // _PIPELINE and AUTO): the warp-specialised pipeline (qs_rollout_policy.cu)
        const int rc = impl == QS_POLICY_TENSOR_FAST
                           ? launch_policy_tc(params, obs_dim, obs, noise, n, norm_stats, norm_eps, norm_clip, obs_norm_out, actions,
                                              actions_clipped, clip_lo, clip_hi, values, logp, (cudaStream_t)stream, &msg)
                           : launch_policy_pipeline(params, obs_dim, obs, noise, n, norm_stats, norm_eps, norm_clip, obs_norm_out, actions,
                                                    actions_clipped, clip_lo, clip_hi, values, logp, (cudaStream_t)stream, &msg);
        if (rc != QS_OK && msg) snprintf(g_policy_error, sizeof(g_policy_error), "%s", msg);
        return rc;
    }
    PolicyArgs a;
    a.params = params; a.obs = obs; a.noise = noise; a.norm = norm_stats; a.obs_norm_out = obs_norm_out;
    a.actions = actions; a.actions_clipped = actions_clipped; a.values = values; a.logp = logp; a.n = n;
    a.norm_eps = norm_eps; a.norm_clip = norm_clip;
    for (int i = 0; i < 4; ++i) { a.lo[i] = clip_lo ? clip_lo[i] : -3.4e38f; a.hi[i] = clip_hi ? clip_hi[i] : 3.4e38f; }
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const size_t smem = policy_smem_bytes(obs_dim);
    const int64_t tiles = (n + TILE - 1) / TILE;
    const unsigned grid = (unsigned)(tiles < sms ? tiles : sms);
    cudaError_t err;
    if (obs_dim == 20) {
        err = cudaFuncSetAttribute(policy_forward_ffma_kernel<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err == cudaSuccess) policy_forward_ffma_kernel<20><<<grid, POLICY_THREADS, smem, (cudaStream_t)stream>>>(a);
    } else {
        err = cudaFuncSetAttribute(policy_forward_ffma_kernel<17>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err == cudaSuccess) policy_forward_ffma_kernel<17><<<grid, POLICY_THREADS, smem, (cudaStream_t)stream>>>(a);
    }
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err != cudaSuccess) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward: %s", cudaGetErrorString(err));
        return QS_ECUDA;
    }
    return QS_OK;
}

int qs_policy_forward_pop(const float* params, int obs_dim, int K, const float* obs, const float* noise, int64_t n,
                          float* actions, float* actions_clipped, const float* clip_lo, const float* clip_hi, float* values,
                          float* logp, void* stream) {
    if (!params || !obs || !actions || !values || !logp || n < 0 || K < 1 || K > 65535 || (obs_dim != 17 && obs_dim != 20)) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward_pop: bad argument (obs_dim 17 or 20, 1 <= K <= 65535, n >= 0)");
        return QS_EINVAL;
    }
    if ((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(obs) | reinterpret_cast<uintptr_t>(noise) |
         reinterpret_cast<uintptr_t>(actions) | reinterpret_cast<uintptr_t>(actions_clipped)) & 15) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward_pop: params, obs, noise, actions and actions_clipped must be 16-byte aligned");
        return QS_EINVAL;
    }
    if (n == 0) return QS_OK;
    PolicyPopArgs q;
    PolicyArgs& a = q.p;
    a.params = params; a.obs = obs; a.noise = noise; a.norm = nullptr; a.obs_norm_out = nullptr;
    a.actions = actions; a.actions_clipped = actions_clipped; a.values = values; a.logp = logp; a.n = n;
    a.norm_eps = 0.f; a.norm_clip = 0.f;
    for (int i = 0; i < 4; ++i) { a.lo[i] = clip_lo ? clip_lo[i] : -3.4e38f; a.hi[i] = clip_hi ? clip_hi[i] : 3.4e38f; }
    q.pstride = PolicyLayout{obs_dim}.total();
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const size_t smem = policy_smem_bytes(obs_dim);
    const int64_t tiles = (n + TILE - 1) / TILE;
    const dim3 grid((unsigned)(tiles < sms ? tiles : sms), (unsigned)K);
    cudaError_t err;
    if (obs_dim == 20) {
        err = cudaFuncSetAttribute(policy_forward_pop_kernel<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err == cudaSuccess) policy_forward_pop_kernel<20><<<grid, POLICY_THREADS, smem, (cudaStream_t)stream>>>(q);
    } else {
        err = cudaFuncSetAttribute(policy_forward_pop_kernel<17>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err == cudaSuccess) policy_forward_pop_kernel<17><<<grid, POLICY_THREADS, smem, (cudaStream_t)stream>>>(q);
    }
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err != cudaSuccess) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward_pop: %s", cudaGetErrorString(err));
        return QS_ECUDA;
    }
    return QS_OK;
}

/* qs_policy_forward with the Gaussian noise drawn inside the kernel (tcgen05 pipeline kernel only). */
int qs_policy_forward_philox(const float* params, int obs_dim, const float* obs, int64_t n, uint64_t noise_seed, uint64_t* counter,
                             int64_t env_id_offset, const double* norm_stats, float norm_eps, float norm_clip, float* obs_norm_out,
                             float* actions, float* actions_clipped, const float* clip_lo, const float* clip_hi, float* values,
                             float* logp, void* stream) {
    if (!params || !obs || !actions || !values || !logp || !counter || n < 0 || (obs_dim != 17 && obs_dim != 20)) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward_philox: bad argument (obs_dim 17 or 20; counter = device u64[2])");
        return QS_EINVAL;
    }
    if (n == 0) return QS_OK;
    if ((reinterpret_cast<uintptr_t>(obs) | reinterpret_cast<uintptr_t>(actions) | reinterpret_cast<uintptr_t>(actions_clipped) |
         reinterpret_cast<uintptr_t>(obs_norm_out) | reinterpret_cast<uintptr_t>(counter)) & 15) {
        snprintf(g_policy_error, sizeof(g_policy_error), "qs_policy_forward_philox: obs, actions, actions_clipped, obs_norm_out and counter must be 16-byte aligned");
        return QS_EINVAL;
    }
    const char* msg = nullptr;
    const int rc = launch_policy_pipeline(params, obs_dim, obs, nullptr, n, norm_stats, norm_eps, norm_clip, obs_norm_out, actions, actions_clipped,
                                          clip_lo, clip_hi, values, logp, (cudaStream_t)stream, &msg, noise_seed, counter, env_id_offset);
    if (rc != QS_OK && msg) snprintf(g_policy_error, sizeof(g_policy_error), "%s", msg);
    return rc;
}

}  // extern "C"
