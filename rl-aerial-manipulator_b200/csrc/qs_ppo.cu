// qs_ppo.cu -- one PPO minibatch update in ONE kernel: gather -> forward (actor + critic MLP, activations kept in shared memory)
// -> clipped-surrogate / value / entropy loss -> backward -> global-norm clipping -> Adam(eps = 1e-5), parameters updated in
// place in the blob the rollout kernels read (include/quadsim.h, qs_policy_forward layout).
//
// Replaces the body of stable_baselines3 PPO.train() for one minibatch (SB3 2.6.0; reference call sites: model.learn(...) of
// initial-implementation-v1/rl_train_vecN.py:13-36 -- batch_size=128, n_epochs=10, clip_range=0.2, ent_coef=0.01,
// learning_rate=2e-4, net_arch=[128,64,64] Tanh -- and initial-implementation-v2/rl_train.py:38-56):
//     advantages = (adv - mean) / (std + 1e-8)                   (torch.std: Bessel)
//     values, log_prob, entropy = policy.evaluate_actions(obs, actions)
//     ratio = exp(log_prob - old_log_prob)
//     policy_loss = -mean(min(adv * ratio, adv * clamp(ratio, 1 - clip, 1 + clip)))
//     value_loss = mse(returns, values);  entropy_loss = -mean(entropy)
//     loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss
//     loss.backward(); clip_grad_norm_(max_grad_norm); Adam.step()
//
// Shape of the work.  30,5xx parameters, minibatches of 128 (the reference) to 65,536 rows: at 128 rows the update is 23 MFLOP --
// launch- and latency-bound, not FLOP-bound, so the contractions run as FP32 FFMA (bit-faithful float32 accumulation, no
// operand rounding) rather than on tensor cores.  The minibatch is split into tiles of 16 rows over the CTAs of a persistent
// grid (8 CTAs at 128 rows): each CTA keeps both nets' W2/W3 in shared memory (the backward pass reads them along the other
// axis), walks its tiles, and holds its share of every weight gradient in REGISTERS across tiles (68 accumulators per thread).
// Partial gradients go to a per-CTA slab; the last CTA to finish (ticket) sums the slabs in fixed order (deterministic), takes
// the global norm, clips and applies Adam.  With several ranks the kernel stops after the summed gradient (qs_ppo_grad), NCCL
// averages it, and qs_ppo_apply does clipping + Adam.
#include "../../include/quadsim.h"
#include "qs_tc.cuh"

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <new>

struct qs_ppo {
    int device, obs_dim, n_params, max_grid;
    float *m, *v;                   // Adam moments, blob layout
    float* partial;                 // [max_grid][n_params] per-CTA gradient slabs
    double* loss_partial;           // [max_grid][8]
    float* grad;                    // [n_params] summed gradient (qs_ppo_grad output when the caller passes none)
    unsigned int* ticket;
    long long* step;                // Adam step count (device: graph-capturable)
};

struct qs_ppo_pop {
    int device, obs_dim, n_params, max_grid, K;
    float *m, *v;                   // [K][n_params] Adam moments, blob layout
    float* partial;                 // [K][max_grid][n_params] per-CTA gradient slabs
    double* loss_partial;           // [K][max_grid][NSTAT]
    unsigned int* ticket;           // [K]
    long long* step;                // [K] Adam step counts
    qs_ppo_hyper* hyper;            // [K] device copy of the hyper-parameters (qs_ppo_pop_set_hyper)
};

namespace qs {
namespace ppo {

using tc::Blob;
using tc::N1;
using tc::N2;
using tc::N3;
using tc::NACT;

constexpr int THREADS = 512, TS = 16;           // threads per CTA, minibatch rows per tile
constexpr int WPAD = 65;                        // row stride of the shared W2 / W3 copies ([k][j], conflict-free along k and j)
constexpr int NSTAT = 8;                        // loss, pg, vf, ent, grad_norm, clip_fraction, approx_kl, n_rows

thread_local char g_error[256] = "";

struct Args {
    float* params;                  // blob (read; written by the fused Adam tail)
    const float *obs, *actions, *old_logp, *adv, *ret;
    const int64_t* idx;             // minibatch row indices into the flat buffers, or null = rows 0..B-1
    int64_t B;
    qs_ppo_hyper hp;
    float *m, *v;
    float* partial;
    double* loss_partial;
    float* grad_out;                // summed (mean-loss) gradient
    float* stats_out;               // f32[NSTAT] or null
    unsigned int* ticket;
    long long* step;
    int n_params;
    int apply;                      // 1: the last CTA clips + applies Adam; 0: stop after grad_out
};

__device__ __forceinline__ double block_sum(double v, double* scratch) {
    // fixed-order tree: warp shuffles, then warp 0 over the per-warp sums
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) scratch[w] = v;
    __syncthreads();
    if (w == 0) {
        v = l < THREADS / 32 ? scratch[l] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (l == 0) scratch[32] = v;
    }
    __syncthreads();
    return scratch[32];
}

// gradient accumulators of one net held by one thread across all tiles of its CTA
template <int D>
struct Acc {
    static constexpr int KW1 = (D + 3) / 4;
    float w1[KW1], w2[16], w3[8], b1, b2, b3, wh, bh;
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < KW1; ++i) w1[i] = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) w2[i] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) w3[i] = 0.f;
        b1 = b2 = b3 = wh = bh = 0.f;
    }
};

struct Smem {
    float w2[2][N1 * WPAD];
    float w3[2][N2 * WPAD];
    float x[TS][32];
    float h1[TS][N1], h2[TS][N2], h3[TS][N3];
    float d1[TS][N1], d2[TS][N2], d3[TS][N3];
    float dh[TS][NACT];             // dL/d(head output): d mean (actor) / d value in column 0 (critic)
    float dls[TS][NACT];            // per-row contribution to d log_std
    float act[TS][NACT], oldlp[TS], advn[TS], ret[TS];
    int valid[TS];
    double red[40];
    float lsum[NSTAT];
    unsigned int last;
};
static_assert(sizeof(Smem) <= 227 * 1024, "shared memory of one CTA");

// forward of one net for the tile in s.x; leaves h1, h2, h3 and the head outputs (out[TS][NACT], column 0 only for the critic)
template <int D>
__device__ __forceinline__ void net_forward(const float* __restrict__ P, const Blob& B, int net, Smem& s, float (*out)[NACT]) {
    const int tid = threadIdx.x;
    {   // layer 1: D -> 128, thread = (neuron j, 4 rows)
        const int j = tid & (N1 - 1), sg = tid >> 7;
        const float* w = P + B.w1(net);
        float a[4];
        const float b = __ldg(P + B.b1(net) + j);
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = b;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float wk = __ldg(w + k * N1 + j);
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = fmaf(s.x[sg * 4 + i][k], wk, a[i]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) s.h1[sg * 4 + i][j] = tanhf(a[i]);
    }
    __syncthreads();
    {   // layer 2: 128 -> 64, thread = (neuron j, 2 rows)
        const int j = tid & (N2 - 1), sg = tid >> 6;
        const float* w = s.w2[net];
        float a0 = __ldg(P + B.b2(net) + j), a1 = a0;
#pragma unroll 8
        for (int k = 0; k < N1; ++k) {
            const float wk = w[k * WPAD + j];
            a0 = fmaf(s.h1[sg * 2][k], wk, a0);
            a1 = fmaf(s.h1[sg * 2 + 1][k], wk, a1);
        }
        s.h2[sg * 2][j] = tanhf(a0);
        s.h2[sg * 2 + 1][j] = tanhf(a1);
    }
    __syncthreads();
    {   // layer 3: 64 -> 64
        const int j = tid & (N3 - 1), sg = tid >> 6;
        const float* w = s.w3[net];
        float a0 = __ldg(P + B.b3(net) + j), a1 = a0;
#pragma unroll 8
        for (int k = 0; k < N2; ++k) {
            const float wk = w[k * WPAD + j];
            a0 = fmaf(s.h2[sg * 2][k], wk, a0);
            a1 = fmaf(s.h2[sg * 2 + 1][k], wk, a1);
        }
        s.h3[sg * 2][j] = tanhf(a0);
        s.h3[sg * 2 + 1][j] = tanhf(a1);
    }
    __syncthreads();
    if (tid < TS * NACT) {   // head: 64 -> 4 (actor) / 1 (critic, column 0 of the padded head)
        const int r = tid >> 2, a = tid & 3;
        const float* wh = P + B.wh(net);
        float o = __ldg(P + B.bh(net) + a);
#pragma unroll 8
        for (int j = 0; j < N3; ++j) o = fmaf(s.h3[r][j], __ldg(wh + j * NACT + a), o);
        out[r][a] = o;
    }
    __syncthreads();
}

// backward of one net from s.dh (dL/d head output); accumulates this thread's share of the gradients
template <int D>
__device__ __forceinline__ void net_backward(const float* __restrict__ P, const Blob& B, int net, Smem& s, Acc<D>& g) {
    const int tid = threadIdx.x;
    // head: dWh[j][a] += sum_r h3[r][j] dh[r][a]  (256 threads), dbh[a] (4 threads)
    if (tid < N3 * NACT) {
        const int j = tid >> 2, a = tid & 3;
        float acc = 0.f;
#pragma unroll
        for (int r = 0; r < TS; ++r) acc = fmaf(s.h3[r][j], s.dh[r][a], acc);
        g.wh += acc;
    } else if (tid < N3 * NACT + NACT) {
        const int a = tid - N3 * NACT;
        float acc = 0.f;
#pragma unroll
        for (int r = 0; r < TS; ++r) acc += s.dh[r][a];
        g.bh += acc;
    }
    {   // d3[r][j] = (sum_a dh[r][a] Wh[j][a]) (1 - h3^2)
        const int j = tid & (N3 - 1), sg = tid >> 6;
        const float4 w = __ldg(reinterpret_cast<const float4*>(P + B.wh(net)) + j);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int r = sg * 2 + i;
            const float h = s.h3[r][j];
            const float d = s.dh[r][0] * w.x + s.dh[r][1] * w.y + s.dh[r][2] * w.z + s.dh[r][3] * w.w;
            s.d3[r][j] = d * (1.0f - h * h);
        }
    }
    __syncthreads();
    {   // dW3[k][j] += sum_r h2[r][k] d3[r][j]: thread = (j, 8 consecutive k);  db3[j]
        const int j = tid & (N3 - 1), kg = tid >> 6;
        float db = 0.f;
#pragma unroll
        for (int r = 0; r < TS; ++r) {
            const float d = s.d3[r][j];
            db += d;
#pragma unroll
            for (int i = 0; i < 8; ++i) g.w3[i] = fmaf(s.h2[r][kg * 8 + i], d, g.w3[i]);
        }
        if (kg == 0) g.b3 += db;
    }
    {   // d2[r][k] = (sum_j d3[r][j] W3[k][j]) (1 - h2^2)
        const int k = tid & (N2 - 1), sg = tid >> 6;
        const float* w = s.w3[net] + k * WPAD;
        float a0 = 0.f, a1 = 0.f;
#pragma unroll 8
        for (int j = 0; j < N3; ++j) {
            const float wj = w[j];
            a0 = fmaf(s.d3[sg * 2][j], wj, a0);
            a1 = fmaf(s.d3[sg * 2 + 1][j], wj, a1);
        }
        const float h0 = s.h2[sg * 2][k], h1 = s.h2[sg * 2 + 1][k];
        s.d2[sg * 2][k] = a0 * (1.0f - h0 * h0);
        s.d2[sg * 2 + 1][k] = a1 * (1.0f - h1 * h1);
    }
    __syncthreads();
    {   // dW2[k][j] += sum_r h1[r][k] d2[r][j]: thread = (j, 16 consecutive k);  db2[j]
        const int j = tid & (N2 - 1), kg = tid >> 6;
        float db = 0.f;
#pragma unroll
        for (int r = 0; r < TS; ++r) {
            const float d = s.d2[r][j];
            db += d;
#pragma unroll
            for (int i = 0; i < 16; ++i) g.w2[i] = fmaf(s.h1[r][kg * 16 + i], d, g.w2[i]);
        }
        if (kg == 0) g.b2 += db;
    }
    {   // d1[r][k] = (sum_j d2[r][j] W2[k][j]) (1 - h1^2): thread = (k, 4 rows)
        const int k = tid & (N1 - 1), sg = tid >> 7;
        const float* w = s.w2[net] + k * WPAD;
        float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
        for (int j = 0; j < N2; ++j) {
            const float wj = w[j];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = fmaf(s.d2[sg * 4 + i][j], wj, a[i]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float h = s.h1[sg * 4 + i][k];
            s.d1[sg * 4 + i][k] = a[i] * (1.0f - h * h);
        }
    }
    __syncthreads();
    {   // dW1[k][j] += sum_r x[r][k] d1[r][j]: thread = (j, KW1 consecutive k);  db1[j]
        const int j = tid & (N1 - 1), kg = tid >> 7;
        float db = 0.f;
#pragma unroll
        for (int r = 0; r < TS; ++r) {
            const float d = s.d1[r][j];
            db += d;
#pragma unroll
            for (int i = 0; i < Acc<D>::KW1; ++i) g.w1[i] = fmaf(s.x[r][kg * Acc<D>::KW1 + i], d, g.w1[i]);   // x is zero beyond D
        }
        if (kg == 0) g.b1 += db;
    }
    __syncthreads();
}

// this thread's accumulators -> the CTA's slab (blob layout)
template <int D>
__device__ __forceinline__ void store_acc(float* __restrict__ slab, const Blob& B, int net, const Acc<D>& g) {
    const int tid = threadIdx.x;
    {
        const int j = tid & (N1 - 1), kg = tid >> 7;
#pragma unroll
        for (int i = 0; i < Acc<D>::KW1; ++i) {
            const int k = kg * Acc<D>::KW1 + i;
            if (k < D) slab[B.w1(net) + k * N1 + j] = g.w1[i];
        }
        if (kg == 0) slab[B.b1(net) + j] = g.b1;
    }
    {
        const int j = tid & (N2 - 1), kg = tid >> 6;
#pragma unroll
        for (int i = 0; i < 16; ++i) slab[B.w2(net) + (kg * 16 + i) * N2 + j] = g.w2[i];
        if (kg == 0) slab[B.b2(net) + j] = g.b2;
#pragma unroll
        for (int i = 0; i < 8; ++i) slab[B.w3(net) + (kg * 8 + i) * N3 + j] = g.w3[i];
        if (kg == 0) slab[B.b3(net) + j] = g.b3;
    }
    if (tid < N3 * NACT) slab[B.wh(net) + tid] = g.wh;
    else if (tid < N3 * NACT + NACT) slab[B.bh(net) + tid - N3 * NACT] = g.bh;
}

// clip by the global norm and apply Adam to params[p] for this thread's p (g = summed gradient in shared memory)
__device__ __forceinline__ void adam_apply(const Args& a, const float* __restrict__ g, double normsq, float* stats_extra) {
    const float total = (float)sqrt(normsq);
    const float coef = fminf(1.0f, a.hp.max_grad_norm / (total + 1e-6f));
    const long long t = *a.step + 1;
    const double bc1 = 1.0 - pow((double)a.hp.beta1, (double)t), bc2 = 1.0 - pow((double)a.hp.beta2, (double)t);
    const float step_size = (float)((double)a.hp.lr / bc1), rsq_bc2 = (float)(1.0 / sqrt(bc2));
    // four parameters per thread and pass: their m / v / parameter loads are all in flight together (one CTA does this alone)
    for (int p0 = threadIdx.x; p0 < a.n_params; p0 += 4 * THREADS) {
        float m[4], v[4], w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = p0 + u * THREADS;
            const bool ok = p < a.n_params;
            m[u] = ok ? a.m[p] : 0.f; v[u] = ok ? a.v[p] : 0.f; w[u] = ok ? a.params[p] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = p0 + u * THREADS;
            if (p >= a.n_params) continue;
            const float gp = g[p] * coef;
            const float mu = m[u] + (gp - m[u]) * (1.0f - a.hp.beta1);                    // exp_avg.lerp_(grad, 1 - beta1)
            const float vu = v[u] * a.hp.beta2 + (1.0f - a.hp.beta2) * gp * gp;           // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
            a.m[p] = mu;
            a.v[p] = vu;
            const float denom = sqrtf(vu) * rsq_bc2 + a.hp.adam_eps;
            a.params[p] = w[u] - step_size * (mu / denom);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) *a.step = t;
    if (stats_extra && threadIdx.x == 0) *stats_extra = total;
}

// the whole update of one agent by the CTAs blockIdx.x = 0 .. gridDim.x - 1 (the solo kernel and the population kernel)
template <int D>
__device__ __forceinline__ void ppo_update_body(const Args& a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& s = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x;
    const Blob B{D};
    const float* __restrict__ P = a.params;

    // ---- stage W2 / W3 of both nets ([k][j] rows padded to WPAD)
    for (int net = 0; net < 2; ++net) {
        for (int i = tid; i < N1 * N2; i += THREADS) s.w2[net][(i >> 6) * WPAD + (i & 63)] = __ldg(P + B.w2(net) + i);
        for (int i = tid; i < N2 * N3; i += THREADS) s.w3[net][(i >> 6) * WPAD + (i & 63)] = __ldg(P + B.w3(net) + i);
    }
    if (tid < NSTAT) s.lsum[tid] = 0.f;
    // ---- advantage statistics of the whole minibatch (every CTA computes the same numbers in the same order)
    float adv_mean = 0.f, adv_rstd = 1.f;
    if (a.hp.normalize_advantage && a.B > 1) {
        double acc = 0.0;
        for (int64_t i = tid; i < a.B; i += THREADS) acc += (double)__ldg(a.adv + (a.idx ? a.idx[i] : i));
        const double mean = block_sum(acc, s.red) / (double)a.B;
        acc = 0.0;
        for (int64_t i = tid; i < a.B; i += THREADS) {
            const double d = (double)__ldg(a.adv + (a.idx ? a.idx[i] : i)) - mean;
            acc += d * d;
        }
        const double var = block_sum(acc, s.red) / (double)(a.B - 1);
        adv_mean = (float)mean;
        adv_rstd = 1.0f / ((float)sqrt(var) + 1e-8f);
    }
    const float ls[NACT] = {__ldg(P + B.log_std()), __ldg(P + B.log_std() + 1), __ldg(P + B.log_std() + 2), __ldg(P + B.log_std() + 3)};
    const float invB = 1.0f / (float)a.B;

    Acc<D> ga, gc;
    ga.zero();
    gc.zero();
    float g_ls = 0.f;                                              // d log_std[a] (threads 0..3)
    float st_pg = 0.f, st_vf = 0.f, st_clip = 0.f, st_kl = 0.f;    // per-row sums (threads 0..TS-1)
    const int64_t tiles = (a.B + TS - 1) / TS;
    __syncthreads();

    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        // ---- gather the tile
        for (int i = tid; i < TS * 32; i += THREADS) {
            const int r = i >> 5, k = i & 31;
            const int64_t q = tile * TS + r;
            float v = 0.f;
            if (q < a.B && k < D) v = __ldg(a.obs + (a.idx ? a.idx[q] : q) * D + k);
            s.x[r][k] = v;
        }
        if (tid < TS) {
            const int64_t q = tile * TS + tid;
            const bool ok = q < a.B;
            const int64_t row = ok ? (a.idx ? a.idx[q] : q) : 0;
            s.valid[tid] = ok ? 1 : 0;
            const float4 ac = ok ? __ldg(reinterpret_cast<const float4*>(a.actions) + row) : make_float4(0.f, 0.f, 0.f, 0.f);
            s.act[tid][0] = ac.x; s.act[tid][1] = ac.y; s.act[tid][2] = ac.z; s.act[tid][3] = ac.w;
            s.oldlp[tid] = ok ? __ldg(a.old_logp + row) : 0.f;
            s.advn[tid] = ok ? (__ldg(a.adv + row) - adv_mean) * adv_rstd : 0.f;
            s.ret[tid] = ok ? __ldg(a.ret + row) : 0.f;
        }
        __syncthreads();

        // ================= actor =================
        net_forward<D>(P, B, 0, s, s.dh);                          // s.dh holds the action means for a moment
        if (tid < TS) {
            const int r = tid;
            float dmean[NACT] = {0.f, 0.f, 0.f, 0.f}, dl[NACT] = {0.f, 0.f, 0.f, 0.f};
            if (s.valid[r]) {
                float z[NACT], logp = 0.f;
#pragma unroll
                for (int q = 0; q < NACT; ++q) {
                    z[q] = (s.act[r][q] - s.dh[r][q]) * expf(-ls[q]);
                    logp += -0.5f * z[q] * z[q] - ls[q] - 0.9189385332046727f;
                }
                const float lr = logp - s.oldlp[r];
                const float ratio = expf(lr);
                const float A = s.advn[r];
                const float lo = 1.0f - a.hp.clip_range, hi = 1.0f + a.hp.clip_range;
                const float s1 = A * ratio, s2 = A * fminf(fmaxf(ratio, lo), hi);
                const bool inside = ratio >= lo && ratio <= hi;
                st_pg += -fminf(s1, s2);
                st_clip += fabsf(ratio - 1.0f) > a.hp.clip_range ? 1.f : 0.f;
                st_kl += (ratio - 1.0f) - lr;
                const float dlogp = (inside || s1 < s2) ? -(A * ratio) * invB : 0.f;
#pragma unroll
                for (int q = 0; q < NACT; ++q) {
                    dmean[q] = dlogp * z[q] * expf(-ls[q]);
                    dl[q] = dlogp * (z[q] * z[q] - 1.0f);
                }
            }
#pragma unroll
            for (int q = 0; q < NACT; ++q) { s.dh[r][q] = dmean[q]; s.dls[r][q] = dl[q]; }
        }
        __syncthreads();
        if (tid < NACT) {
#pragma unroll
            for (int r = 0; r < TS; ++r) g_ls += s.dls[r][tid];
        }
        net_backward<D>(P, B, 0, s, ga);

        // ================= critic =================
        net_forward<D>(P, B, 1, s, s.dh);                          // column 0 = value
        if (tid < TS) {
            const int r = tid;
            float dv = 0.f;
            if (s.valid[r]) {
                const float e = s.dh[r][0] - s.ret[r];
                st_vf += e * e;
                dv = a.hp.vf_coef * 2.0f * e * invB;
            }
            s.dh[r][0] = dv; s.dh[r][1] = 0.f; s.dh[r][2] = 0.f; s.dh[r][3] = 0.f;
        }
        __syncthreads();
        net_backward<D>(P, B, 1, s, gc);
    }

    // ---- this CTA's slab + loss partials
    float* slab = a.partial + (size_t)blockIdx.x * a.n_params;
    store_acc<D>(slab, B, 0, ga);
    store_acc<D>(slab, B, 1, gc);
    if (tid < NACT) slab[B.log_std() + tid] = g_ls;
    if (tid < TS) {   // fixed-order sum over the TS row threads (all in warp 0)
        float v4[4] = {st_pg, st_vf, st_clip, st_kl};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float v = v4[q];
#pragma unroll
            for (int o = TS / 2; o > 0; o >>= 1) v += __shfl_down_sync(0x0000ffffu, v, o, TS);
            if (tid == 0) a.loss_partial[(size_t)blockIdx.x * NSTAT + q] = (double)v;
        }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s.last = atomicAdd(a.ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if (!s.last) return;
    __threadfence();
    if (tid == 0) *a.ticket = 0u;

    // ---- the last CTA: fixed-order sum of the slabs -> g (shared memory, aliasing the dead tile buffers), norm, [clip + Adam]
    float* g = reinterpret_cast<float*>(smem_raw);                // n_params floats <= sizeof(Smem) (checked on the host)
    double nsq = 0.0;
    __syncthreads();
    for (int p0 = tid; p0 < a.n_params; p0 += 4 * THREADS) {          // four parameters per thread and pass: 4 x grid loads in flight
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
        for (unsigned c = 0; c < gridDim.x; ++c) {                    // slabs in CTA order: the sum is deterministic
            const float* slab_c = a.partial + (size_t)c * a.n_params;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int p = p0 + u * THREADS;
                if (p < a.n_params) acc[u] += __ldcg(slab_c + p);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = p0 + u * THREADS;
            if (p >= a.n_params) continue;
            // the entropy bonus: d(-ent_coef * mean(entropy))/d log_std = -ent_coef
            if (p >= B.log_std()) acc[u] -= a.hp.ent_coef;
            g[p] = acc[u];
            nsq += (double)acc[u] * (double)acc[u];
            if (a.grad_out) a.grad_out[p] = acc[u];
        }
    }
    __shared__ double red2[40];
    nsq = block_sum(nsq, red2);
    __shared__ float st[NSTAT];
    if (tid < 4) {
        double v = 0.0;
        for (unsigned c = 0; c < gridDim.x; ++c) v += __ldcg(a.loss_partial + (size_t)c * NSTAT + tid);
        st[tid] = (float)(v / (double)a.B);
    }
    __syncthreads();
    if (tid == 0 && a.stats_out) {
        const float ent = -(4.0f * (0.5f + 0.9189385332046727f) + ls[0] + ls[1] + ls[2] + ls[3]);
        a.stats_out[0] = st[0] + a.hp.ent_coef * ent + a.hp.vf_coef * st[1];
        a.stats_out[1] = st[0];
        a.stats_out[2] = st[1];
        a.stats_out[3] = ent;
        a.stats_out[4] = (float)sqrt(nsq);
        a.stats_out[5] = st[2];
        a.stats_out[6] = st[3];
        a.stats_out[7] = (float)a.B;
    }
    if (a.apply) adam_apply(a, g, nsq, nullptr);
}

template <int D>
__global__ void __launch_bounds__(THREADS, 1) ppo_update_kernel(const Args a) {
    ppo_update_body<D>(a);
}

// several ranks: clipping + Adam on an already averaged gradient
__global__ void __launch_bounds__(THREADS, 1) ppo_apply_kernel(const Args a, const float* __restrict__ grad) {
    __shared__ double red[40];
    double nsq = 0.0;
    for (int p = threadIdx.x; p < a.n_params; p += THREADS) {
        const double gp = (double)grad[p];
        nsq += gp * gp;
    }
    nsq = block_sum(nsq, red);
    adam_apply(a, grad, nsq, a.stats_out ? a.stats_out + 4 : nullptr);
}

// population: blockIdx.y = agent.  The agent's Args live in shared memory, so the body reads them like the solo kernel's
// parameter-space Args instead of holding 15 per-agent pointers in registers.
struct PopArgs {
    float* params;                  // [K][n_params]
    const float *obs, *actions, *old_logp, *adv, *ret;    // the shared flat rollout buffers
    const int64_t* idx;             // [K][idx_stride]
    int64_t idx_stride, B;
    const qs_ppo_hyper* hp;         // device [K]
    float *m, *v, *partial;         // [K][n_params], [K][n_params], [K][max_grid][n_params]
    double* loss_partial;           // [K][max_grid][NSTAT]
    float* stats_out;               // [K][NSTAT] or null
    unsigned int* ticket;           // [K]
    long long* step;                // [K]
    int n_params, max_grid;
};

template <int D>
__global__ void __launch_bounds__(THREADS, 1) ppo_update_pop_kernel(const PopArgs p) {
    __shared__ Args a;
    if (threadIdx.x == 0) {
        const int k = blockIdx.y;
        const size_t np = (size_t)p.n_params;
        a.params = p.params + k * np;
        a.obs = p.obs; a.actions = p.actions; a.old_logp = p.old_logp; a.adv = p.adv; a.ret = p.ret;
        a.idx = p.idx + k * p.idx_stride;
        a.B = p.B;
        a.hp = p.hp[k];
        a.m = p.m + k * np;
        a.v = p.v + k * np;
        a.partial = p.partial + (size_t)k * p.max_grid * np;
        a.loss_partial = p.loss_partial + (size_t)k * p.max_grid * NSTAT;
        a.grad_out = nullptr;
        a.stats_out = p.stats_out ? p.stats_out + (size_t)k * NSTAT : nullptr;
        a.ticket = p.ticket + k;
        a.step = p.step + k;
        a.n_params = p.n_params;
        a.apply = 1;
    }
    __syncthreads();
    ppo_update_body<D>(a);
}

static int fail(const char* what, cudaError_t err) {
    snprintf(g_error, sizeof(g_error), "%s: %s", what, cudaGetErrorString(err));
    return QS_ECUDA;
}

static int launch_update(qs_ppo* o, float* params, const float* obs, const float* actions, const float* old_logp, const float* adv,
                         const float* ret, const int64_t* idx, int64_t B, const qs_ppo_hyper* hp, float* grad_out, float* stats_out,
                         int apply, cudaStream_t st) {
    Args a;
    memset(&a, 0, sizeof(a));
    a.params = params; a.obs = obs; a.actions = actions; a.old_logp = old_logp; a.adv = adv; a.ret = ret; a.idx = idx; a.B = B;
    a.hp = *hp; a.m = o->m; a.v = o->v; a.partial = o->partial; a.loss_partial = o->loss_partial; a.grad_out = grad_out;
    a.stats_out = stats_out; a.ticket = o->ticket; a.step = o->step; a.n_params = o->n_params; a.apply = apply;
    const int64_t tiles = (B + TS - 1) / TS;
    const unsigned grid = (unsigned)(tiles < o->max_grid ? tiles : o->max_grid);
    cudaError_t err;
    if (o->obs_dim == 20) {
        err = cudaFuncSetAttribute(ppo_update_kernel<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
        if (err == cudaSuccess) ppo_update_kernel<20><<<grid, THREADS, sizeof(Smem), st>>>(a);
    } else {
        err = cudaFuncSetAttribute(ppo_update_kernel<17>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
        if (err == cudaSuccess) ppo_update_kernel<17><<<grid, THREADS, sizeof(Smem), st>>>(a);
    }
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err != cudaSuccess) return fail("ppo_update_kernel", err);
    return QS_OK;
}

static int launch_update_pop(qs_ppo_pop* o, const PopArgs& a, cudaStream_t st) {
    // per agent the grid of the solo kernel (launch_update): min(tiles, max_grid) CTAs, so every agent's tiling and slab-sum
    // order, and with them its arithmetic, are those of qs_ppo_update
    const int64_t tiles = (a.B + TS - 1) / TS;
    const dim3 grid((unsigned)(tiles < o->max_grid ? tiles : o->max_grid), (unsigned)o->K);
    cudaError_t err;
    if (o->obs_dim == 20) {
        err = cudaFuncSetAttribute(ppo_update_pop_kernel<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
        if (err == cudaSuccess) ppo_update_pop_kernel<20><<<grid, THREADS, sizeof(Smem), st>>>(a);
    } else {
        err = cudaFuncSetAttribute(ppo_update_pop_kernel<17>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
        if (err == cudaSuccess) ppo_update_pop_kernel<17><<<grid, THREADS, sizeof(Smem), st>>>(a);
    }
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err != cudaSuccess) return fail("ppo_update_pop_kernel", err);
    return QS_OK;
}

}  // namespace ppo
}  // namespace qs

using namespace qs::ppo;

extern "C" {

const char* qs_ppo_last_error(void) { return g_error; }

void qs_ppo_default_hyper(qs_ppo_hyper* hp) {
    if (!hp) return;
    hp->clip_range = 0.2f; hp->ent_coef = 0.0f; hp->vf_coef = 0.5f; hp->max_grad_norm = 0.5f;
    hp->lr = 3e-4f; hp->beta1 = 0.9f; hp->beta2 = 0.999f; hp->adam_eps = 1e-5f; hp->normalize_advantage = 1; hp->reserved = 0;
}

int qs_ppo_n_params(int obs_dim) { return obs_dim == 17 || obs_dim == 20 ? qs::tc::Blob{obs_dim}.log_std() + NACT : -1; }

int qs_ppo_create(int device, int obs_dim, qs_ppo** out) {
    if (!out || (obs_dim != 17 && obs_dim != 20)) { snprintf(g_error, sizeof(g_error), "qs_ppo_create: bad argument (obs_dim 17 or 20)"); return QS_EINVAL; }
    cudaError_t err = cudaSetDevice(device);
    if (err != cudaSuccess) return fail("qs_ppo_create", err);
    qs_ppo* o = new (std::nothrow) qs_ppo();
    if (!o) { snprintf(g_error, sizeof(g_error), "qs_ppo_create: out of host memory"); return QS_EINVAL; }
    memset(o, 0, sizeof(*o));
    o->device = device; o->obs_dim = obs_dim; o->n_params = qs_ppo_n_params(obs_dim);
    if ((size_t)o->n_params * sizeof(float) > sizeof(Smem)) { delete o; snprintf(g_error, sizeof(g_error), "qs_ppo_create: gradient does not fit the tail's shared memory"); return QS_EINVAL; }
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    o->max_grid = sms > 0 ? sms : 148;
    const size_t pb = sizeof(float) * (size_t)o->n_params;
    if ((err = cudaMalloc(&o->m, pb)) != cudaSuccess || (err = cudaMalloc(&o->v, pb)) != cudaSuccess || (err = cudaMalloc(&o->grad, pb)) != cudaSuccess ||
        (err = cudaMalloc(&o->partial, pb * o->max_grid)) != cudaSuccess ||
        (err = cudaMalloc(&o->loss_partial, sizeof(double) * NSTAT * o->max_grid)) != cudaSuccess ||
        (err = cudaMalloc(&o->ticket, sizeof(unsigned int))) != cudaSuccess || (err = cudaMalloc(&o->step, sizeof(long long))) != cudaSuccess ||
        (err = cudaMemset(o->m, 0, pb)) != cudaSuccess || (err = cudaMemset(o->v, 0, pb)) != cudaSuccess ||
        (err = cudaMemset(o->ticket, 0, sizeof(unsigned int))) != cudaSuccess || (err = cudaMemset(o->step, 0, sizeof(long long))) != cudaSuccess ||
        (err = cudaDeviceSynchronize()) != cudaSuccess) {
        qs_ppo_destroy(o);
        return fail("qs_ppo_create", err);
    }
    *out = o;
    return QS_OK;
}

int qs_ppo_destroy(qs_ppo* o) {
    if (!o) return QS_OK;
    cudaSetDevice(o->device);
    cudaDeviceSynchronize();
    cudaFree(o->m); cudaFree(o->v); cudaFree(o->grad); cudaFree(o->partial); cudaFree(o->loss_partial); cudaFree(o->ticket); cudaFree(o->step);
    delete o;
    return QS_OK;
}

int qs_ppo_state(qs_ppo* o, float** m, float** v, long long** step, float** grad) {
    if (!o) { snprintf(g_error, sizeof(g_error), "qs_ppo_state: null handle"); return QS_EINVAL; }
    if (m) *m = o->m;
    if (v) *v = o->v;
    if (step) *step = o->step;
    if (grad) *grad = o->grad;
    return QS_OK;
}

static int check_batch(const char* who, qs_ppo* o, const void* params, const float* obs, const float* actions, const float* old_logp,
                       const float* adv, const float* ret, int64_t B, const qs_ppo_hyper* hp) {
    if (!o || !params || !obs || !actions || !old_logp || !adv || !ret || !hp || B < 1) {
        snprintf(g_error, sizeof(g_error), "%s: null argument or empty minibatch", who);
        return QS_EINVAL;
    }
    if (reinterpret_cast<uintptr_t>(actions) & 15) { snprintf(g_error, sizeof(g_error), "%s: actions must be 16-byte aligned", who); return QS_EINVAL; }
    const cudaError_t err = cudaSetDevice(o->device);
    if (err != cudaSuccess) return fail(who, err);
    return QS_OK;
}

int qs_ppo_update(qs_ppo* o, float* params, const float* obs, const float* actions, const float* old_logp, const float* advantages,
                  const float* returns, const int64_t* idx, int64_t B, const qs_ppo_hyper* hp, float* stats_out, void* stream) {
    const int rc = check_batch("qs_ppo_update", o, params, obs, actions, old_logp, advantages, returns, B, hp);
    if (rc != QS_OK) return rc;
    return launch_update(o, params, obs, actions, old_logp, advantages, returns, idx, B, hp, nullptr, stats_out, 1, (cudaStream_t)stream);
}

int qs_ppo_grad(qs_ppo* o, const float* params, const float* obs, const float* actions, const float* old_logp, const float* advantages,
                const float* returns, const int64_t* idx, int64_t B, const qs_ppo_hyper* hp, float* grad_out, float* stats_out, void* stream) {
    const int rc = check_batch("qs_ppo_grad", o, params, obs, actions, old_logp, advantages, returns, B, hp);
    if (rc != QS_OK) return rc;
    return launch_update(o, const_cast<float*>(params), obs, actions, old_logp, advantages, returns, idx, B, hp, grad_out ? grad_out : o->grad,
                         stats_out, 0, (cudaStream_t)stream);
}

int qs_ppo_apply(qs_ppo* o, float* params, const float* grad, const qs_ppo_hyper* hp, float* stats_out, void* stream) {
    if (!o || !params || !hp) { snprintf(g_error, sizeof(g_error), "qs_ppo_apply: null argument"); return QS_EINVAL; }
    cudaError_t err = cudaSetDevice(o->device);
    if (err != cudaSuccess) return fail("qs_ppo_apply", err);
    Args a;
    memset(&a, 0, sizeof(a));
    a.params = params; a.hp = *hp; a.m = o->m; a.v = o->v; a.step = o->step; a.n_params = o->n_params; a.stats_out = stats_out;
    ppo_apply_kernel<<<1, THREADS, 0, (cudaStream_t)stream>>>(a, grad ? grad : o->grad);
    err = cudaGetLastError();
    if (err != cudaSuccess) return fail("ppo_apply_kernel", err);
    return QS_OK;
}

int qs_ppo_pop_destroy(qs_ppo_pop* o) {
    if (!o) return QS_OK;
    cudaSetDevice(o->device);
    cudaDeviceSynchronize();
    cudaFree(o->m); cudaFree(o->v); cudaFree(o->partial); cudaFree(o->loss_partial); cudaFree(o->ticket); cudaFree(o->step);
    cudaFree(o->hyper);
    delete o;
    return QS_OK;
}

int qs_ppo_pop_create(int device, int obs_dim, int K, qs_ppo_pop** out) {
    if (!out || (obs_dim != 17 && obs_dim != 20) || K < 1 || K > 65535) {
        snprintf(g_error, sizeof(g_error), "qs_ppo_pop_create: bad argument (obs_dim 17 or 20, 1 <= K <= 65535)");
        return QS_EINVAL;
    }
    cudaError_t err = cudaSetDevice(device);
    if (err != cudaSuccess) return fail("qs_ppo_pop_create", err);
    qs_ppo_pop* o = new (std::nothrow) qs_ppo_pop();
    if (!o) { snprintf(g_error, sizeof(g_error), "qs_ppo_pop_create: out of host memory"); return QS_EINVAL; }
    memset(o, 0, sizeof(*o));
    o->device = device; o->obs_dim = obs_dim; o->n_params = qs_ppo_n_params(obs_dim); o->K = K;
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    o->max_grid = sms > 0 ? sms : 148;
    const size_t pb = sizeof(float) * (size_t)o->n_params * K;
    qs_ppo_hyper* h = new (std::nothrow) qs_ppo_hyper[K];
    if (!h) { delete o; snprintf(g_error, sizeof(g_error), "qs_ppo_pop_create: out of host memory"); return QS_EINVAL; }
    for (int k = 0; k < K; ++k) qs_ppo_default_hyper(h + k);
    if ((err = cudaMalloc(&o->m, pb)) != cudaSuccess || (err = cudaMalloc(&o->v, pb)) != cudaSuccess ||
        (err = cudaMalloc(&o->partial, pb * o->max_grid)) != cudaSuccess ||
        (err = cudaMalloc(&o->loss_partial, sizeof(double) * NSTAT * o->max_grid * K)) != cudaSuccess ||
        (err = cudaMalloc(&o->ticket, sizeof(unsigned int) * K)) != cudaSuccess || (err = cudaMalloc(&o->step, sizeof(long long) * K)) != cudaSuccess ||
        (err = cudaMalloc(&o->hyper, sizeof(qs_ppo_hyper) * K)) != cudaSuccess ||
        (err = cudaMemset(o->m, 0, pb)) != cudaSuccess || (err = cudaMemset(o->v, 0, pb)) != cudaSuccess ||
        (err = cudaMemset(o->ticket, 0, sizeof(unsigned int) * K)) != cudaSuccess ||
        (err = cudaMemset(o->step, 0, sizeof(long long) * K)) != cudaSuccess ||
        (err = cudaMemcpy(o->hyper, h, sizeof(qs_ppo_hyper) * K, cudaMemcpyHostToDevice)) != cudaSuccess ||
        (err = cudaDeviceSynchronize()) != cudaSuccess) {
        delete[] h;
        qs_ppo_pop_destroy(o);
        return fail("qs_ppo_pop_create", err);
    }
    delete[] h;
    *out = o;
    return QS_OK;
}

int qs_ppo_pop_set_hyper(qs_ppo_pop* o, const qs_ppo_hyper* hp, void* stream) {
    if (!o || !hp) { snprintf(g_error, sizeof(g_error), "qs_ppo_pop_set_hyper: null argument"); return QS_EINVAL; }
    cudaError_t err = cudaSetDevice(o->device);
    if (err == cudaSuccess) err = cudaMemcpyAsync(o->hyper, hp, sizeof(qs_ppo_hyper) * o->K, cudaMemcpyHostToDevice, (cudaStream_t)stream);
    if (err != cudaSuccess) return fail("qs_ppo_pop_set_hyper", err);
    return QS_OK;
}

int qs_ppo_pop_state(qs_ppo_pop* o, float** m, float** v, long long** step) {
    if (!o) { snprintf(g_error, sizeof(g_error), "qs_ppo_pop_state: null handle"); return QS_EINVAL; }
    if (m) *m = o->m;
    if (v) *v = o->v;
    if (step) *step = o->step;
    return QS_OK;
}

int qs_ppo_pop_update(qs_ppo_pop* o, float* params, const float* obs, const float* actions, const float* old_logp,
                      const float* advantages, const float* returns, const int64_t* idx, int64_t idx_stride, int64_t B,
                      float* stats_out, void* stream) {
    if (!params || !obs || !actions || !old_logp || !advantages || !returns || !idx || B < 1 || idx_stride < B) {
        snprintf(g_error, sizeof(g_error), "qs_ppo_pop_update: null argument, empty minibatch or idx_stride < B");
        return QS_EINVAL;
    }
    if ((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(actions)) & 15) {
        snprintf(g_error, sizeof(g_error), "qs_ppo_pop_update: params and actions must be 16-byte aligned");
        return QS_EINVAL;
    }
    if ((reinterpret_cast<uintptr_t>(idx) & 7) | (reinterpret_cast<uintptr_t>(stats_out) & 3)) {
        snprintf(g_error, sizeof(g_error), "qs_ppo_pop_update: idx must be 8-byte and stats_out 4-byte aligned");
        return QS_EINVAL;
    }
    if (!o) { snprintf(g_error, sizeof(g_error), "qs_ppo_pop_update: null handle"); return QS_EINVAL; }
    const cudaError_t err = cudaSetDevice(o->device);
    if (err != cudaSuccess) return fail("qs_ppo_pop_update", err);
    PopArgs a;
    memset(&a, 0, sizeof(a));
    a.params = params; a.obs = obs; a.actions = actions; a.old_logp = old_logp; a.adv = advantages; a.ret = returns;
    a.idx = idx; a.idx_stride = idx_stride; a.B = B; a.hp = o->hyper; a.m = o->m; a.v = o->v; a.partial = o->partial;
    a.loss_partial = o->loss_partial; a.stats_out = stats_out; a.ticket = o->ticket; a.step = o->step;
    a.n_params = o->n_params; a.max_grid = o->max_grid;
    return launch_update_pop(o, a, (cudaStream_t)stream);
}

}  // extern "C"
