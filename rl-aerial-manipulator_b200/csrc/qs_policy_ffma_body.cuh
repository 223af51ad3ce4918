// qs_policy_ffma_body.cuh -- the statements of the FFMA policy forward kernel (qs_policy.cu), included INSIDE the body of both
// policy_forward_ffma_kernel and policy_forward_pop_kernel.  Computes rows [0, p.n) of the PolicyArgs `p` in scope with the CTAs
// blockIdx.x = 0 .. gridDim.x - 1.  It is a statement fragment rather than a __forceinline__ function because a function boundary
// changes how the compiler unrolls the blob-staging loop, i.e. the SASS of the shipped single-policy kernel.
    constexpr int RS = TILE;                       // activation row stride (floats)
    extern __shared__ __align__(16) float smem[];
    const PolicyLayout L{OBS};
    float* sP = smem;                              // parameters
    const int ptotal = (L.total() + 3) & ~3;
    float* sX = sP + ptotal;                       // [OBS][RS]   normalised obs tile, k-major (shared by both halves)
    float* sHa = sX + OBS * RS;                    // per half: [128][RS] (H1, later H3) and [64][RS] (H2)
    constexpr int HALF_FLOATS = H1 * RS + H2 * RS;
    float* sOut = sHa + 2 * HALF_FLOATS;           // [TILE][8]: 4 means, value
    __shared__ double s_mean[32], s_istd[32];   // float64 like SB3's normalize_obs (see qs_vecnorm.cu)

    const int tid = threadIdx.x;
    for (int i = tid; i < L.total(); i += POLICY_THREADS) sP[i] = __ldg(p.params + i);
    if (tid < OBS) {
        double m = 0.0, is = 1.0;
        if (p.norm) {
            m = p.norm[1 + tid];
            is = 1.0 / sqrt(p.norm[1 + OBS + tid] + (double)p.norm_eps);
        }
        s_mean[tid] = m;
        s_istd[tid] = is;
    }
    __syncthreads();

    const int net = tid >> 7;                      // 0 actor, 1 critic
    const int t = tid & 127;
    float* H1s = sHa + net * HALF_FLOATS;
    float* H2s = H1s + H1 * RS;
    const int64_t n_tiles = (p.n + TILE - 1) / TILE;

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t e0 = tile * TILE;
        const int valid = (int)((p.n - e0) < TILE ? (p.n - e0) : TILE);
        // ---- obs tile: coalesced global read, (normalise), transposed store
        for (int i = tid; i < TILE * OBS; i += POLICY_THREADS) {
            const int e = i / OBS, k = i - e * OBS;
            float x = 0.f;
            if (e < valid) {
                x = __ldcs(p.obs + e0 * OBS + i);
                if (p.norm) {
                    x = (float)(((double)x - s_mean[k]) * s_istd[k]);
                    x = fminf(fmaxf(x, -p.norm_clip), p.norm_clip);
                    if (p.obs_norm_out) p.obs_norm_out[e0 * OBS + i] = x;
                }
            }
            sX[k * RS + e] = x;
        }
        __syncthreads();
        // ---- trunk (per half)
        layer<OBS, H1, RS>(sX, sP + L.w1(net), sP + L.b1(net), H1s, t);
        half_barrier(net);
        layer<H1, H2, RS>(H1s, sP + L.w2(net), sP + L.b2(net), H2s, t);
        half_barrier(net);
        layer<H2, H3, RS>(H2s, sP + L.w3(net), sP + L.b3(net), H1s, t);   // H3 overwrites H1
        half_barrier(net);
        // ---- heads: actor 4 outputs, critic 1; thread t -> env t%64, output pair t/64
        {
            const int e = t & 63, pair = t >> 6;
            const float* Wh = sP + L.wh(net);
            if (net == 0) {
                float m0 = sP[L.bh(0) + 2 * pair], m1 = sP[L.bh(0) + 2 * pair + 1];
#pragma unroll 8
                for (int k = 0; k < H3; ++k) {
                    const float h = H1s[k * RS + e];
                    m0 = fmaf(h, Wh[k * NACT + 2 * pair], m0);
                    m1 = fmaf(h, Wh[k * NACT + 2 * pair + 1], m1);
                }
                sOut[e * 8 + 2 * pair] = m0;
                sOut[e * 8 + 2 * pair + 1] = m1;
            } else if (pair == 0) {
                float v = sP[L.bh(1)];
#pragma unroll 8
                for (int k = 0; k < H3; ++k) v = fmaf(H1s[k * RS + e], Wh[k * NACT], v);
                sOut[e * 8 + 4] = v;
            }
        }
        __syncthreads();
        // ---- sample, log-prob, clip, store (64 threads, one env each; float4 rows -> coalesced)
        if (tid < valid) {
            const int64_t e = e0 + tid;
            const float4 mu = *reinterpret_cast<const float4*>(sOut + tid * 8);
            const float ls[4] = {sP[L.log_std()], sP[L.log_std() + 1], sP[L.log_std() + 2], sP[L.log_std() + 3]};
            float4 eps = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.noise) eps = __ldcs(reinterpret_cast<const float4*>(p.noise) + e);
            float4 a;
            a.x = fmaf(__expf(ls[0]), eps.x, mu.x);
            a.y = fmaf(__expf(ls[1]), eps.y, mu.y);
            a.z = fmaf(__expf(ls[2]), eps.z, mu.z);
            a.w = fmaf(__expf(ls[3]), eps.w, mu.w);
            const float HALF_LOG_2PI = 0.9189385332046727f;
            const float lp = -0.5f * (eps.x * eps.x + eps.y * eps.y + eps.z * eps.z + eps.w * eps.w) - (ls[0] + ls[1] + ls[2] + ls[3]) -
                             4.0f * HALF_LOG_2PI;
            reinterpret_cast<float4*>(p.actions)[e] = a;
            if (p.actions_clipped) {
                float4 c;
                c.x = fminf(fmaxf(a.x, p.lo[0]), p.hi[0]);
                c.y = fminf(fmaxf(a.y, p.lo[1]), p.hi[1]);
                c.z = fminf(fmaxf(a.z, p.lo[2]), p.hi[2]);
                c.w = fminf(fmaxf(a.w, p.lo[3]), p.hi[3]);
                reinterpret_cast<float4*>(p.actions_clipped)[e] = c;
            }
            p.values[e] = sOut[tid * 8 + 4];
            p.logp[e] = lp;
        }
        __syncthreads();
    }
