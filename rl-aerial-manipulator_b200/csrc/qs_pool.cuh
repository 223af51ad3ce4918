// qs_pool.cuh -- HBM layout of the hidden env state ("state pool") and its register pack/unpack.
//
// Layout: tile-major array of struct-of-arrays tiles.  A tile is the record of one warp's 32 envs: the per-env record is SLOTS
// scalars of the kernel's arithmetic type (the two 32-bit bookkeeping words are bit-cast into the last slot(s)); slot group v
// (4 floats / 2 doubles) of the tile is a 512-byte plane (lane * 16), left-over slots (SLOTS % vector width) follow as scalar
// planes (lane * sizeof(Real)):
//     tile t of the pool at  base + t * TILE_BYTES,   plane v at + v * 512,   tail plane k at + NVEC * 512 + k * 32 * sizeof(Real)
// so a warp reads and writes ONE contiguous, 128-byte aligned block per step (2688 B for v2/f32) with LDG.128/STG.128 that are
// 512 contiguous bytes each -- every DRAM page the tile touches is used completely, where n-major planes ((v * n + e) * 16)
// made each tile six separate 512-byte streams.  The pool is allocated for whole tiles; envs past n in the last tile are padding.
//
//   v2 f32: 13 state + 3 waypoint + final_yaw + last_distance + ep_return + 2 words = 21 slots = 84 B/env
//   v2 f64: 19 doubles + 1 packed word pair                                         = 20 slots = 160 B/env
//   v1 f32: 13 + 6 + 3 (final_yaw unused, kept for a uniform layout) + 2            = 24 slots = 96 B/env
//   v1 f64:                                                                           23 slots = 184 B/env
#pragma once
#include "qs_env.cuh"
#include <string.h>

namespace qs {

template <typename Real> struct VecOf;
template <> struct VecOf<float> { using type = float4; static constexpr int W = 4; };
template <> struct VecOf<double> { using type = double2; static constexpr int W = 2; };

template <typename Real, int VER>
struct PoolLayout {
    static constexpr int NWP = EnvTraits<VER>::NWP;
    static constexpr int NREAL = 13 + 3 * NWP + 3;
    static constexpr int SLOTS = NREAL + (sizeof(Real) == 4 ? 2 : 1);
    static constexpr int W = VecOf<Real>::W;
    static constexpr int NVEC = SLOTS / W;
    static constexpr int NTAIL = SLOTS % W;
    static constexpr int BYTES = SLOTS * (int)sizeof(Real);
    static constexpr int TILE_BYTES = 32 * BYTES;                     // NVEC * 512 + NTAIL * 32 * sizeof(Real)
    static constexpr int TAIL_OFF = NVEC * 512;
};

#if defined(__CUDACC__)
__device__ __forceinline__ float u32_as_real(uint32_t a, float) { return __uint_as_float(a); }
__device__ __forceinline__ uint32_t real_as_u32(float v) { return __float_as_uint(v); }

template <typename Real, int VER>
__device__ __forceinline__ void pool_unpack(const Real* slot, EnvState<Real, VER>& s);

template <typename Real, int VER>
__device__ __forceinline__ void pool_load(const void* __restrict__ base, int64_t n, int64_t e, EnvState<Real, VER>& s) {
    using L = PoolLayout<Real, VER>;
    using V = typename VecOf<Real>::type;
    Real slot[L::NVEC * L::W + (L::NTAIL ? L::NTAIL : 1)];
    (void)n;
    const unsigned char* tb0 = reinterpret_cast<const unsigned char*>(base) + (e >> 5) * (int64_t)L::TILE_BYTES;
    const int ln = (int)(e & 31);
    const V* vb = reinterpret_cast<const V*>(tb0) + ln;
#pragma unroll
    for (int v = 0; v < L::NVEC; ++v) {
        const V x = __ldg(vb + v * 32);
        if (L::W == 4) {
            const float4 f = *reinterpret_cast<const float4*>(&x);
            slot[4 * v + 0] = (Real)f.x; slot[4 * v + 1] = (Real)f.y; slot[4 * v + 2] = (Real)f.z; slot[4 * v + 3] = (Real)f.w;
        } else {
            const double2 f = *reinterpret_cast<const double2*>(&x);
            slot[2 * v + 0] = (Real)f.x; slot[2 * v + 1] = (Real)f.y;
        }
    }
    const Real* tb = reinterpret_cast<const Real*>(tb0 + L::TAIL_OFF) + ln;
#pragma unroll
    for (int t = 0; t < L::NTAIL; ++t) slot[L::NVEC * L::W + t] = __ldg(tb + t * 32);
    pool_unpack<Real, VER>(slot, s);
}

template <typename Real, int VER>
__device__ __forceinline__ void pool_unpack(const Real* slot, EnvState<Real, VER>& s) {
    using L = PoolLayout<Real, VER>;
    int k = 0;
#pragma unroll
    for (int i = 0; i < 13; ++i) s.y[i] = slot[k++];
#pragma unroll
    for (int j = 0; j < L::NWP; ++j) { s.wp[j][0] = slot[k++]; s.wp[j][1] = slot[k++]; s.wp[j][2] = slot[k++]; }
    s.final_yaw = slot[k++];
    s.last_d = slot[k++];
    s.ep_ret = slot[k++];
    if (sizeof(Real) == 4) {
        s.bits = __float_as_uint((float)slot[k]);
        s.episode = __float_as_uint((float)slot[k + 1]);
    } else {
        const long long w = __double_as_longlong((double)slot[k]);
        s.bits = (uint32_t)((unsigned long long)w & 0xFFFFFFFFull);
        s.episode = (uint32_t)((unsigned long long)w >> 32);
    }
}

template <typename Real, int VER>
__device__ __forceinline__ void pool_store(void* __restrict__ base, int64_t n, int64_t e, const EnvState<Real, VER>& s) {
    using L = PoolLayout<Real, VER>;
    using V = typename VecOf<Real>::type;
    Real slot[L::NVEC * L::W + (L::NTAIL ? L::NTAIL : 1)];
    int k = 0;
#pragma unroll
    for (int i = 0; i < 13; ++i) slot[k++] = s.y[i];
#pragma unroll
    for (int j = 0; j < L::NWP; ++j) { slot[k++] = s.wp[j][0]; slot[k++] = s.wp[j][1]; slot[k++] = s.wp[j][2]; }
    slot[k++] = s.final_yaw;
    slot[k++] = s.last_d;
    slot[k++] = s.ep_ret;
    if (sizeof(Real) == 4) {
        slot[k] = (Real)__uint_as_float(s.bits);
        slot[k + 1] = (Real)__uint_as_float(s.episode);
    } else {
        slot[k] = (Real)__longlong_as_double((long long)(((unsigned long long)s.episode << 32) | (unsigned long long)s.bits));
    }
    (void)n;
    unsigned char* tb0 = reinterpret_cast<unsigned char*>(base) + (e >> 5) * (int64_t)L::TILE_BYTES;
    const int ln = (int)(e & 31);
    V* vb = reinterpret_cast<V*>(tb0) + ln;
#pragma unroll
    for (int v = 0; v < L::NVEC; ++v) {
        V x;
        if (L::W == 4) {
            float4 f = make_float4((float)slot[4 * v], (float)slot[4 * v + 1], (float)slot[4 * v + 2], (float)slot[4 * v + 3]);
            x = *reinterpret_cast<V*>(&f);
        } else {
            double2 f = make_double2((double)slot[2 * v], (double)slot[2 * v + 1]);
            x = *reinterpret_cast<V*>(&f);
        }
        vb[v * 32] = x;
    }
    Real* tb = reinterpret_cast<Real*>(tb0 + L::TAIL_OFF) + ln;
#pragma unroll
    for (int t = 0; t < L::NTAIL; ++t) tb[t * 32] = slot[L::NVEC * L::W + t];
}
#endif  // __CUDACC__

}  // namespace qs
