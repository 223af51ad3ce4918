// qs_tc.cuh -- tcgen05 / TMEM / mbarrier helpers and the MlpPolicy operand layouts shared by the policy-forward kernel
// (qs_policy_tc.cu) and the fused rollout kernel (qs_rollout.cu).  sm_100a only.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace qs {
namespace tc {

constexpr int ROWS = 128;
constexpr int K1 = 32;
constexpr int N1 = 128, N2 = 64, N3 = 64, NACT = 4;
// B operands carry the bias as one extra input: layer 1 uses the spare padding column k = OBS of X (set to 1.0); layers 2/3
// get one extra k-step of 16 whose A operand is a constant TMEM chunk (1, 0, ..., 0) -- the epilogue adds no bias.
constexpr int KB = 16;
constexpr int W1_BYTES = (K1 / 8) * N1 * 16, W2_BYTES = ((N1 + KB) / 8) * N2 * 16, W3_BYTES = ((N2 + KB) / 8) * N3 * 16;
constexpr int W_SET = 2 * (W1_BYTES + W2_BYTES + W3_BYTES);          // both nets, one precision part: 65536
constexpr int OFF_W1 = 0, OFF_W2 = 2 * W1_BYTES, OFF_W3 = OFF_W2 + 2 * W2_BYTES;
constexpr int C_B1 = 0, C_B2 = C_B1 + 2 * N1, C_B3 = C_B2 + 2 * N2, C_WH = C_B3 + 2 * N3, C_BH = C_WH + 2 * N3 * NACT,
              C_LS = C_BH + 2 * NACT, C_TOTAL = C_LS + NACT;
constexpr int TMEM_COLS = 512;

struct Blob {
    int obs;
    __host__ __device__ int per_net() const { return obs * N1 + N1 + N1 * N2 + N2 + N2 * N3 + N3 + N3 * NACT + NACT; }
    __host__ __device__ int w1(int net) const { return net * per_net(); }
    __host__ __device__ int b1(int net) const { return w1(net) + obs * N1; }
    __host__ __device__ int w2(int net) const { return b1(net) + N1; }
    __host__ __device__ int b2(int net) const { return w2(net) + N1 * N2; }
    __host__ __device__ int w3(int net) const { return b2(net) + N2; }
    __host__ __device__ int b3(int net) const { return w3(net) + N2 * N3; }
    __host__ __device__ int wh(int net) const { return b3(net) + N3; }
    __host__ __device__ int bh(int net) const { return wh(net) + N3 * NACT; }
    __host__ __device__ int log_std() const { return 2 * per_net(); }
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
__host__ __device__ constexpr uint32_t make_idesc(int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(ROWS >> 4) << 24);
}
// D[tmem] (+)= A[tmem] . B[smem]^T
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// One lane of a converged warp.  The MMA issue runs under a warp-uniform branch + this election so that descriptors and TMEM
// addresses stay in uniform registers: issued from a divergent `if (thread == 0)`, every UTCHMMA costs an ELECT/R2UR waterfall
// loop (~100 cycles per MMA measured, 8.7k of the 23k cycles a tile took).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
// the loaded registers are valid only after this; tying them to the asm keeps the compiler from hoisting their uses above it
__device__ __forceinline__ void tmem_ld_wait32(uint32_t* v) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]),
                   "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]),
                   "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]),
                   "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
        "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float tanh_mufu(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// Four tanh on one MUFU.RCP.  u_i = 2*log2(e)*x_i (the scale lives in the weights): tanh(x) = 1 - 2/a with a = 2^u + 1, and
// 1/a = (b*c*d) / (a*b*c*d): 5 MUFU per 4 elements instead of 8; the extra FMULs run on the FMA pipe, which the epilogue leaves
// idle.  Error: ~3 ulp of 1/a <= 2e-7 absolute.
// The clamp, the +1 and a power-of-two scale are ONE instruction (r02): a_i' = sat(2^u_i * s + s) = min(2^u_i + 1, 2^31) * s
// with s = 2^-31 (FFMA.SAT; exact scaling, the same rounding as the add), so a_i' lies in [2^-31, 1], the product of four in
// [2^-124, 1] (no overflow, no flush), and beyond 2^u + 1 = 2^31 tanh is 1.0f to the last bit anyway.  The scale comes back with
// the -2 of tanh = 1 - 2/a: 1/a_i = s / a_i'.  19 instructions per four activations instead of 23 for an explicit min and FADD.
// A NaN exponent leaves the group non-finite (sat flushes NaN to 0 -> 1/0), which the next layer's MMAs spread over the row.
__device__ __forceinline__ void tanh4_from_exponents(const uint32_t* v, float* y) {
    float a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float t;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(__uint_as_float(v[i])));
        asm("fma.rn.ftz.sat.f32 %0, %1, %2, %2;" : "=f"(a[i]) : "f"(t), "f"(4.656612873077393e-10f));     // 2^-31
    }
    const float p = a[0] * a[1], q = a[2] * a[3];
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p * q));
    r *= -9.313225746154785e-10f;            // -2 s = -2^-30
    const float rp = r * q, rq = r * p;      // -2/(a0 a1), -2/(a2 a3)
    y[0] = fmaf(rp, a[1], 1.0f);
    y[1] = fmaf(rp, a[0], 1.0f);
    y[2] = fmaf(rq, a[3], 1.0f);
    y[3] = fmaf(rq, a[2], 1.0f);
}
// Eight tanh as two groups of four.  One MUFU.RCP for all eight (each group's product lifted by 2^62 so that both fit one float)
// measured 279.3 vs 279.7 us per 1M-env launch on B200 (r02), i.e. nothing, for one more rounding on the way to 1/a.
__device__ __forceinline__ void tanh8_from_exponents(const uint32_t* v, float* y) {
    tanh4_from_exponents(v, y);
    tanh4_from_exponents(v + 4, y + 4);
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
// (a, b) -> packed hi halves and packed lo halves, a = hi_a + lo_a to ~21 bits.  hi is the float truncated to float16's
// 10 explicit mantissa bits (a LOP3, exactly representable), lo the exact remainder rounded to float16.
__device__ __forceinline__ void split_h2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const float ah = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u);
    const float bh = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
    hi = pack_h2(ah, bh);
    lo = pack_h2(a - ah, b - bh);
}

// weights [K][N] float32 (input-major blob) -> float16 hi (and lo) canonical B operands [N rows][KP], zero padded;
// input index `kbias` carries the bias (its A element is the constant 1); everything is multiplied by `scale`
template <bool PRECISE, int NT>
__device__ __forceinline__ void stage_weights(const float* __restrict__ w, const float* __restrict__ bias, int K, int kbias, int KP, int N,
                                              float scale, unsigned char* dst_hi, unsigned char* dst_lo, int tid) {
    for (int i = tid; i < (KP / 8) * N; i += NT) {
        const int c = i / N, n = i - c * N;
        uint32_t ph[4], pl[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k0 = c * 8 + 2 * j, k1 = k0 + 1;
            const float a = scale * (k0 < K ? __ldg(w + (int64_t)k0 * N + n) : (k0 == kbias ? __ldg(bias + n) : 0.f));
            const float b = scale * (k1 < K ? __ldg(w + (int64_t)k1 * N + n) : (k1 == kbias ? __ldg(bias + n) : 0.f));
            split_h2(a, b, ph[j], pl[j]);
        }
        *reinterpret_cast<uint4*>(dst_hi + (size_t)i * 16) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
        if (PRECISE) *reinterpret_cast<uint4*>(dst_lo + (size_t)i * 16) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
    }
}

// one loaded 32-column accumulator chunk of this thread's row (bias already inside) -> tanh (float32 in y)
template <bool PRECISE>
__device__ __forceinline__ void tanh32(const uint32_t* v, float* y) {
    if (PRECISE) {
#pragma unroll
        for (int i = 0; i < 32; i += 4) tanh4_from_exponents(v + i, y + i);
    } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) y[i] = tanh_mufu(__uint_as_float(v[i]));
    }
}

// y[32] -> packed float16 hi (16 columns at taddr) and, if PRECISE, lo (16 columns at taddr + 16): in place over the chunk
template <bool PRECISE>
__device__ __forceinline__ void put32(uint32_t taddr, const float* y) {
    uint32_t h[16], l[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) split_h2(y[2 * j], y[2 * j + 1], h[j], l[j]);
    tmem_st16(taddr, h);
    if (PRECISE) tmem_st16(taddr + 16, l);
}

}  // namespace tc
}  // namespace qs
