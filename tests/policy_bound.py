"""TEST INFRASTRUCTURE ONLY -- a propagated forward-error bound for the policy kernels, and NumPy emulations of their operand
arithmetic (the emulations exist to test the bound: tests/test_policy_bound_cpu.py).

`forward_with_bound(sd, obs, impl, norm)` returns the float64 forward of SB3's MlpPolicy (oracle/sb3_oracle.mlp_policy_forward,
with the kernel's own clip / clamp of the input applied) and a per-element bound on |kernel - oracle| for mean[n,4] and value[n].
The bound is a first-order forward error analysis carried layer by layer in float64.  For layer l with weights W, bias b, exact
input x, input error e and padded input count K:

    |dz| <= |W| e + (u_op + n_acc u_acc) (|W| (|x| + e) + |b|) + f (sum_k |W[:,k]| + sum_k (|x_k| + e_k) + 1)
    e_l   = min(2, L |dz|) + eps_tanh,       L = max sech^2 on [z - |dz|, z + |dz|]

and the float32 FFMA heads add (H3 + 2) 2^-24 (|w_h| (|h| + e) + |b_h|) to |w_h| e.  e_0 is the error of the normalised input.

Constants (derived from the code in csrc/; u_* relative, f absolute, in the unscaled domain):

fp32 (qs_policy.cu, policy_forward_ffma_kernel)
    u_op = f = 0: the operands are the float32 weights and activations themselves.
    u_acc = 2^-24, n_acc = K: acc starts at the bias and takes K round-to-nearest fmaf.
    eps_tanh = 2^-20: fast_tanh = 1 - __fdividef(2, __expf(2z) + 1).  A relative error d of t = __expf(2z) moves 2/(t+1) by
        2t/(t+1)^2 d; the CUDA guide's __expf bound (2 + 1.173 |2z|) ulp times 2t/(t+1)^2 peaks below 2 ulp = 2^-22 (near
        |z| = 0.5); t + 1 rounds (<= 2 * 2^-24 on 2/(t+1) <= 2), __fdividef is 2 ulp (<= 2^-21 on a quotient <= 2), 1 - q rounds
        (2^-24): 2^-22 + 2^-23 + 2^-21 + 2^-24 < 2^-20.
    e_0 = 2^-23 |v|: (x - mean) * istd in float64 (three float64 roundings), one rounding to float32 (2^-24), doubled.

tensor (the warp-specialised pipeline, qs_rollout_impl.cuh; weights staged by qs_tc.cuh::stage_weights, activations and inputs
split by split_h2_rn)
    Weights are scaled by sc = fl32(2 log2 e) (2^-24) and rounded to float32 (2^-24); hi = the scaled weight truncated to 10
    mantissa bits (remainder < 2^-10 |w|), lo = f16_rn(remainder) (2^-11 of the remainder: 2^-21 |w|).  Activations: hi =
    f16_rn(x), lo = f16_rn(x - hi) (x - hi is exact): 2^-11 * 2^-11 |x| = 2^-22 |x|.  The dropped lo*lo product is at most
    2^-10 |w| * 2^-11 |x| = 2^-21 |w x|.  Sum: u_op = 2^-21 + 2^-22 + 2^-21 + 2 * 2^-24 < 3 * 2^-21.
    f = 2^-25: below 2^-14 float16 is subnormal with spacing 2^-24, so hi (weights only: the truncated value is re-rounded) and lo
    carry an absolute error of 2^-25 each in the scaled domain.  Per product that is <= 2 * 2^-25 |x| / sc < 2^-25 |x| for a
    weight and 2^-25 sc |w| / sc = 2^-25 |w| for an activation; the bias row multiplies the exact constant 1.
    u_acc = 2^-23: tcgen05 kind::f16 accumulates in float32 with a rounding mode NVIDIA does not document; 2^-23 assumes
    truncation.  n_acc = K (the padded K including the bias row: 32, 144, 80), one rounding per accumulated product.
    eps_tanh = 2^-20: tanh4_from_exponents.  ex2.approx.ftz (taken as 2^-22 relative) enters 2/a with the factor 2t/(t+1)^2 <=
    1/2 (2^-23); the saturating FFMA (2^-24 on a_i), the three products of the a's (3 * 2^-24), rcp.approx.ftz (2^-23, PTX: 1 ulp)
    and r * q (2^-24) are relative errors of 2/a <= 2: 2 * (6 * 2^-24 + 2^-23); the final FFMA rounds to 2^-24.  The other three
    a's cancel exactly (the same registers sit in numerator and denominator).  Total 2^-23 + 2^-21 + 2^-22 + 2^-24 < 2^-20.
    e_0 = 2^-22 |v| + 2^-23 istd |mean - fl32(mean)|: stage_x computes fl(fl(fl(x - m_hi) - m_lo) * fl32(istd)): two subtraction
    roundings (2^-24 each, on values within |v| / istd + |m_lo|), the multiply and the rounded istd (2^-24 each on |v|).  The
    +-norm_clip clip is 1-Lipschitz, so the error is taken at min(|v|, 2 norm_clip).  The +-60000 float16-range clamp of the
    layer-1 operand is part of the operation: the oracle applies it too.

tensor_fast (the three-chain kernel, qs_policy_tc.cu with PRECISE = false)
    u_op = 2^-9 + 2^-20: weights and activations are single float16 truncated to 10 mantissa bits (qs_tc.cuh::split_h2, hi
    only): 2^-10 each, and their product.  (2^-11 would hold for round-to-nearest; the kernel truncates.)
    f = 2^-25 as for tensor (no scaling: 2^-25 |x| + 2^-25 |w|).  u_acc = 2^-23, n_acc = K as for tensor.
    eps_tanh = 2^-10: tanh.approx.f32 (PTX: maximum relative error 2^-10.987, |tanh| <= 1).
    e_0 as for tensor (the same stage_obs_row arithmetic).

Out of scope: weights whose scaled value overflows float16 (|w| > 65504 / (2 log2 e) ~ 22,700).
"""
from __future__ import annotations

import numpy as np

H1, H2, H3, NACT = 128, 64, 64, 4
SC = float(np.float32(2.0 * np.log2(np.e)))          # the float32 scale the tensor kernels multiply weights by
F16_RANGE = 60000.0

CONST = {
    "fp32": dict(u_op=0.0, f=0.0, u_acc=2.0 ** -24, eps_tanh=2.0 ** -20, e0_rel=2.0 ** -23, e0_lo=0.0, clamp=False),
    "tensor": dict(u_op=3 * 2.0 ** -21, f=2.0 ** -25, u_acc=2.0 ** -23, eps_tanh=2.0 ** -20, e0_rel=2.0 ** -22, e0_lo=2.0 ** -23, clamp=True),
    "tensor_fast": dict(u_op=2.0 ** -9 + 2.0 ** -20, f=2.0 ** -25, u_acc=2.0 ** -23, eps_tanh=2.0 ** -10, e0_rel=2.0 ** -22, e0_lo=2.0 ** -23,
                        clamp=True),
}
HEAD_U = (H3 + 2) * 2.0 ** -24                        # 64 float32 FFMA per head output, + the partial-sum add and the bias


def padded_k(obs_dim: int) -> tuple:
    """K of each layer as the tensor kernels issue it: inputs + the bias row, padded to 16 (layer 1 to 32)."""
    return (32, H1 + 16, H2 + 16), (obs_dim, H1, H2)


def layers(sd, net):
    g = lambda k: np.asarray(sd[k], np.float64)
    return [(g(f"mlp_extractor.{net}.{i}.weight"), g(f"mlp_extractor.{net}.{i}.bias")) for i in (0, 2, 4)]


def heads(sd):
    g = lambda k: np.asarray(sd[k], np.float64)
    return (g("action_net.weight"), g("action_net.bias")), (g("value_net.weight"), g("value_net.bias"))


def normalised_input(obs, impl, norm=None, eps=1e-8, clip=10.0):
    """The exact input the kernel approximates and the bound e_0 on its error.  norm: float64 (count, mean[d], var[d])."""
    c = CONST[impl]
    x = np.asarray(obs, np.float64)
    if norm is None:
        v, e0 = x, np.zeros_like(x)
    else:
        norm = np.asarray(norm, np.float64)
        d = x.shape[1]
        mean, var = norm[1:1 + d], norm[1 + d:1 + 2 * d]
        istd = 1.0 / np.sqrt(var + np.float64(np.float32(eps)))
        u = (x - mean) * istd
        m_lo = np.abs(mean - mean.astype(np.float32).astype(np.float64))
        e0 = c["e0_rel"] * np.minimum(np.abs(u), 2 * clip) + c["e0_lo"] * istd * m_lo
        v = np.clip(u, -np.float64(np.float32(clip)), np.float64(np.float32(clip)))
    if c["clamp"]:
        v = np.clip(v, -F16_RANGE, F16_RANGE)
    return v, e0


def _net_bound(Ls, head, x, e, c, ks):
    for (W, b), K in zip(Ls, ks):
        aW = np.abs(W)
        ax = np.abs(x) + e
        z = x @ W.T + b
        dz = (e @ aW.T + (c["u_op"] + K * c["u_acc"]) * (ax @ aW.T + np.abs(b))
              + c["f"] * (aW.sum(1)[None, :] + ax.sum(1, keepdims=True) + 1.0))
        t = np.minimum(np.maximum(np.abs(z) - dz, 0.0), 300.0)
        L = 1.0 / np.cosh(t) ** 2
        x, e = np.tanh(z), np.minimum(2.0, L * dz) + c["eps_tanh"]
    Wh, bh = head
    out = x @ Wh.T + bh
    aWh = np.abs(Wh)
    return out, e @ aWh.T + HEAD_U * ((np.abs(x) + e) @ aWh.T + np.abs(bh))


def forward_with_bound(sd, obs, impl, norm=None, eps=1e-8, clip=10.0, e0=None):
    """(mean[n,4], value[n], bound_mean[n,4], bound_value[n]) in float64.  `obs`: the raw float32 rows the kernel reads (or,
    with e0 given, rows whose error bound is e0: e.g. the kernel's own normalised rows with e0 = 0)."""
    c = CONST["tensor" if impl == "auto" else impl]
    x, e = normalised_input(obs, "tensor" if impl == "auto" else impl, norm, eps, clip)
    if e0 is not None:
        e = np.broadcast_to(np.asarray(e0, np.float64), x.shape)
    kp, kk = padded_k(x.shape[1])
    ks = kk if c is CONST["fp32"] else kp
    a_head, v_head = heads(sd)
    mean, bm = _net_bound(layers(sd, "policy_net"), a_head, x, e, c, ks)
    val, bv = _net_bound(layers(sd, "value_net"), v_head, x, e, c, ks)
    return mean, val[:, 0], bm, bv[:, 0]


def oracle_outputs(sd, mean, noise):
    """actions and log-prob from a mean as SB3 computes them (DiagGaussianDistribution), float64."""
    ls = np.asarray(sd["log_std"], np.float64)
    eps = np.zeros_like(mean) if noise is None else np.asarray(noise, np.float64)
    return mean + np.exp(ls) * eps, np.sum(-0.5 * eps ** 2 - ls - 0.5 * np.log(2 * np.pi), axis=1)


def max_ratio(got_mean, got_value, mean, value, bm, bv):
    """max over the batch of |got - oracle| / bound, for mean and value."""
    rm = np.abs(np.asarray(got_mean, np.float64) - mean) / bm
    rv = np.abs(np.asarray(got_value, np.float64) - value) / bv
    return float(rm.max()), float(rv.max())


# ---- NumPy emulations of the operand arithmetic ------------------------------------------------------------------------------
f32 = lambda a: np.asarray(a, np.float64).astype(np.float32).astype(np.float64)
f16 = lambda a: np.asarray(a, np.float64).astype(np.float32).astype(np.float16).astype(np.float64)


def trunc10(a):
    """float32 -> float16 value with the mantissa truncated to 10 bits (qs_tc.cuh::split_h2's hi, LOP3 then cvt.rn)."""
    u = np.asarray(a, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)
    return u.view(np.float32).astype(np.float16).astype(np.float64)


def split_rn(a):
    a = f32(a)
    hi = f16(a)
    return hi, f16(a - hi)


def split_trunc(a):
    a = f32(a)
    hi = trunc10(a)
    return hi, f16(a - hi)


def _norm_f32(obs, norm, eps, clip, mean_lo=True):
    """stage_obs_row / stage_x: ((x - m_hi) - m_lo) * istd in float32 (mean_lo=False: a float32 mean, the planted defect)."""
    x = f32(obs)
    d = x.shape[1]
    mean, var = norm[1:1 + d], norm[1 + d:1 + 2 * d]
    m_hi = f32(mean)
    m_lo = f32(mean - m_hi) if mean_lo else 0.0 * m_hi
    istd = f32(1.0 / np.sqrt(var + np.float64(np.float32(eps))))
    v = f32(f32(f32(x - m_hi) - m_lo) * istd)
    return np.clip(v, -np.float32(clip), np.float32(clip))


def emulate(sd, obs, impl, norm=None, eps=1e-8, clip=10.0, defect=None):
    """Forward with the kernel's operand arithmetic (float64 accumulation: the accumulation error is not emulated).
    impl: "fp32" (float32 throughout), "tensor" (split float16, round-to-nearest activations, truncated weights, scaled by sc),
    "tensor_fast" (single truncated float16).  defect (tensor only): "lo_dropped" (single round-to-nearest float16 operands),
    "bias_row" (layer 2's bias row staged one row early, over the last weight row), "w2_halves" (the two 64-column halves of W2
    swapped), "head_split" (the second partial head sum lost), "mean_f32" (normalisation with a float32 mean).
    Returns (mean[n,4], value[n])."""
    if impl == "fp32":
        x = f32(obs) if norm is None else f32(np.clip((np.asarray(obs, np.float64) - norm[1:1 + obs.shape[1]])
                                                         / np.sqrt(norm[1 + obs.shape[1]:] + np.float64(np.float32(eps))), -clip, clip))
        x = x.astype(np.float32)

        def net(Ls, head):
            h = x
            for W, b in Ls:
                z = h @ W.T.astype(np.float32) + b.astype(np.float32)
                with np.errstate(over="ignore"):
                    t = np.exp(np.float32(2.0) * z)
                h = (np.float32(1.0) - np.float32(2.0) / (t + np.float32(1.0))).astype(np.float32)
            Wh, bh = head
            return (h @ Wh.T.astype(np.float32) + bh.astype(np.float32)).astype(np.float64)
    else:
        x = f32(obs) if norm is None else _norm_f32(obs, norm, eps, clip, mean_lo=defect != "mean_f32")
        x = np.clip(x, -F16_RANGE, F16_RANGE)
        fast = impl == "tensor_fast"
        sc = 1.0 if fast else SC

        def split_x(a):
            if fast:
                return trunc10(f32(a)), 0.0
            hi, lo = split_rn(a)
            return (hi, 0.0) if defect == "lo_dropped" else (hi, lo)

        def split_w(a):
            if fast:
                return trunc10(f32(a)), 0.0
            if defect == "lo_dropped":
                return f16(a), 0.0
            return split_trunc(a)

        def act(u):
            return f32(np.tanh(u)) if fast else f32(1.0 - 2.0 / (np.exp2(np.minimum(u, 1000.0)) + 1.0))

        def net(Ls, head):
            h = x
            for li, (W, b) in enumerate(Ls):
                W, b = W.copy(), b.copy()
                if li == 1 and defect == "w2_halves":
                    W = np.concatenate([W[:, 64:], W[:, :64]], axis=1)
                xs = np.concatenate([h, np.ones((h.shape[0], 1))], axis=1)
                Wb = np.concatenate([W, b[:, None]], axis=1)
                if li == 1 and defect == "bias_row":
                    Wb[:, -2], Wb[:, -1] = Wb[:, -1], 0.0
                wh, wl = split_w(f32(sc * f32(Wb)))
                xh, xl = split_x(xs)
                u = xh @ wh.T + xh @ (wl.T if np.ndim(wl) else 0.0 * wh.T) + (xl @ wh.T if np.ndim(xl) else 0.0)
                h = act(u)
            Wh, bh = head
            if defect == "head_split":
                return f32(h[:, :32] @ f32(Wh[:, :32]).T + f32(bh))
            return f32(h @ f32(Wh).T + f32(bh))
    a_head, v_head = heads(sd)
    return net(layers(sd, "policy_net"), a_head), net(layers(sd, "value_net"), v_head)[:, 0]


# ---- weight sets and inputs, generated from seeds -----------------------------------------------------------------------------
def _shipped(golden_dir, tag):
    z = np.load(f"{golden_dir}/policy_{tag}.npz")
    return {k[2:]: z[k].astype(np.float32) for k in z.files if k.startswith("w.")}


def weight_sets(golden_dir, obs_dim):
    """name -> SB3 state_dict (float32) for `obs_dim` (17 or 20): the sets of the policy-bound tests."""
    from rl_aerial_manipulator_b200.ppo import init_state_dict
    ship = _shipped(golden_dir, "v2" if obs_dim == 20 else "v1")
    rng = np.random.default_rng(obs_dim)
    out = {"shipped": ship}
    for s in (0, 1):
        out[f"init_seed{s}"] = init_state_dict(obs_dim, s)
    out["init_perturbed"] = {k: (np.asarray(v, np.float32) + 0.05 * rng.standard_normal(np.shape(v))).astype(np.float32)
                             for k, v in init_state_dict(obs_dim, 2).items()}
    tl = {}
    for k, v in ship.items():                                    # "trained-like": rescaled shipped layers plus noise
        tl[k] = (v * rng.uniform(0.5, 2.0) + 0.02 * rng.standard_normal(v.shape)).astype(np.float32)
    vh = tl["value_net.weight"]
    tl["value_net.weight"] = (vh * (100.0 / np.abs(vh).max())).astype(np.float32)
    tl["log_std"] = rng.uniform(-3.0, 1.0, NACT).astype(np.float32)
    out["trained_like"] = tl
    wr = {}
    for k, v in ship.items():                                    # wide range: |w| = 10^U(-8, 0.5), exact zeros, an all-zero column
        w = (np.sign(rng.standard_normal(v.shape)) * 10.0 ** rng.uniform(-8.0, 0.5, v.shape)).astype(np.float32)
        w[rng.random(v.shape) < 0.05] = 0.0
        if w.ndim == 2 and k.startswith("mlp_extractor"):
            w[:, 3] = 0.0
        wr[k] = w
    wr["log_std"] = ship["log_std"].copy()
    out["wide_range"] = wr
    sat = {k: v.copy() for k, v in ship.items()}                 # saturating: layer-1 biases +-20
    for net in ("policy_net", "value_net"):
        k = f"mlp_extractor.{net}.0.bias"
        sat[k] = (20.0 * np.sign(rng.standard_normal(sat[k].shape))).astype(np.float32)
    out["saturating"] = sat
    out["near_zero"] = {k: (v * np.float32(1e-3) if k != "log_std" else v) for k, v in ship.items()}   # 1 - 2/(2^u + 1) cancels
    return out


def input_sets(obs_dim, rows=512, seed=0):
    """name -> (raw float32 obs[rows, obs_dim], float64 VecNormalize stats (count, mean, var) or None)."""
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((rows, obs_dim))
    out = {f"randn_x{s:g}": ((base * s).astype(np.float32), None) for s in (1e-3, 0.7, 3.0, 30.0)}
    # VecNormalize statistics with a near-constant column (quaternion w: mean 1 - 3e-5) and a zero-variance column (normalised by
    # sqrt(eps) alone), both with a mean 0.45 float32 ulp off a float32 value; a quarter of the rows land exactly on +-norm_clip
    mean = rng.uniform(-2, 2, obs_dim)
    var = rng.uniform(0.2, 4.0, obs_dim)
    mean[6], var[6] = float(np.float32(1.0 - 3.1e-5)) + 0.45 * 2.0 ** -24, (1e-4) ** 2 / 12
    mean[7], var[7] = float(np.float32(123.456)) + 0.45 * 2.0 ** -17, 0.0
    stats = np.concatenate([[1e6], mean, var])
    x = mean + base * np.sqrt(var) * 2.0
    x[:, 6] = 1.0 - 1e-4 * rng.random(rows)
    x[:, 7] = np.float32(mean[7])
    k = rows // 4
    istd = 1.0 / np.sqrt(var + np.float64(np.float32(1e-8)))
    x[:k, 0] = mean[0] + 10.0 / istd[0] * np.sign(base[:k, 0])
    x = x.astype(np.float32)
    out["vecnorm"] = (x, stats)
    big = (np.sign(base) * 59999.0).astype(np.float32)
    big[rows // 2:] = (np.sign(base[rows // 2:]) * 1e5).astype(np.float32)
    out["clamp_pm60000"] = (big, None)
    return out
