"""The PPO update kernel (csrc/qs_ppo.cu: qs_ppo_grad, qs_ppo_update, qs_ppo_apply) and QuadPPO.train() against the float64 PPO
oracle (oracle/ppo_oracle.py, itself pinned to torch autograd in tests/test_ppo.py), over what one configuration does not reach:
every hyperparameter and all eight statistics, the minibatch sizes where the 16-row tiling and the persistent grid change shape,
inputs that saturate the tanh layers and the probability ratio, gradient clipping and Adam over 50 updates, the multi-rank split
qs_ppo_grad -> average -> qs_ppo_apply, whole training passes, and the refusals of the C-ABI.

Tolerances.  The gradient bar of the existing tests, 2e-5 * max|g|, holds wherever it applied before (moderate minibatches,
unsaturated inputs).  The other bounds are a few times the worst error measured on a B200 (see each constant).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as po
from test_ppo import perturbed_state_dict, random_minibatch

pytestmark = pytest.mark.gpu

QS_EINVAL = -1

# Measured on an NVIDIA B200 (1000 W power limit); every bound is a few times the worst measured error.
GRAD_TOL = 2e-5          # |g_kernel - g_oracle| / max|g_oracle|, the bar of tests/test_ppo.py.  Worst measured 1.4e-6 over the
STAT_TOL = 2e-5          # matrix and every shape including B = 65,536 (8.3e-7); statistics (relative to max(1, |s|)) 6.3e-7.
# saturating inputs (|obs| ~ 100, ratios e^+-3, z = 4 sigma): measured 7.9e-6 (gradient), 4.7e-6 (statistics, log_std = +1)
GRAD_TOL_SATURATED = 2e-5
# 50 qs_ppo_update calls against 50 oracle updates: parameters (absolute, measured 1.8e-6), the pre-clip gradient norm of every
# step (relative, measured 2.8e-7).  Adam's m and v, relative to their largest element, here and in the split and train() tests
# (measured 7.0e-7).
PARAM_TOL_50, NORM_TOL_50, MOMENT_TOL = 1e-5, 1e-6, 5e-6
# QuadPPO.train(), 3 epochs of 5-6 minibatches: parameters (absolute, measured 1.8e-7)
PARAM_TOL_TRAIN = 1e-6


def f32(x):
    """The kernel reads its hyperparameters as float32: the oracle gets the same values (1 - float32(0.999) alone differs from
    0.001 by 1.3e-5 relative, which would show in Adam's v)."""
    return float(np.float32(x))


F32_BETAS = (f32(0.9), f32(0.999))


def dev(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def blob(d, D):
    from rl_aerial_manipulator_b200.policy import pack_params
    return pack_params({k: np.asarray(v, np.float64) for k, v in d.items()}, D)


def log_ratio(sd, D, obs, act, oldlp):
    net = po.make_torch_actor_critic({k: np.asarray(v, np.float64) for k, v in sd.items()}, D, torch.float64)
    with torch.no_grad():
        _, lp, _ = net.evaluate_actions(torch.from_numpy(np.asarray(obs, np.float64)), torch.from_numpy(np.asarray(act, np.float64)))
    return lp.numpy() - np.asarray(oldlp, np.float64)


def kernel_grad(sd, D, buffers, idx, hp):
    """qs_ppo_grad on a fresh handle: (gradient blob, statistics); the parameters must come back untouched."""
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel
    params = torch.from_numpy(blob(sd, D)).cuda()
    before = params.clone()
    opt = PpoUpdateKernel(params, D, **hp)
    g = opt.gradient(*dev(*buffers), None if idx is None else torch.from_numpy(idx).cuda()).cpu().numpy()
    stats = opt.read_stats()
    assert torch.equal(params, before), "qs_ppo_grad wrote the parameters"
    assert int(opt.adam_state()[2].item()) == 0 and not opt.adam_state()[0].any(), "qs_ppo_grad touched the Adam state"
    opt.close()
    return g, stats


def oracle_grad(sd, D, rows, hp):
    keys = ("clip_range", "ent_coef", "vf_coef", "normalize_advantage")
    stats, grads = po.minibatch_grads(sd, *rows, **{k: (f32(hp[k]) if k != "normalize_advantage" else hp[k]) for k in keys if k in hp})
    stats["grad_norm"] = float(np.sqrt(sum((v ** 2).sum() for v in grads.values())))
    stats["batch_size"] = len(rows[0])
    return blob(grads, D), stats


def check(sd, D, buffers, idx, hp, grad_tol=GRAD_TOL, stat_tol=STAT_TOL, label=""):
    """qs_ppo_grad against the oracle on the rows `idx` of `buffers` (None: all rows): every gradient, all eight statistics."""
    rows = buffers if idx is None else tuple(b[idx] for b in buffers)
    g, sk = kernel_grad(sd, D, buffers, idx, hp)
    want, so = oracle_grad(sd, D, rows, hp)
    scale = np.abs(want).max()
    err_g = np.abs(g - want).max() / scale
    errs = {k: abs(sk[k] - so[k]) / max(1.0, abs(so[k])) for k in ("loss", "policy_gradient_loss", "value_loss", "entropy_loss", "approx_kl")}
    errs["grad_norm"] = abs(sk["grad_norm"] - so["grad_norm"]) / so["grad_norm"]
    print(f"measured {label}: grad {err_g:.3g} stats {max(errs.values()):.3g} ({max(errs, key=errs.get)})")
    assert np.isfinite(g).all() and err_g < grad_tol, (err_g, scale)
    for k, e in errs.items():
        assert e < stat_tol, (k, sk[k], so[k])
    # clip_fraction counts rows; a row whose float64 ratio lies within float32 reach of 1 +- clip_range may count either way
    lr = log_ratio(sd, D, *rows[:3])
    near = int((np.abs(np.abs(np.expm1(lr)) - f32(hp["clip_range"])) < 1e-4 * np.exp(lr)).sum())
    assert abs(sk["clip_fraction"] - so["clip_fraction"]) <= (near + 0.5) / len(rows[0]), (sk["clip_fraction"], so["clip_fraction"], near)
    assert sk["batch_size"] == len(rows[0])
    return so


# ---------------------------------------------------------------------------------------------------------------------------------
# hyperparameters
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [17, 20])
@pytest.mark.parametrize("vf_coef", [0.5, 1.0])
@pytest.mark.parametrize("clip_range", [0.1, 0.3])
@pytest.mark.parametrize("ent_coef", [0.0, 0.01])
@pytest.mark.parametrize("normalize_advantage", [True, False])
def test_grad_hyperparameter_matrix(normalize_advantage, ent_coef, clip_range, vf_coef, D):
    """qs_ppo_grad over normalize_advantage x ent_coef x clip_range x vf_coef x obs_dim: 3001 rows drawn through idx from a larger
    buffer (188 tiles over the persistent grid), every gradient and statistic against the oracle."""
    rng = np.random.default_rng([D, int(vf_coef * 10), int(clip_range * 10), int(ent_coef * 100), int(normalize_advantage)])
    sd = perturbed_state_dict(D, 7)
    B, total = 3001, 5000
    buffers = random_minibatch(rng, total, D, sd)
    idx = rng.permutation(total)[:B].astype(np.int64)
    hp = dict(clip_range=clip_range, ent_coef=ent_coef, vf_coef=vf_coef, normalize_advantage=normalize_advantage)
    so = check(sd, D, buffers, idx, hp, label=f"matrix {normalize_advantage} {ent_coef} {clip_range} {vf_coef} {D}")
    assert 0.05 < so["clip_fraction"] < 0.95                 # both branches of the clipped surrogate carry rows


# ---------------------------------------------------------------------------------------------------------------------------------
# minibatch shapes
# ---------------------------------------------------------------------------------------------------------------------------------
def _rows(spec):
    """B for a spec: an int, or 16*G +- k with G the SM count (= the kernel's grid limit) read from the device."""
    if isinstance(spec, int):
        return spec
    G = torch.cuda.get_device_properties(0).multi_processor_count
    return {"16G-1": 16 * G - 1, "16G": 16 * G, "16G+1": 16 * G + 1}[spec]


@pytest.mark.parametrize("gather", ["rows", "idx"])
@pytest.mark.parametrize("spec", [1, 2, 15, 16, 17, 33, "16G-1", "16G", "16G+1", 65536])
def test_grad_minibatch_shapes(spec, gather):
    """One row (no advantage normalisation, as SB3's len == 1 rule), partial / exact / one-more tiles, exactly one tile per CTA of
    the grid and one tile more, and the production batch_size 65,536 (~28 tiles of register-resident gradient per CTA); rows 0..B-1
    without an index list, and rows gathered through a permutation of a buffer twice as large."""
    B = _rows(spec)
    D = 20
    rng = np.random.default_rng(B)
    sd = perturbed_state_dict(D, 12)
    if gather == "rows":
        buffers, idx = random_minibatch(rng, B, D, sd), None
    else:
        total = 2 * B + 7
        buffers = random_minibatch(rng, total, D, sd)
        idx = rng.permutation(total)[:B].astype(np.int64)
    hp = dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, normalize_advantage=True)
    check(sd, D, buffers, idx, hp, label=f"shape {B} {gather}")


@pytest.mark.parametrize("normalize_advantage", [True, False])
def test_grad_constant_advantages(normalize_advantage):
    """128 rows with one advantage value: std 0, (A - mean) / (0 + 1e-8) = 0 when normalising, so only the value and entropy terms
    carry gradient (the action head's gradient must vanish)."""
    D, B = 20, 128
    rng = np.random.default_rng(5)
    sd = perturbed_state_dict(D, 13)
    obs, act, oldlp, adv, ret = random_minibatch(rng, B, D, sd)
    adv = np.full(B, 1.7, np.float32)
    hp = dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, normalize_advantage=normalize_advantage)
    so = check(sd, D, (obs, act, oldlp, adv, ret), None, hp, label=f"constant adv {normalize_advantage}")
    if normalize_advantage:
        assert so["policy_gradient_loss"] == 0.0
        g, sk = kernel_grad(sd, D, (obs, act, oldlp, adv, ret), None, hp)
        from rl_aerial_manipulator_b200.policy import unpack_params
        assert not unpack_params(g, D)["action_net.weight"].any() and sk["policy_gradient_loss"] == 0.0


# ---------------------------------------------------------------------------------------------------------------------------------
# saturating inputs
# ---------------------------------------------------------------------------------------------------------------------------------
SATURATION = ["obs_x100", "old_logp_plus_3", "old_logp_minus_3", "zero_advantage_rows", "log_std_minus_2", "log_std_plus_1"]


@pytest.mark.parametrize("case", SATURATION)
def test_grad_saturating_inputs(case):
    """Unnormalised observations of magnitude ~100 (1 - h^2 -> 0 in every tanh layer), old log-probabilities shifted by +-3 (ratios
    e^-+3: more than 90 % of the rows clipped), half the rows with A = 0 (no advantage normalisation), and log_std at -2 / +1 with
    every action 4 sigma from the mean."""
    D, B = 20, 2000
    rng = np.random.default_rng(SATURATION.index(case))
    sd = perturbed_state_dict(D, 14)
    normalize = True
    obs = rng.standard_normal((B, D)).astype(np.float32)
    act = (rng.standard_normal((B, 4)) * 1.5).astype(np.float32)
    adv = (rng.standard_normal(B) * 3 + 1).astype(np.float32)
    ret = (rng.standard_normal(B) * 10).astype(np.float32)
    shift = 0.0
    if case == "obs_x100":
        obs *= 100
    elif case.startswith("old_logp"):
        shift = 3.0 if case.endswith("plus_3") else -3.0
    elif case == "zero_advantage_rows":
        adv[rng.random(B) < 0.5] = 0.0
        normalize = False
    else:
        sd["log_std"][:] = -2.0 if case.endswith("minus_2") else 1.0
        net = po.make_torch_actor_critic({k: v.astype(np.float64) for k, v in sd.items()}, D, torch.float64)
        with torch.no_grad():
            mean = net.action_net(net.mlp_extractor["policy_net"](torch.from_numpy(obs).double())).numpy()
        act = (mean + 4.0 * np.exp(sd["log_std"].astype(np.float64)) * rng.choice([-1.0, 1.0], (B, 4))).astype(np.float32)
    lr0 = log_ratio(sd, D, obs, act, np.zeros(B))
    oldlp = (lr0 + shift + 0.3 * rng.standard_normal(B)).astype(np.float32)
    hp = dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, normalize_advantage=normalize)
    so = check(sd, D, (obs, act, oldlp, adv, ret), None, hp, grad_tol=GRAD_TOL_SATURATED, stat_tol=GRAD_TOL_SATURATED,
               label=f"saturation {case}")
    if case.startswith("old_logp"):
        assert so["clip_fraction"] > 0.9
    if case == "obs_x100":
        h = np.tanh(obs.astype(np.float64) @ sd["mlp_extractor.policy_net.0.weight"].T.astype(np.float64))
        assert np.mean(1.0 - h ** 2 < 1e-6) > 0.5                # most first-layer units are saturated


# ---------------------------------------------------------------------------------------------------------------------------------
# clipping and Adam over 50 updates
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_grad_norm", [1e9, 0.5, 1e-3])
def test_fifty_updates_clipping_and_adam(max_grad_norm):
    """50 consecutive qs_ppo_update calls with non-default lr / betas / eps against 50 oracle updates: the pre-clip gradient norm
    of every step, then parameters, Adam's m and v and the step count.  max_grad_norm 1e9 never clips, 1e-3 clips every step."""
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel
    D, B = 20, 512
    rng = np.random.default_rng(int(-np.log10(max_grad_norm)) + 50)
    sd = perturbed_state_dict(D, 15)
    hp = dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, max_grad_norm=max_grad_norm)
    lr, betas, eps = 1e-3, (0.85, 0.99), 1e-7
    params = torch.from_numpy(blob(sd, D)).cuda()
    opt = PpoUpdateKernel(params, D, learning_rate=lr, betas=betas, eps=eps, **hp)
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    st64 = po.adam_init(sd64)
    norms, errs = [], []
    for it in range(50):
        batch = random_minibatch(rng, B, D, {k: v.astype(np.float32) for k, v in sd64.items()})
        opt.update(*dev(*batch))
        s = po.update(sd64, st64, tuple(np.asarray(x, np.float64) for x in batch), lr=f32(lr), betas=(f32(betas[0]), f32(betas[1])),
                      eps=f32(eps), **{k: f32(v) for k, v in hp.items()})
        k = opt.read_stats()
        norms.append(s["grad_norm"])
        errs.append(abs(k["grad_norm"] - s["grad_norm"]) / s["grad_norm"])
    if max_grad_norm == 1e9:
        assert max(norms) < max_grad_norm
    elif max_grad_norm == 1e-3:
        assert min(norms) > max_grad_norm
    m, v, step = opt.adam_state()
    err_p = np.abs(params.cpu().numpy() - blob(sd64, D)).max()
    m_o, v_o = blob(st64["m"], D), blob(st64["v"], D)
    err_m = np.abs(m.cpu().numpy() - m_o).max() / np.abs(m_o).max()
    err_v = np.abs(v.cpu().numpy() - v_o).max() / np.abs(v_o).max()
    print(f"measured adam {max_grad_norm}: params {err_p:.3g} m {err_m:.3g} v {err_v:.3g} norm {max(errs):.3g} "
          f"(norms {min(norms):.3g}..{max(norms):.3g})")
    assert max(errs) < NORM_TOL_50, max(errs)
    assert int(step.item()) == 50 == st64["step"]
    assert err_p < PARAM_TOL_50 and err_m < MOMENT_TOL and err_v < MOMENT_TOL, (err_p, err_m, err_v)
    opt.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# the multi-rank split: qs_ppo_grad -> average -> qs_ppo_apply
# ---------------------------------------------------------------------------------------------------------------------------------
def _lib():
    from rl_aerial_manipulator_b200._cabi import load_library
    return load_library()


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def test_split_grad_average_apply_vs_oracle():
    """Two half-minibatches through qs_ppo_grad (each normalises its own advantages, as each rank does), their mean, then
    qs_ppo_apply: against the oracle's clip + Adam on the mean of the two half-gradients.  Step 1 passes the averaged gradient
    explicitly; step 2 leaves one half in the handle's own buffer (grad_out NULL), averages in place there and applies with
    grad NULL.  stats_out of qs_ppo_apply: the pre-clip norm in element 4, the other elements untouched."""
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel
    lib = _lib()
    D, half, total = 20, 300, 2000
    rng = np.random.default_rng(21)
    sd = perturbed_state_dict(D, 16)
    buffers = random_minibatch(rng, total, D, sd)
    d_buf = dev(*buffers)
    hp = dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5)
    params = torch.from_numpy(blob(sd, D)).cuda()
    opt = PpoUpdateKernel(params, D, learning_rate=3e-4, **hp)
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    st64 = po.adam_init(sd64)
    m, v, step = opt.adam_state()
    hgrad = C.c_void_p()
    assert lib.qs_ppo_state(opt._h, None, None, None, C.byref(hgrad)) == 0
    handle_grad = torch.empty(0, device="cuda")
    for it in range(2):
        perm = rng.permutation(total)
        idx = [perm[:half].astype(np.int64), perm[half:2 * half].astype(np.int64)]
        g = [torch.zeros_like(params) for _ in range(2)]
        for h in range(2):
            out = None if (it == 1 and h == 0) else g[h]
            assert lib.qs_ppo_grad(opt._h, _p(params), *(_p(x) for x in d_buf), _p(torch.from_numpy(idx[h]).cuda()), half,
                                   C.byref(opt.hp), _p(out), _p(opt.stats), _stream()) == 0
        stats = torch.full((8,), -1.0, device="cuda")
        if it == 0:
            avg = (g[0] + g[1]) * 0.5
            assert lib.qs_ppo_apply(opt._h, _p(params), _p(avg), C.byref(opt.hp), _p(stats), _stream()) == 0
        else:
            assert not g[0].any()                                 # grad_out NULL: the half went to the handle's buffer
            hg = torch.as_tensor(_DeviceView(hgrad.value, params.numel()), device="cuda")
            hg.add_(g[1]).mul_(0.5)
            assert lib.qs_ppo_apply(opt._h, _p(params), None, C.byref(opt.hp), _p(stats), _stream()) == 0
        grads = [po.minibatch_grads(sd64, *(np.asarray(b[i], np.float64) for b in buffers), clip_range=f32(0.2), ent_coef=f32(0.01),
                                    vf_coef=0.5)[1] for i in idx]
        mean = {k: 0.5 * (grads[0][k] + grads[1][k]) for k in grads[0]}
        norm = po.clip_grad_norm(mean, 0.5)
        po.adam_step(sd64, mean, st64, f32(3e-4), betas=F32_BETAS)
        s = stats.cpu().numpy()
        assert abs(s[4] - norm) < STAT_TOL * norm and (np.delete(s, 4) == -1.0).all(), (s, norm)
    err_p = np.abs(params.cpu().numpy() - blob(sd64, D)).max()
    m_o, v_o = blob(st64["m"], D), blob(st64["v"], D)
    err_m = np.abs(m.cpu().numpy() - m_o).max() / np.abs(m_o).max()
    err_v = np.abs(v.cpu().numpy() - v_o).max() / np.abs(v_o).max()
    print(f"measured split: params {err_p:.3g} m {err_m:.3g} v {err_v:.3g}")
    assert int(step.item()) == 2
    assert err_p < PARAM_TOL_50 and err_m < MOMENT_TOL and err_v < MOMENT_TOL, (err_p, err_m, err_v)
    opt.close()


class _DeviceView:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}


def test_update_equals_grad_then_apply_on_one_rank():
    """qs_ppo_update (fused clip + Adam tail) and qs_ppo_grad + qs_ppo_apply on the same minibatches agree to float32 rounding
    over five steps: the two paths differ only in the order of the float64 norm reduction."""
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel
    D, B = 17, 700
    rng = np.random.default_rng(22)
    sd = perturbed_state_dict(D, 17)
    hp = dict(clip_range=0.2, ent_coef=0.01, vf_coef=0.5, max_grad_norm=0.5, learning_rate=1e-3)
    pa, pb = (torch.from_numpy(blob(sd, D)).cuda() for _ in range(2))
    oa, ob = PpoUpdateKernel(pa, D, **hp), PpoUpdateKernel(pb, D, **hp)
    lib = _lib()
    for it in range(5):
        batch = dev(*random_minibatch(rng, B, D, sd))
        oa.update(*batch)
        ob.gradient(*batch)
        assert lib.qs_ppo_apply(ob._h, _p(pb), _p(ob.grad), C.byref(ob.hp), _p(ob.stats), _stream()) == 0
        na, nb = oa.read_stats()["grad_norm"], ob.read_stats()["grad_norm"]
        assert abs(na - nb) <= 2e-7 * na, (na, nb)
    a, b = pa.cpu().numpy(), pb.cpu().numpy()
    ulps = np.abs(a - b) / np.spacing(np.abs(a).astype(np.float32))
    print(f"measured update vs grad+apply: {ulps.max():.3g} ulp")
    assert ulps.max() <= 4, ulps.max()                              # measured: bit-identical
    (ma, va, sa), (mb, vb, sb) = oa.adam_state(), ob.adam_state()
    torch.testing.assert_close(ma, mb, rtol=1e-6, atol=0)
    torch.testing.assert_close(va, vb, rtol=1e-6, atol=0)
    assert int(sa.item()) == int(sb.item()) == 5
    oa.close()
    ob.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# a whole QuadPPO.train() pass
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch_size", [64, 59])
def test_quad_ppo_train_pass_vs_oracle(batch_size):
    """QuadPPO.train() on rollout buffers filled with synthetic data (8 steps x 37 envs = 296 rows): 3 epochs of permuted
    minibatches, batch 64 leaving a ragged 40-row last one, batch 59 a one-row last one; one Adam state through all of them.
    The permutations are regenerated from a clone of ppo.gen and fed to the oracle's train_pass.  Parameters, Adam state and
    step count after the pass; the returned statistics against the oracle's last minibatch (QuadPPO.train reports the last
    minibatch's statistics, where SB3 logs the mean over all minibatches)."""
    from rl_aerial_manipulator_b200.batched_env import BatchedQuadEnv
    from rl_aerial_manipulator_b200.ppo import QuadPPO
    T, n, D, n_epochs = 8, 37, 20, 3
    total = T * n
    env = BatchedQuadEnv(n, env_version=2, precision="f32", seed=0)
    hp = dict(clip_range=0.15, ent_coef=0.01, vf_coef=0.7, max_grad_norm=0.5, learning_rate=3e-4)
    ppo = QuadPPO(env, n_steps=T, batch_size=batch_size, n_epochs=n_epochs, policy_impl="fp32", seed=batch_size, **hp)
    sd = perturbed_state_dict(D, 18)
    ppo.policy.params.copy_(torch.from_numpy(blob(sd, D)))
    rng = np.random.default_rng(batch_size)
    buffers = random_minibatch(rng, total, D, sd)
    for name, x in zip(("obs", "actions", "logp", "advantages", "returns"), buffers):
        getattr(ppo, name).copy_(torch.from_numpy(x).reshape(getattr(ppo, name).shape))
    gen = torch.Generator(device="cuda")
    gen.set_state(ppo.gen.get_state())
    stats_k = ppo.train()
    perms = [torch.randperm(total, device="cuda", generator=gen).cpu().numpy() for _ in range(n_epochs)]
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    st64 = po.adam_init(sd64)
    stats = po.train_pass(sd64, st64, buffers, perms, batch_size, lr=f32(hp["learning_rate"]), betas=F32_BETAS,
                          **{k: f32(v) for k, v in hp.items() if k != "learning_rate"})
    sizes = [len(i) for i in po.minibatches(perms[0], batch_size)]
    assert sizes[-1] == {64: 40, 59: 1}[batch_size]
    m, v, step = ppo.opt.adam_state()
    assert int(step.item()) == st64["step"] == n_epochs * len(sizes)
    err_p = np.abs(ppo.policy.params.cpu().numpy() - blob(sd64, D)).max()
    m_o, v_o = blob(st64["m"], D), blob(st64["v"], D)
    err_m = np.abs(m.cpu().numpy() - m_o).max() / np.abs(m_o).max()
    err_v = np.abs(v.cpu().numpy() - v_o).max() / np.abs(v_o).max()
    print(f"measured train {batch_size}: params {err_p:.3g} m {err_m:.3g} v {err_v:.3g}")
    assert err_p < PARAM_TOL_TRAIN and err_m < MOMENT_TOL and err_v < MOMENT_TOL, (err_p, err_m, err_v)
    last = stats[-1]
    errs = {k: abs(stats_k[k] - last[k]) / max(1.0, abs(last[k])) for k in ("loss", "policy_gradient_loss", "value_loss", "entropy_loss",
                                                                             "approx_kl", "clip_fraction")}
    errs["grad_norm"] = abs(stats_k["grad_norm"] - last["grad_norm"]) / last["grad_norm"]
    print(f"measured train {batch_size} statistics: {max(errs.values()):.3g} ({max(errs, key=errs.get)})")
    assert max(errs.values()) < STAT_TOL, errs
    assert stats_k["batch_size"] == sizes[-1]
    env.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------------------------------
def test_refusals():
    """QS_EINVAL and a message, nothing launched: an empty minibatch, misaligned actions, obs_dim outside {17, 20}, NULL buffers."""
    from rl_aerial_manipulator_b200.ppo import PpoUpdateKernel
    lib = _lib()
    h = C.c_void_p()
    for D in (0, 18, 21):
        assert lib.qs_ppo_create(0, D, C.byref(h)) == QS_EINVAL and b"obs_dim 17 or 20" in lib.qs_ppo_last_error()
    assert lib.qs_ppo_n_params(18) == -1
    D, B = 20, 64
    sd = perturbed_state_dict(D, 19)
    params = torch.from_numpy(blob(sd, D)).cuda()
    before = params.clone()
    opt = PpoUpdateKernel(params, D)
    obs, act, oldlp, adv, ret = dev(*random_minibatch(np.random.default_rng(0), B, D, sd))
    act_mis = torch.zeros(B * 4 + 1, device="cuda")[1:]           # 4 bytes past a 16-byte boundary
    args = [_p(obs), _p(act), _p(oldlp), _p(adv), _p(ret)]

    def both(a, n, msg):
        for fn, extra in ((lib.qs_ppo_update, ()), (lib.qs_ppo_grad, (_p(opt.grad),))):
            rc = fn(opt._h, _p(params), *a, None, n, C.byref(opt.hp), *extra, _p(opt.stats), _stream())
            assert rc == QS_EINVAL and msg in lib.qs_ppo_last_error(), (fn, rc, lib.qs_ppo_last_error())

    both(args, 0, b"empty minibatch")
    both(args, -5, b"empty minibatch")
    both([args[0], _p(act_mis)] + args[2:], B, b"16-byte aligned")
    for i in range(5):
        both(args[:i] + [None] + args[i + 1:], B, b"null argument")
    assert lib.qs_ppo_update(None, _p(params), *args, None, B, C.byref(opt.hp), None, _stream()) == QS_EINVAL
    assert lib.qs_ppo_apply(opt._h, None, _p(opt.grad), C.byref(opt.hp), None, _stream()) == QS_EINVAL
    assert lib.qs_ppo_apply(opt._h, _p(params), _p(opt.grad), None, None, _stream()) == QS_EINVAL
    assert b"null argument" in lib.qs_ppo_last_error()
    torch.cuda.synchronize()
    assert torch.equal(params, before) and int(opt.adam_state()[2].item()) == 0
    opt.update(obs, act, oldlp, adv, ret)                          # the handle still works after the refusals
    assert int(opt.adam_state()[2].item()) == 1 and not torch.equal(params, before)
    opt.close()
