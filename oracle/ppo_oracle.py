"""TEST INFRASTRUCTURE ONLY -- restatement of Stable-Baselines3's PPO minibatch update (SB3 2.6.0 `PPO.train`, as the reference
calls it: initial-implementation-v1/rl_train_vecN.py:13-36, initial-implementation-v2/rl_train.py:27-56), twice:

  * NumPy float64, forward AND hand-derived backward (`minibatch_grads`, `clip_grad_norm`, `adam_step`, `update`; `train_pass`
    for a whole PPO.train): the checker of the CUDA update kernel (csrc/qs_ppo.cu);
  * torch autograd (`TorchActorCritic`, `ppo_loss`, `torch_update`): the same update the way SB3 itself computes it
    (nn.Linear / Tanh modules, autograd, clip_grad_norm_, torch.optim.Adam(eps=1e-5)); pins the NumPy backward
    (tests/test_ppo.py) and is the second checker of the kernel.

Parity unpinned against SB3 itself: stable_baselines3 is not installable in this image; both restatements follow its source.
Nothing in the product package imports this module.
"""
from __future__ import annotations

import math

import numpy as np

H1, H2, H3, NACT = 128, 64, 64, 4
LOG_2PI = math.log(2.0 * math.pi)


# ---------------------------------------------------------------------------------------------------------------------
# NumPy float64: forward + backward by hand
# ---------------------------------------------------------------------------------------------------------------------
def _mlp_forward(sd, net, x):
    acts = [x]
    for i in (0, 2, 4):
        x = np.tanh(x @ sd[f"mlp_extractor.{net}.{i}.weight"].T + sd[f"mlp_extractor.{net}.{i}.bias"])
        acts.append(x)
    return acts


def _mlp_backward(sd, net, acts, d_out, grads):
    """d_out = dL/d(last hidden activation); fills grads of the three Linear layers of `net`."""
    d = d_out
    for li, i in zip((3, 2, 1), (4, 2, 0)):
        dz = d * (1.0 - acts[li] ** 2)
        grads[f"mlp_extractor.{net}.{i}.weight"] = dz.T @ acts[li - 1]
        grads[f"mlp_extractor.{net}.{i}.bias"] = dz.sum(0)
        d = dz @ sd[f"mlp_extractor.{net}.{i}.weight"]


def minibatch_grads(sd, obs, actions, old_logp, advantages, returns, clip_range=0.2, ent_coef=0.0, vf_coef=0.5,
                    normalize_advantage=True):
    """One minibatch of PPO.train (clip_range_vf=None): returns (stats, grads) with stats = loss, policy_gradient_loss,
    value_loss, entropy_loss, clip_fraction, approx_kl and grads keyed like the SB3 state dict.  clip_fraction and approx_kl
    are SB3's diagnostics: mean(|ratio - 1| > clip_range) and mean((ratio - 1) - log_ratio)."""
    sd = {k: np.asarray(v, np.float64) for k, v in sd.items()}
    obs, actions = np.asarray(obs, np.float64), np.asarray(actions, np.float64)
    old_logp, adv, ret = (np.asarray(a, np.float64) for a in (old_logp, advantages, returns))
    B = obs.shape[0]
    if normalize_advantage and B > 1:
        adv = (adv - adv.mean()) / (adv.std(ddof=1) + 1e-8)            # torch.std: Bessel's correction
    pa, va = _mlp_forward(sd, "policy_net", obs), _mlp_forward(sd, "value_net", obs)
    mean = pa[3] @ sd["action_net.weight"].T + sd["action_net.bias"]
    values = (va[3] @ sd["value_net.weight"].T + sd["value_net.bias"])[:, 0]
    log_std = sd["log_std"]
    z = (actions - mean) / np.exp(log_std)
    logp = (-0.5 * z ** 2 - log_std - 0.5 * LOG_2PI).sum(1)
    entropy = (0.5 + 0.5 * LOG_2PI + log_std).sum()
    log_ratio = logp - old_logp
    ratio = np.exp(log_ratio)
    s1, s2 = adv * ratio, adv * np.clip(ratio, 1 - clip_range, 1 + clip_range)
    pg = -np.minimum(s1, s2).mean()
    vf = ((returns - values) ** 2).mean()
    ent = -entropy
    loss = pg + ent_coef * ent + vf_coef * vf
    # ---- backward
    inside = (ratio >= 1 - clip_range) & (ratio <= 1 + clip_range)
    # d min(s1, s2) / d ratio: A where the unclipped term is the (strict) minimum or the clip is inactive, else 0
    d_ratio = np.where(inside | (s1 < s2), adv, 0.0)
    d_logp = -(d_ratio * ratio) / B
    grads = {}
    d_mean = d_logp[:, None] * z / np.exp(log_std)
    grads["log_std"] = (d_logp[:, None] * (z ** 2 - 1.0)).sum(0) - ent_coef * np.ones(NACT)
    grads["action_net.weight"] = d_mean.T @ pa[3]
    grads["action_net.bias"] = d_mean.sum(0)
    _mlp_backward(sd, "policy_net", pa, d_mean @ sd["action_net.weight"], grads)
    d_val = (vf_coef * 2.0 * (values - ret) / B)[:, None]
    grads["value_net.weight"] = d_val.T @ va[3]
    grads["value_net.bias"] = d_val.sum(0)
    _mlp_backward(sd, "value_net", va, d_val @ sd["value_net.weight"], grads)
    stats = {"loss": loss, "policy_gradient_loss": pg, "value_loss": vf, "entropy_loss": ent,
             "clip_fraction": float(np.mean(np.abs(ratio - 1.0) > clip_range)), "approx_kl": float(np.mean((ratio - 1.0) - log_ratio))}
    return stats, grads


def clip_grad_norm(grads, max_norm):
    """torch.nn.utils.clip_grad_norm_: scale every gradient by min(1, max_norm / (total_norm + 1e-6)); returns the norm."""
    total = math.sqrt(sum(float((g ** 2).sum()) for g in grads.values()))
    coef = min(1.0, max_norm / (total + 1e-6))
    for k in grads:
        grads[k] = grads[k] * coef
    return total


def adam_init(sd):
    return {"step": 0, "m": {k: np.zeros_like(np.asarray(v, np.float64)) for k, v in sd.items()},
            "v": {k: np.zeros_like(np.asarray(v, np.float64)) for k, v in sd.items()}}


def adam_step(sd, grads, state, lr, betas=(0.9, 0.999), eps=1e-5):
    """torch.optim.Adam (no weight decay, no amsgrad), in place on float64 copies."""
    state["step"] += 1
    t = state["step"]
    b1, b2 = betas
    bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
    for k, g in grads.items():
        m, v = state["m"][k], state["v"][k]
        m += (g - m) * (1.0 - b1)
        v *= b2
        v += (1.0 - b2) * g * g
        sd[k] = sd[k] - (lr / bc1) * m / (np.sqrt(v) / math.sqrt(bc2) + eps)


def update(sd, state, batch, lr=2e-4, clip_range=0.2, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5, normalize_advantage=True,
           betas=(0.9, 0.999), eps=1e-5):
    """One full minibatch update in float64; sd (float64 dict) and state are modified in place.  Returns the loss statistics
    with the pre-clip gradient norm and the minibatch size."""
    stats, grads = minibatch_grads(sd, *batch, clip_range=clip_range, ent_coef=ent_coef, vf_coef=vf_coef,
                                   normalize_advantage=normalize_advantage)
    stats["grad_norm"] = clip_grad_norm(grads, max_grad_norm)
    stats["batch_size"] = len(batch[0])
    adam_step(sd, grads, state, lr, betas=betas, eps=eps)
    return stats


def minibatches(perm, batch_size):
    """RolloutBuffer.get(batch_size): consecutive slices of one epoch's permutation, the ragged last one kept."""
    total = len(perm)
    bs = min(batch_size, total)
    return [perm[start:start + bs] for start in range(0, total, bs)]


def train_pass(sd, state, buffers, perms, batch_size, **hp):
    """PPO.train in float64: one epoch per permutation in `perms`, each cut into minibatches by `minibatches`, one `update`
    per minibatch with one Adam state threaded through all of them.  `buffers` = (obs, actions, old_logp, advantages,
    returns), flattened to rows.  sd and state are modified in place; returns every minibatch's statistics in order."""
    buffers = tuple(np.asarray(b, np.float64) for b in buffers)
    out = []
    for perm in perms:
        for idx in minibatches(np.asarray(perm), batch_size):
            out.append(update(sd, state, tuple(b[idx] for b in buffers), **hp))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# torch autograd: the update the way SB3 computes it
# ---------------------------------------------------------------------------------------------------------------------
def make_torch_actor_critic(sd: dict, obs_dim: int, dtype=None):
    import torch
    import torch.nn as nn

    class TorchActorCritic(nn.Module):
        """SB3 ActorCriticPolicy(net_arch=[128, 64, 64], Tanh) with SB3's parameter names."""

        def __init__(self):
            super().__init__()
            mk = lambda: nn.Sequential(nn.Linear(obs_dim, H1), nn.Tanh(), nn.Linear(H1, H2), nn.Tanh(), nn.Linear(H2, H3), nn.Tanh())
            self.mlp_extractor = nn.ModuleDict({"policy_net": mk(), "value_net": mk()})
            self.action_net, self.value_net = nn.Linear(H3, NACT), nn.Linear(H3, 1)
            self.log_std = nn.Parameter(torch.zeros(NACT))
            if dtype is not None:
                self.to(dtype)
            self.load_state_dict({k: torch.as_tensor(np.asarray(v)) for k, v in sd.items()})

        def evaluate_actions(self, obs, actions):
            """ActorCriticPolicy.evaluate_actions: values, log_prob(actions), entropy."""
            mean = self.action_net(self.mlp_extractor["policy_net"](obs))
            values = self.value_net(self.mlp_extractor["value_net"](obs))[:, 0]
            logp = (-0.5 * ((actions - mean) / self.log_std.exp()) ** 2 - self.log_std - 0.5 * LOG_2PI).sum(1)
            entropy = (0.5 + 0.5 * LOG_2PI + self.log_std).sum().expand_as(logp)
            return values, logp, entropy

    return TorchActorCritic()


def ppo_loss(values, logp, entropy, old_logp, advantages, returns, clip_range: float, ent_coef: float, vf_coef: float,
             normalize_advantage: bool = True):
    """SB3 PPO.train loss for one minibatch (clip_range_vf=None), torch."""
    import torch

    if normalize_advantage and advantages.numel() > 1:
        advantages = (advantages - advantages.mean()) / (advantages.std() + 1e-8)
    ratio = torch.exp(logp - old_logp)
    pg = -torch.min(advantages * ratio, advantages * torch.clamp(ratio, 1 - clip_range, 1 + clip_range)).mean()
    vf = torch.nn.functional.mse_loss(returns, values)
    ent = -entropy.mean()
    return pg + ent_coef * ent + vf_coef * vf, pg, vf, ent


def torch_update(net, opt, batch, clip_range=0.2, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5, normalize_advantage=True):
    """One minibatch update with autograd + clip_grad_norm_ + opt.step(); returns (loss, pg, vf, ent, grad_norm, clip_fraction,
    approx_kl) as floats, the last two computed as SB3 2.6.0's PPO.train does."""
    import torch
    import torch.nn as nn

    obs, act, oldlp, adv, ret = batch
    values, logp, entropy = net.evaluate_actions(obs, act)
    loss, pg, vf, ent = ppo_loss(values, logp, entropy, oldlp, adv, ret, clip_range, ent_coef, vf_coef, normalize_advantage)
    with torch.no_grad():
        log_ratio = logp - oldlp
        ratio = torch.exp(log_ratio)
        clip_fraction = torch.mean((torch.abs(ratio - 1) > clip_range).float())
        approx_kl = torch.mean((ratio - 1) - log_ratio)
    opt.zero_grad(set_to_none=False)
    loss.backward()
    gn = nn.utils.clip_grad_norm_(net.parameters(), max_grad_norm)
    opt.step()
    return tuple(float(x.detach()) for x in (loss, pg, vf, ent, gn, clip_fraction, approx_kl))
