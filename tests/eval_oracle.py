"""NumPy restatement of stable_baselines3.common.evaluation.evaluate_policy's episode loop (SB3 2.6.0), driven by given per-step done
flags, Monitor returns and lengths instead of a policy and an env:

    episode_counts = np.zeros(n_envs, dtype="int")
    episode_count_targets = np.array([(n_eval_episodes + i) // n_envs for i in range(n_envs)], dtype="int")
    observations = env.reset()
    while (episode_counts < episode_count_targets).any():
        actions, states = model.predict(observations, ...)
        new_observations, rewards, dones, infos = env.step(actions)
        for i in range(n_envs):
            if episode_counts[i] < episode_count_targets[i]:
                if dones[i]:
                    episode_rewards.append(info["episode"]["r"]); episode_lengths.append(info["episode"]["l"])
                    episode_counts[i] += 1
Test infrastructure only."""
import numpy as np


def sb3_episodes(E, flags, ep_return, ep_len):
    """flags u8[T, G] (QS_FLAG_* bits; done = terminated | truncated), ep_return / ep_len [T, G] (read where done).
    Returns dict: ret / len / flags / step / env_id of the recorded episodes in SB3's order; remaining[T] = envs below their
    target after each step (0 once the loop has ended); slot-major arrays slot_ret / slot_len / slot_flags / slot_step where env
    i's k-th episode sits at sum(targets[:i]) + k."""
    T, G = flags.shape
    counts = np.zeros(G, dtype=np.int64)
    tgt = np.array([(E + i) // G for i in range(G)], dtype=np.int64)
    base = np.concatenate([[0], np.cumsum(tgt)[:-1]])
    rec = {k: [] for k in ("ret", "len", "flags", "step", "env_id")}
    slot = {k: np.zeros(E, dtype=dt) for k, dt in (("ret", np.float64), ("len", np.int32), ("flags", np.uint8), ("step", np.int32))}
    remaining = np.zeros(T, dtype=np.int64)
    for t in range(T):
        if not (counts < tgt).any():
            break
        for i in range(G):
            if counts[i] < tgt[i] and (flags[t, i] & 3):
                for k, v in (("ret", float(ep_return[t, i])), ("len", int(ep_len[t, i])), ("flags", int(flags[t, i])), ("step", t)):
                    rec[k].append(v)
                    slot[k][base[i] + counts[i]] = v
                rec["env_id"].append(i)
                counts[i] += 1
        remaining[t] = int((counts < tgt).sum())
    out = {k: np.array(v) for k, v in rec.items()}
    out.update({"slot_" + k: v for k, v in slot.items()}, remaining=remaining, targets=tgt, base=base)
    return out


def random_streams(rng, T, G, p_done=0.1, f64=True):
    """Random done streams: flags with terminated / truncated / info bits, returns and lengths (garbage where not done)."""
    done = rng.random((T, G)) < p_done
    bits = rng.integers(0, 256, (T, G)).astype(np.uint8) & np.uint8(0xFC)
    kind = rng.integers(1, 4, (T, G)).astype(np.uint8)              # 1 terminated, 2 truncated, 3 both
    flags = np.where(done, bits | kind, bits).astype(np.uint8)
    ret = rng.normal(0, 1000, (T, G))
    ret = ret if f64 else ret.astype(np.float32)
    ln = rng.integers(1, 2001, (T, G)).astype(np.int32)
    return flags, ret, ln
