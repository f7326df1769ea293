"""Helpers of the action-repeat tests (swarm_step_repeat): what one repeat-K call must report, folded from the K single
steps of a twin env that does not auto-reset."""
import numpy as np


def substep_elapsed(elapsed0, K, max_steps):
    """TimeLimit counters after each substep of one call -> (elapsed (K,E) int64, truncated (K,E) bool).  elapsed
    advances by one per substep; max_steps <= 0 is no TimeLimit."""
    el = np.asarray(elapsed0, dtype=np.int64)[None, :] + np.arange(1, K + 1, dtype=np.int64)[:, None]
    return el, (el >= max_steps) if max_steps > 0 else np.zeros(el.shape, dtype=bool)


def fold_substeps(rewards, dones):
    """rewards (K,E) f32 and dones (K,E) bool of K single steps -> (reward (E,) f32, done (E,) bool, last (E,) int):
    each env stops at its first done substep (`last`, else K - 1); reward is the FP32 sum of its stepped substeps'
    rewards in substep order, starting from the first substep's; done is the last stepped substep's."""
    rewards = np.asarray(rewards, dtype=np.float32)
    dones = np.asarray(dones, dtype=bool)
    K, E = rewards.shape
    last = np.where(dones.any(axis=0), dones.argmax(axis=0), K - 1)
    reward = rewards[0].copy()
    for s in range(1, K):
        on = s <= last
        reward[on] = reward[on] + rewards[s][on]          # float32 + float32: one rounding, like __fadd_rn
    return reward, dones[last, np.arange(E)], last
