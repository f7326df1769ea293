"""Helpers of the per-env physics tests (SwarmPhysics), built on the unchanged oracle: the NumPy restatement of a
SWARM_PHYSICS_RESAMPLE row and an oracle step with explicit constants."""
import numpy as np

from oracle import philox
from oracle import swarm_oracle as so

COLUMNS = ("noise", "gravity", "wind", "F", "L", "dt")
STREAM_PHYSICS = 5
DEFAULT_ROW = np.array([so.NOISE, so.GRAVITY, so.WIND_SPEED, so.F_ATTR, so.L_ATTR, so.DT], dtype=np.float64)


def resampled_row(seed, env_id, episode, lo, hi):
    """Row drawn by the reset of global env `env_id` whose episode word (before the reset's increment) is `episode`:
    column c = lo + (hi - lo) u (each operation rounded once), u = uniform pair c // 2 of Philox stream 5, .x / .y."""
    u = philox.uniform_pairs(seed, env_id, episode, STREAM_PHYSICS, 3).reshape(6)
    lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
    return lo + (hi - lo) * u


def resampled_rows(seed, env_ids, episodes, lo, hi):
    return np.stack([resampled_row(seed, int(g), int(ep), lo, hi) for g, ep in zip(env_ids, episodes)])


def step_with(x, xa, actions, noise_a, noise_x, row, add_wind=True):
    """so.step with the constants of `row` ({noise, gravity, wind, F, L, dt}) for a batch that shares them; in place on
    x, xa.  Returns (reward, v)."""
    noise, grav, wind, F, L, dt = [float(c) for c in row]
    va = np.array(actions, dtype=np.float64, copy=True)
    if add_wind:
        va[..., 0] += wind
    so.move_(xa, va, noise * np.asarray(noise_a, dtype=np.float64), dt)
    v, reward = so.forces(x, xa, F, L, wind, grav)
    so.move_(x, v.copy(), noise * np.asarray(noise_x, dtype=np.float64), dt)
    return reward, v


def random_rows(n, rng, F=(0.2, 0.9), L=(2.0, 20.0), wind=(-2.0, 2.0), gravity=(-2.0, 0.5), dt=(0.01, 0.1),
                noise=(0.0, 1e-3)):
    """n rows spread over the given ranges (SwarmPhysics column order)."""
    rows = np.empty((n, 6), dtype=np.float64)
    for c, rng_c in enumerate((noise, gravity, wind, F, L, dt)):
        rows[:, c] = rng.uniform(rng_c[0], rng_c[1], size=n)
    return rows
