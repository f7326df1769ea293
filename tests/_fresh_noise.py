"""Test helpers for fresh per-step noise (SWARM_STEP_FRESH_NOISE: the reference with SURVEY Q1 fixed, step k of an episode
uses noise row N_BURN_IN + k), built on the unchanged oracle (oracle/swarm_oracle.py, oracle/philox.py).

  noise_rows        rows row0.. of the Philox noise streams 3 / 4 of one episode (what swarm_philox_noise_rows exports)
  draw_reset_full   the reference's reset draws in its order, keeping all 138 rows of the noise tables
  FreshOracleRunner so.OracleRunner that keeps each env's episode tables and steps env e with row N_BURN_IN + elapsed[e]
"""
import numpy as np

from oracle import philox as ph
from oracle import swarm_oracle as so

TABLE_ROWS = 128 + so.N_BURN_IN       # multiagent.py:55-56: one row per burn-in step + one per step of a 128-step episode


def noise_rows(seed, env_id, episode, row0, n_rows, n_locusts, n_agents=so.N_AGENTS):
    """-> (an (n_rows,A,2), pn (n_rows,N,2)), unscaled, FP32 Box-Muller as the device draws them (oracle/philox.py)."""
    rows = range(row0, row0 + n_rows)
    an = np.stack([ph.normal_pairs(seed, env_id, episode, ph.STREAM_NOISE_A, r, n_agents) for r in rows])
    pn = np.stack([ph.normal_pairs(seed, env_id, episode, ph.STREAM_NOISE_X, r, n_locusts) for r in rows])
    return an, pn


def draw_reset_full(rs, n_locusts, n_agents=so.N_AGENTS):
    """so.draw_reset_numpy (same draws, same order) without cutting the noise tables to rows 0..10."""
    x0 = rs.rand(n_locusts, 2)
    xa0 = rs.rand(n_agents, 2)
    burn = rs.normal(size=(so.N_BURN_IN, n_agents, 2))
    an = rs.normal(size=(TABLE_ROWS, n_agents, 2))
    pn = rs.normal(size=(TABLE_ROWS, n_locusts, 2))
    return x0, xa0, burn, an, pn


class FreshOracleRunner(so.OracleRunner):
    """so.OracleRunner with the frozen index fixed: the draws of an episode carry as many noise rows as it reads, and the
    step proper of env e uses row N_BURN_IN + elapsed[e] of them (IndexError when a table runs out, like the fixed
    reference).  Auto-reset and TimeLimit are the base class's."""

    def __init__(self, n_envs, n_locusts, draws, **kw):
        self.tables = [None] * n_envs

        def keep(e, episode):
            d = draws(e, episode)
            self.tables[e] = (d[3], d[4])
            return d

        super(FreshOracleRunner, self).__init__(n_envs, n_locusts, keep, **kw)

    def step(self, actions):
        rows = so.N_BURN_IN + self.elapsed
        for e in range(self.E):          # the base step reads self.na / self.nx; a reset inside it sets row 10 again
            self.na[e], self.nx[e] = self.tables[e][0][rows[e]], self.tables[e][1][rows[e]]
        return super(FreshOracleRunner, self).step(actions)
