"""Mirror of fed_gym/agents/paac/environment_creator.py:16-20 (SwarmEnvironmentCreator).

``create_environment()`` keeps the reference meaning (one 'Swarm-v0' env, 128-step TimeLimit);
``create_batched_environment(E, ...)`` is what the device-resident learner uses instead of E of them.
``noise``: "frozen" (the reference) or "fresh" (SURVEY Q1 fixed), see BatchedSwarmEnv.
``final_obs=True``: the batched env also keeps each ended episode's terminal state and observation (BatchedSwarmEnv).
``physics``: per-env physics of the batched envs (BatchedSwarmEnv's ``physics``: "table" or {column: (lo, hi)}).
"""
from ...envs import multiagent as ma


class SwarmEnvironmentCreator(object):
    def __init__(self, n_locusts=None, grid_size=84, math_mode="fast", noise="frozen", physics=None):
        self.num_actions = 2
        self.n_locusts = n_locusts
        self.grid_size = grid_size
        self.math_mode = math_mode
        self.noise = noise
        self.physics = physics

    def create_environment(self):
        return ma.make("Swarm-v0", fresh_noise=self.noise == "fresh")

    def create_batched_environment(self, num_envs, seed=0, env_id_offset=0, device=None, final_obs=False):
        return ma.BatchedSwarmEnv(num_envs, n_locusts=self.n_locusts, grid_size=self.grid_size,
                                  max_episode_steps=ma.REGISTRY["Swarm-v0"]["max_episode_steps"], seed=seed,
                                  env_id_offset=env_id_offset, device=device, math_mode=self.math_mode,
                                  auto_reset=True, rasterize=True, noise=self.noise, final_obs=final_obs,
                                  physics=self.physics)
