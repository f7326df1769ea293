"""Host-side mirror of fed_gym/agents/paac/runners.py:7-66 (Runners / GridRunners).

The reference shares six RawArray-backed numpy arrays between the learner and W worker processes
and synchronises them with queues.  Here the six "shared variables" are CUDA tensors owned by the
runner and updated in place by kernels on the current stream:

  update_environments()  one swarm_step launch (step + TimeLimit + auto-reset + rasterise) followed
                         by one swarm_expand_obs launch; returns immediately (asynchronous, like
                         the reference's queue put, runners.py:45-50)
  wait_updated()         records nothing and blocks nothing for same-stream consumers (the policy
                         forward is enqueued behind the step); pass sync=True to block the host.
"""
import torch

from .emulator_runner import SwarmRunner


class GridRunners(object):
    def __init__(self, emulators, workers=None, variables=None, emulator_class=SwarmRunner, coord=None,
                 grid_size=84, expand=True):
        """emulators: a BatchedSwarmEnv (the whole emulator batch).  ``workers`` is accepted for
        signature compatibility (runners.py:57) and ignored: there are no worker processes."""
        env = emulators
        if env.G != grid_size:
            raise ValueError("env grid_size %d != runner grid_size %d" % (env.G, grid_size))
        self.env = env
        self.workers = workers
        self.coord = coord
        self.emulator_class = emulator_class
        self.expand = expand
        E, A, G, d = env.E, env.A, env.G, env.device
        self.states = torch.zeros(E, A, G, G, 3, dtype=torch.float32, device=d) if expand else None
        # histories: unused by ConvSingleAgentPolicyNetwork (paac.py:355-356) -> empty placeholder
        self.histories = torch.zeros(E, A, 0, dtype=torch.float32, device=d)
        self.rewards = torch.zeros(E, A, dtype=torch.float32, device=d)
        self.episode_over = torch.zeros(E, A, dtype=torch.float32, device=d)
        self.actions = env.actions                      # (E,A,2) f32, written in place by the learner
        self.variables = [self.states, self.histories, env.positions, self.rewards, self.episode_over, self.actions]
        self._started = False
        self.final_info = {}

    def start(self, states_out=None):
        """runners.py:34-36.  Initial reset + first observation (paac.py:247-251 does this in the parent).
        states_out: optional (E,A,G,G,3) tensor that receives the expanded observation instead of self.states."""
        self.env.reset()
        self.env.observe()
        if states_out is not None:
            self.env.local_states(out=states_out)
        elif self.expand:
            self.env.local_states(out=self.states)
        self._started = True

    def stop(self):
        self._started = False

    def get_shared_variables(self):
        return self.variables

    def update_environments(self, states_out=None, grid_out=None, positions_out=None, final_grid_out=None,
                            final_positions_out=None):
        """states_out: optional (E,A,G,G,3) tensor that receives the new expanded observation directly (the
        device-resident learner points it at its rollout ring, saving one 847 KB/env copy per step).
        final_grid_out / final_positions_out: the same for the terminal observation of the envs whose episode ended
        (an env built with final_obs=True; its info dict -- terminated, truncated, final_* -- is self.final_info)."""
        if self.coord is not None and self.coord.should_stop():
            self.stop()
            return
        env = self.env
        if getattr(env, "final_obs", False):
            _, reward, done, self.final_info = env.step(self.actions, rasterize=True, auto_reset=True, grid_out=grid_out,
                                                        positions_out=positions_out, final_grid_out=final_grid_out,
                                                        final_positions_out=final_positions_out)
        else:
            _, reward, done, _ = env.step(self.actions, rasterize=True, auto_reset=True, grid_out=grid_out,
                                          positions_out=positions_out)
        if grid_out is not None:
            pass                                    # compact consumer: no expanded observation at all
        elif states_out is not None:
            env.local_states(out=states_out)
        elif self.expand:
            env.local_states(out=self.states)
        # reward / done scalars broadcast over the agent axis (emulator_runner.py:147-148)
        self.rewards.copy_(reward[:, None].expand_as(self.rewards))
        self.episode_over.copy_(done[:, None].expand_as(self.episode_over))

    def wait_updated(self, sync=False):
        if sync:
            torch.cuda.current_stream(self.env.device).synchronize()


Runners = GridRunners
