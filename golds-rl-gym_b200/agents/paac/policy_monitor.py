"""Mirror of fed_gym/agents/paac/policy_monitor.py:129-208 (SwarmPolicyMonitor).

One seeded evaluation episode on 'Swarm-eval-v0' (seed 192, 128-step TimeLimit) with the current policy:
copy the learner's parameters, reset, then predict -> sample -> transform_actions_for_env -> step ->
process_state -> get_local_states until done; track the best score and dump its action sequence to
``swarm-eval.json`` as {"score": float, "actions": [T][A][2]} -- the file scripts/make_swarm_gif.py of the
reference replays (make_swarm_gif.py:62-67).  Summaries keep the reference tags eval/total_reward and
eval/episode_length (returned as a dict; a tensorboard SummaryWriter is used when one is passed in).

The eval env is the E=1 view of the batched CUDA env, the observation the rasteriser kernel's.  With ``action_repeat``
K > 1 (the training envs' action repeat) each chosen action is stepped K times, stopping at done, and the rewards are
summed, so that eval scores are on the scale of the training rewards; the episode length counts decisions.
"""
import copy
import json
import logging
import os
import time

import numpy as np
import torch

from ...envs import multiagent as ma
from .emulator_runner import SwarmRunner


class SwarmPolicyMonitor(object):
    def __init__(self, env=None, global_policy_net=None, state_processor=None, summary_writer=None, saver=None,
                 network_conf=None, out_dir=".", fresh_noise=False, action_repeat=1):
        # fresh_noise: the default eval env follows the training envs' noise mode (SURVEY Q1 fixed or not)
        self.env = env if env is not None else ma.make("Swarm-eval-v0", fresh_noise=fresh_noise)
        self.global_policy_net = global_policy_net
        self.state_processor = state_processor
        self.summary_writer = summary_writer
        self.best_score = -np.inf
        self.out_dir = out_dir
        self.action_repeat = int(action_repeat)
        if self.action_repeat < 1:
            raise ValueError("action_repeat must be >= 1")
        self.policy_net = self._create_policy_estimator(global_policy_net)

    @staticmethod
    def _create_policy_estimator(global_net):
        net = copy.deepcopy(global_net)
        for p in net.parameters():
            p.requires_grad_(False)
        return net

    def copy_params(self):
        """make_copy_params_op (policy_monitor.py:39-42): global -> local evaluation net."""
        self.policy_net.load_state_dict(self.global_policy_net.state_dict())

    def get_action_from_policy(self, processed_state, history=None, positions=None, sess=None):
        """policy_monitor.py:131-135: mu + sigma * N(0,1) drawn from numpy's global RNG, then clipped."""
        dev = next(self.policy_net.parameters()).device
        pred = self.policy_net.predict(torch.as_tensor(processed_state, dtype=torch.float32, device=dev))
        mu, sigma = pred["mu"].cpu().numpy().astype(np.float64), pred["sigma"].cpu().numpy().astype(np.float64)
        raw = (mu + sigma * np.random.normal(size=mu.shape)).astype(np.float32)
        a = torch.as_tensor(raw, device=dev).contiguous()
        return SwarmRunner.transform_actions_for_env(a).cpu().numpy()

    def _save_actions(self, score, actions):
        with open(os.path.join(self.out_dir, "swarm-eval.json"), "w") as f:
            json.dump({"score": score, "actions": actions}, f)

    def _observe(self, state):
        g = self.state_processor.process_state(state)                       # (G,G,2) float64, sets .positions
        dev = next(self.policy_net.parameters()).device
        obs = SwarmRunner.get_local_states(torch.as_tensor(g, dtype=torch.float32, device=dev),
                                           torch.as_tensor(self.state_processor.positions, device=dev))
        return obs                                                          # (A,G,G,3)

    def eval_once(self, sess=None, max_sequence_length=5, actions=None, global_step=0):
        self.copy_params()
        state = self.env.reset()
        obs = self._observe(state)
        done, total_reward, episode_length, rewards, taken = False, 0.0, 0, [], []
        while not done:
            action = self.get_action_from_policy(obs) if actions is None else np.asarray(actions.get(), dtype=np.float32)
            taken.append(np.asarray(action).tolist())
            reward = 0.0
            for _ in range(self.action_repeat):
                state, r, done, _ = self.env.step(action)
                reward += float(r)
                if done:
                    break
            obs = self._observe(state)
            total_reward += float(reward)
            episode_length += 1
            rewards.append(float(reward))
        if total_reward > self.best_score:
            self.best_score = total_reward
            self._save_actions(total_reward, taken)
        summary = {"eval/total_reward": total_reward, "eval/episode_length": episode_length}
        if self.summary_writer is not None:
            for k, v in summary.items():
                self.summary_writer.add_scalar(k, v, global_step)
            self.summary_writer.flush()
        logging.info("Eval results at step %d: avg_reward %s, std_reward %s, episode_length %d",
                     global_step, np.mean(rewards), np.std(rewards), episode_length)
        return total_reward, episode_length, rewards

    def continuous_eval(self, eval_every, sess=None, coord=None, max_seq_length=5, max_evals=None):
        n = 0
        while (coord is None or not coord.should_stop()) and (max_evals is None or n < max_evals):
            self.eval_once(max_sequence_length=max_seq_length)
            n += 1
            time.sleep(eval_every)
