"""Device-resident mirror of fed_gym/agents/paac/paac.py:216-419 (GridPAACLearner) and of the optimiser
wiring in fed_gym/agents/paac/actor_learner.py:31-119.

Same algorithm and hyper-parameters as the reference (T = max_local_steps rollout, n-step returns bootstrapped
from V(s_T), advantages / scale, Adam with linear LR annealing, global-norm clipping), but nothing leaves the
GPU between the policy forward and env.step:

  predict -> sample (mu + sigma * N(0,1)) -> transform_actions_for_env (in place) -> shared_actions
          -> GridRunners.update_environments()  = ONE swarm_step launch + ONE swarm_expand_obs launch
  and the T rollout steps are replayed as one CUDA graph (launch-bound at 32 emulators).

Multi-GPU: one process per GPU, the emulator batch is sharded (sharding.shard_envs, global env ids key the
reset RNG), parameters are broadcast from rank 0 and the flat FP32 gradient (8.84 MB) is all-reduced (mean) over
NCCL once per update -- the only collective; clipping and Adam then run identically on every rank.

Reference quirks at this boundary (SURVEY.md section 8a), selectable:
  reward_indexing="reference"  rewards[t, e_idx] for e_idx < E only (paac.py:331-338, Q6); "per_agent" = fixed
  mask_terminals=False         returns bootstrap through episode ends (paac.py:363 commented mask, Q7)
  bootstrap_truncated=True     (with mask_terminals=True) a TimeLimit truncation is bootstrapped from V of the episode's
                               terminal observation instead of being cut to 0 like a termination:
                               ret_t = r_t + gamma [(1 - done_t) ret_t+1 + truncated_t (1 - terminated_t) V(final_t)]
"""
import logging
import time

import torch
import torch.distributed as dist

from ... import sharding
from .emulator_runner import SwarmRunner
from .runners import GridRunners


class GridPAACLearner(object):
    N_AGENTS = 10

    def __init__(self, network_creator, environment_creator, args, emulator_class=SwarmRunner, state_processor=None,
                 device=None, reward_indexing="reference", mask_terminals=False, use_cuda_graph=True,
                 compact_obs="auto", net_precision="fp32", bootstrap_truncated=False):
        self.args = args
        self.emulator_class = emulator_class
        self.max_local_steps = args.max_local_steps
        self.num_actions = args.num_actions
        self.initial_lr = args.initial_lr
        self.lr_annealing_steps = args.lr_annealing_steps
        self.max_global_steps = args.max_global_steps
        self.gamma = args.gamma
        self.clip_norm = args.clip_norm
        self.clip_norm_type = args.clip_norm_type
        self.reward_indexing = reward_indexing
        self.mask_terminals = mask_terminals
        if bootstrap_truncated and not mask_terminals:
            raise ValueError("bootstrap_truncated=True needs mask_terminals=True (without the mask every return already "
                             "runs on through the episode end)")
        self.bootstrap_truncated = bool(bootstrap_truncated)
        self.use_cuda_graph = use_cuda_graph
        # compact_obs: the net consumes (grid (E,G,G,2), positions (E,A,2)) through forward_compact -- exactly the
        # same function of the observation, without ever materialising the reference's (E,A,G,G,3) layout
        self._compact_request = compact_obs
        torch.backends.cudnn.benchmark = True       # fixed shapes: let cuDNN pick its fastest algorithms once
        # net_precision: "fp32" = true FP32 like the reference's TF graph (networks.py:165-167): TF32 is switched OFF for
        # cuDNN convolutions and cuBLAS matmuls (PyTorch leaves it on for convolutions by default); "tf32" lets both use
        # TF32 tensor cores; "bf16" runs forward/backward under autocast (FP32 master weights).  Process-wide switches.
        if net_precision not in ("fp32", "tf32", "bf16"):
            raise ValueError("net_precision must be fp32, tf32 or bf16")
        self.net_precision = net_precision
        torch.backends.cudnn.allow_tf32 = net_precision != "fp32"
        torch.backends.cuda.matmul.allow_tf32 = net_precision != "fp32"
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank() if self.world > 1 else 0
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())

        self.total_emulators = args.emulator_counts
        first, self.emulator_counts = sharding.shard_envs(self.total_emulators, self.world, self.rank)
        extra = dict(final_obs=True) if self.bootstrap_truncated else {}
        self.env = environment_creator.create_batched_environment(
            self.emulator_counts, seed=getattr(args, "random_seed", 3), env_id_offset=first, device=self.device, **extra)
        self.N_AGENTS = self.env.A
        self.real_batch_size = self.emulator_counts * self.N_AGENTS
        # "auto": the factorised path pays off once the policy batch is large enough to be bandwidth/FLOP bound
        # (measured: 1.64x at 1024 emulators/GPU, 0.93x at 32 where the update is launch-latency bound)
        self.compact_obs = (self.emulator_counts >= 128) if self._compact_request == "auto" else bool(self._compact_request)

        torch.manual_seed(getattr(args, "random_seed", 3))          # same initial weights on every rank
        self.network = network_creator().to(self.device)
        if self.world > 1:
            for p in self.network.parameters():
                dist.broadcast(p.data, src=0)
        torch.manual_seed(getattr(args, "random_seed", 3) + 7919 * (self.rank + 1))   # per-rank action noise

        # flat gradient buffer: every p.grad is a view into it, so the all-reduce and the norm are one op each
        params = [p for p in self.network.parameters()]
        self.flat_grad = torch.zeros(sum(p.numel() for p in params), dtype=torch.float32, device=self.device)
        off = 0
        for p in params:
            p.grad = self.flat_grad[off:off + p.numel()].view_as(p)
            off += p.numel()
        self.lr_t = torch.tensor(float(self.initial_lr), dtype=torch.float32, device=self.device)
        self.optimizer = torch.optim.Adam(params, lr=self.lr_t, betas=(0.9, 0.999), eps=1e-8, capturable=True,
                                          foreach=True)
        self.runners = GridRunners(self.env, workers=getattr(args, "emulator_workers", None), variables=None,
                                   emulator_class=emulator_class, coord=None, grid_size=self.env.G, expand=False)
        self.global_step = 0
        self.global_norm = torch.zeros((), device=self.device)
        self._graph = None
        self._alloc()

    # ------------------------------------------------------------------ buffers
    def _alloc(self):
        T, B, G, d = self.max_local_steps, self.real_batch_size, self.env.G, self.device
        E, A = self.emulator_counts, self.N_AGENTS
        # observation ring: slot t is the state the policy saw at step t, slot T the bootstrap state
        if self.compact_obs:
            self.states = None
            self.grids = torch.zeros(T + 1, E, G, G, 2, dtype=torch.float32, device=d)
            self.positions = torch.zeros(T + 1, E, A, 2, dtype=torch.uint8, device=d)
        else:
            self.states = torch.zeros(T + 1, E, A, G, G, 3, dtype=torch.float32, device=d)
        self.actions = torch.zeros(T, B, self.num_actions, dtype=torch.float32, device=d)
        self.values = torch.zeros(T, B, dtype=torch.float32, device=d)
        self.rewards = torch.zeros(T, B, dtype=torch.float32, device=d)
        self.not_over = torch.ones(T, B, dtype=torch.float32, device=d)
        self.y_batch = torch.zeros(T, B, dtype=torch.float32, device=d)
        self.adv_batch = torch.zeros(T, B, dtype=torch.float32, device=d)
        if self.bootstrap_truncated:
            # slot t: the terminal observation of the envs whose episode ended at step t (compact in both obs modes),
            # and the step's done split
            self.final_grids = torch.zeros(T, E, G, G, 2, dtype=torch.float32, device=d)
            self.final_positions = torch.zeros(T, E, A, 2, dtype=torch.uint8, device=d)
            self.terminated = torch.zeros(T, B, dtype=torch.float32, device=d)
            self.truncated = torch.zeros(T, B, dtype=torch.float32, device=d)
        # episode statistics, accumulated on the device (read back only when logging)
        self.episode_return = torch.zeros(E, dtype=torch.float32, device=d)
        self.finished_return_sum = torch.zeros((), dtype=torch.float64, device=d)
        self.finished_episodes = torch.zeros((), dtype=torch.int64, device=d)

    # ------------------------------------------------------------------ rollout
    @staticmethod
    def choose_next_actions(network, num_actions, states, histories=None, agent_positions=None, session=None):
        """paac.py:412-419."""
        out = network.predict(states)
        mu, sigma, v = out["mu"], out["sigma"], out["vs"]
        return mu + sigma * torch.randn_like(mu), v

    def _autocast(self):
        return torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.net_precision == "bf16")

    def _predict(self, t):
        with self._autocast():
            if self.compact_obs:
                out = self.network.predict_compact(self.grids[t], self.positions[t])
            else:
                out = self.network.predict(self.states[t].view(self.real_batch_size, *self.states.shape[3:]))
        return {k: v.float() for k, v in out.items()}

    def _rollout_step(self, t):
        E, A = self.emulator_counts, self.N_AGENTS
        out = self._predict(t)
        next_actions, v = out["mu"] + out["sigma"] * torch.randn_like(out["mu"]), out["vs"]      # paac.py:412-419
        next_actions = self.emulator_class.transform_actions_for_env(next_actions.contiguous())   # in place
        self.runners.actions.copy_(next_actions.view(E, A, self.num_actions))
        self.actions[t].copy_(next_actions)
        self.values[t].copy_(v)
        # one fused step launch + one expand launch, straight into the next ring slot
        fin = dict(final_grid_out=self.final_grids[t], final_positions_out=self.final_positions[t]) \
            if self.bootstrap_truncated else {}
        if self.compact_obs:
            self.runners.update_environments(grid_out=self.grids[t + 1], positions_out=self.positions[t + 1], **fin)
        else:
            self.runners.update_environments(states_out=self.states[t + 1], **fin)
        if self.bootstrap_truncated:
            self.terminated[t].copy_(self.env.terminated.to(torch.float32).repeat_interleave(A))
            self.truncated[t].copy_(self.env.truncated.to(torch.float32).repeat_interleave(A))
        reward, over = self.env.reward, self.env.done_u8
        if self.reward_indexing == "reference":
            self.rewards[t, :E].copy_(reward)                      # paac.py:338  rewards[t, e_idx], e_idx < E
        else:
            self.rewards[t].copy_(reward.repeat_interleave(A))
        self.not_over[t].copy_((1 - over.to(torch.float32)).repeat_interleave(A))
        self.episode_return += reward
        fin = over.to(torch.bool)
        self.finished_return_sum += (self.episode_return * fin).sum(dtype=torch.float64)
        self.finished_episodes += fin.sum()
        self.episode_return.masked_fill_(fin, 0.0)

    def _rollout(self):
        for t in range(self.max_local_steps):
            self._rollout_step(t)

    def _returns(self):
        T = self.max_local_steps
        ret = self._predict(T)["vs"].clone()                                # paac.py:351-358
        if self.bootstrap_truncated:
            # V of every terminal observation of the rollout in one forward (T E envs); weight 0 where no episode was
            # truncated (the slots of the other envs hold stale, finite observations)
            E, A = self.emulator_counts, self.N_AGENTS
            with self._autocast():
                v_fin = self.network.predict_compact(self.final_grids.view(T * E, *self.final_grids.shape[2:]),
                                                     self.final_positions.view(T * E, A, 2))["vs"].float()
            boot = v_fin.view(T, -1) * self.truncated * (1.0 - self.terminated)
        for t in reversed(range(T)):                                        # paac.py:362-365
            if self.bootstrap_truncated:
                ret = self.rewards[t] + self.gamma * (ret * self.not_over[t] + boot[t])
            else:
                ret = self.rewards[t] + self.gamma * ret * (self.not_over[t] if self.mask_terminals else 1.0)
            self.y_batch[t].copy_(ret)
            self.adv_batch[t].copy_(ret - self.values[t])

    # ------------------------------------------------------------------ update
    def _train_step(self):
        T, B = self.max_local_steps, self.real_batch_size
        E, A = self.emulator_counts, self.N_AGENTS
        if self.compact_obs:
            obs, pos = self.grids[:T].view(T * E, *self.grids.shape[2:]), self.positions[:T].view(T * E, A, 2)
        else:
            obs, pos = self.states[:T].view(T * B, *self.states.shape[3:]), None
        with self._autocast():
            out = self.network.losses(obs, self.actions.view(T * B, self.num_actions),
                                      self.adv_batch.view(-1) / self.network.scale, self.y_batch.view(-1), positions=pos)
        self.flat_grad.zero_()
        out["loss"].backward()
        sharding.allreduce_mean_(self.flat_grad)
        if self.clip_norm_type == "global":                      # tf.clip_by_global_norm (actor_learner.py:55-60)
            norm = torch.linalg.vector_norm(self.flat_grad)
            self.flat_grad *= self.clip_norm / torch.clamp(norm, min=self.clip_norm)
        elif self.clip_norm_type == "local":                     # tf.clip_by_norm per variable
            for p in self.network.parameters():
                n = torch.linalg.vector_norm(p.grad)
                p.grad *= self.clip_norm / torch.clamp(n, min=self.clip_norm)
            norm = torch.linalg.vector_norm(self.flat_grad)
        elif self.clip_norm_type == "ignore":
            norm = torch.linalg.vector_norm(self.flat_grad)
        else:
            raise Exception("Norm type not recognized")
        self.global_norm.copy_(norm)
        self.optimizer.step()
        return out

    def get_lr(self):
        """actor_learner.py:115-119."""
        if self.global_step <= self.lr_annealing_steps:
            return self.initial_lr - (self.global_step * self.initial_lr / self.lr_annealing_steps)
        return 0.0

    def _update_body(self):
        """T rollout steps, n-step returns, one optimiser step -- all enqueued on the current stream."""
        T = self.max_local_steps
        self._rollout()
        with torch.no_grad():
            self._returns()
        self._train_step()
        self._carry_over()

    def _obs_tensors(self):
        return (self.grids, self.positions) if self.compact_obs else (self.states,)

    def _carry_over(self):
        """The bootstrap state opens the next rollout."""
        for ring in self._obs_tensors():
            ring[0].copy_(ring[self.max_local_steps])

    def start(self):
        """Initial reset + first observation into ring slot 0 (paac.py:247-251)."""
        if self.compact_obs:
            self.runners.start()
            self.grids[0].copy_(self.env.grid)
            self.positions[0].copy_(self.env.positions)
        else:
            self.runners.start(states_out=self.states[0])

    def _capture(self):
        """Warm up on a side stream (cuDNN autotune, allocator, optimiser state) with lr = 0, undo the warm-up,
        then capture the whole update (rollout + returns + backward + all-reduce + Adam) as ONE CUDA graph."""
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        keep_t = self._obs_tensors() + (self.episode_return, self.finished_return_sum, self.finished_episodes)
        with torch.cuda.stream(s):
            sd = self.env.state_dict()
            keep = [t.clone() for t in keep_t]
            lr = self.lr_t.clone()
            self.lr_t.zero_()
            for _ in range(2):
                self._update_body()
            self.lr_t.copy_(lr)
            for st in self.optimizer.state.values():          # forget the warm-up moments and step counts
                for v in st.values():
                    if torch.is_tensor(v):
                        v.zero_()
            self.env.load_state_dict(sd)
            for dst, src in zip(keep_t, keep):
                dst.copy_(src)
        torch.cuda.current_stream(self.device).wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            self._update_body()
        self._graph = g        # capturing does not execute: state is untouched

    def update(self):
        """One PAAC update: T rollout steps for every emulator + one optimiser step.  All statistics stay on
        the device; the only host work is the learning-rate scalar."""
        self.global_step += self.max_local_steps * self.total_emulators
        self.lr_t.fill_(self.get_lr())                 # paac.py:373: the rate of the step count AFTER the rollout
        if self.use_cuda_graph:
            if self._graph is None:
                self._capture()
            self._graph.replay()
        else:
            self._update_body()

    def scalars(self):
        """The training scalars the reference writes as TF summaries: ``global_norm`` (actor_learner.py:83) and
        ``rl/reward`` = mean total reward of the episodes finished so far (paac.py:152-155, 384-395), plus the step
        count and learning rate.  One device->host read: call it when logging, not every update."""
        n = int(self.finished_episodes.item())
        return {"global_step": int(self.global_step), "global_norm": float(self.global_norm.item()),
                "rl/reward": float(self.finished_return_sum.item()) / n if n else 0.0, "rl/episodes": n,
                "learning_rate": float(self.get_lr())}

    def train(self, max_updates=None, log_every=None, monitor=None, eval_every=30.0, summary_dir=None):
        """paac.py:226-406 without the TF session.  ``monitor``: a SwarmPolicyMonitor evaluated every
        ``eval_every`` seconds (the reference does this from a thread, paac.py:277-282; here between updates,
        on rank 0).  ``summary_dir``: where rank 0 appends scalars() as JSON lines (``summaries.jsonl``) at every
        log point -- the stand-in for the reference's TF summary writer.  Returns the mean frames/s."""
        import json
        import os
        self.start()
        summary_f = None
        if summary_dir is not None and self.rank == 0:
            os.makedirs(summary_dir, exist_ok=True)
            summary_f = open(os.path.join(summary_dir, "summaries.jsonl"), "a")
        counter, start = 0, time.time()
        log_every = log_every or max(1, int(5048 / self.total_emulators))
        global_step_start = self.global_step
        loop_start = time.time()
        last_eval = time.time()
        while self.global_step < self.max_global_steps and (max_updates is None or counter < max_updates):
            self.update()
            counter += 1
            if monitor is not None and self.rank == 0 and time.time() - last_eval >= eval_every:
                torch.cuda.synchronize(self.device)
                monitor.eval_once(global_step=self.global_step)
                last_eval = time.time()
            if counter % log_every == 0 and self.rank == 0:
                torch.cuda.synchronize(self.device)
                now = time.time()
                sc = self.scalars()
                avg = sc["rl/reward"]
                if summary_f is not None:
                    summary_f.write(json.dumps(sc) + "\n")
                    summary_f.flush()
                logging.info("Ran %d steps, at %.1f steps/s (%.1f steps/s avg), mean finished-episode reward %.3f, "
                             "grad norm %.3f", self.global_step,
                             log_every * self.max_local_steps * self.total_emulators / (now - loop_start),
                             (self.global_step - global_step_start) / (now - start), avg, float(self.global_norm.item()))
                loop_start = now
        torch.cuda.synchronize(self.device)
        if summary_f is not None:
            summary_f.write(json.dumps(self.scalars()) + "\n")
            summary_f.close()
        return (self.global_step - global_step_start) / max(time.time() - start, 1e-9)

    def cleanup(self):
        self.runners.stop()
