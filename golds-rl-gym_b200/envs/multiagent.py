"""Host-side mirror of fed_gym/envs/multiagent.py (reference :7-115) on top of the C ABI.

``BatchedSwarmEnv``  E independent swarm envs resident on one GPU; reset()/step() enqueue
                     kernels on the current torch stream and never synchronise.
``SwarmEnv``         the reference's single-env gym surface (numpy in / numpy out, same class
                     constants, same global-numpy-RNG draw order) as an E=1 view of the above.

No arithmetic happens in Python: every call below is one C-ABI entry point of
libswarm_b200.so (include/swarm_b200.h).  There is no CPU fallback.
"""
import ctypes

import numpy as np
import torch

from .. import _native as nat


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class _on(object):
    """Make ``device`` the current CUDA device around a ctypes call (the C side launches on the CURRENT device;
    the torch ops carry their own CUDAGuard).  Free when it already is."""
    __slots__ = ("idx", "prev")

    def __init__(self, device):
        self.idx = device.index if device.index is not None else torch.cuda.current_device()

    def __enter__(self):
        self.prev = torch.cuda.current_device()
        if self.prev != self.idx:
            torch.cuda.set_device(self.idx)

    def __exit__(self, *exc):
        if self.prev != self.idx:
            torch.cuda.set_device(self.prev)
        return False


class InjectedDraws(object):
    """Device copies of one reset's random draws for the whole batch (SwarmInjectedDraws)."""

    def __init__(self, x0, xa0, burn_actions, agent_noise, particle_noise, device):
        def dev(a):
            return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(device) \
                if not torch.is_tensor(a) else a.to(device=device, dtype=torch.float64).contiguous()

        self.x0, self.xa0, self.burn_actions = dev(x0), dev(xa0), dev(burn_actions)
        self.agent_noise, self.particle_noise = dev(agent_noise), dev(particle_noise)
        self.c = nat.SwarmInjectedDraws(_ptr(self.x0), _ptr(self.xa0), _ptr(self.burn_actions),
                                        _ptr(self.agent_noise), _ptr(self.particle_noise))

    def tensors(self):
        return [self.x0, self.xa0, self.burn_actions, self.agent_noise, self.particle_noise]

    def check(self, E, N, A, nb):
        want = [(E, N, 2), (E, A, 2), (E, nb, A, 2), (E, nb + 1, A, 2), (E, nb + 1, N, 2)]
        got = [tuple(t.shape) for t in (self.x0, self.xa0, self.burn_actions, self.agent_noise, self.particle_noise)]
        if want != got:
            raise ValueError("injected draws have shapes %s, expected %s" % (got, want))


class BatchedSwarmEnv(object):
    """E swarm envs on one GPU.  State tensors are owned here and updated in place by the kernels
    (like the reference, whose returned arrays alias its internal state, multiagent.py:42-44).

    reset() -> (x (E,N,2) f64, xa (E,A,2) f64)
    step(actions (E,A,2)) -> ((x, xa), reward (E,) f32, done (E,) bool, {})
    With ``rasterize=True`` (default) the step kernel also writes ``self.grid`` (E,G,G,2) f32 and
    ``self.positions`` (E,A,2) u8 -- SwarmStateProcessor.process_state of the returned state.
    With ``auto_reset=True`` finished envs are reset inside the step (SwarmRunner._run semantics).
    With ``noise="fresh"`` every step draws the next row of the episode's noise tables (the reference with
    SURVEY Q1 fixed) instead of re-using row N_BURN_IN; the default ``"frozen"`` is the reference as it is.
    With ``final_obs=True`` step() also keeps what the auto-reset overwrites (swarm_step_final) and returns it as the info
    dict: ``terminated`` (reward >= 0) and ``truncated`` (TimeLimit) as (E,) bool, and for the envs that are done the
    terminal state ``final_x`` / ``final_xa`` and, when rasterising, its observation ``final_grid`` / ``final_positions``
    (the rows of the other envs keep their old bytes).  They alias buffers of the env, like reward and done.
    With ``physics`` every env has its own noise, gravity, wind, F, L and dt: row e of ``self.physics`` (E,6) f64, columns
    ``_native.PHYSICS_COLUMNS`` (SwarmPhysics).  ``"table"`` fills it from the class constants and leaves it to the
    caller, who may write rows between calls; a dict of per-column ranges such as ``{"F": (0.3, 0.7), "L": (5, 15)}``
    draws each env's row anew, uniformly, at every reset of that env (explicit or auto-reset), inside the kernels.
    """

    # fed_gym/envs/multiagent.py:8-21
    N_LOCUSTS = 80
    N_AGENTS = 10
    NOISE = 0.0001
    GRAVITY = -1
    WIND_SPEED = 1
    F = 0.5
    L = 10
    dt = 0.05
    N_BURN_IN = 10

    def __init__(self, num_envs, n_locusts=None, n_agents=None, grid_size=84, max_episode_steps=128,
                 seed=0, env_id_offset=0, device=None, math_mode="fast", auto_reset=True, rasterize=True,
                 binding="torch", tuning=0, noise="frozen", cluster=None, final_obs=False, physics=None):
        """binding: "torch" = the hot calls go through torch.ops.swarm_b200.* (the C ABI as a PyTorch
        extension, csrc/torch_binding.cpp), "ctypes" = straight into the C ABI.  Same kernels either way.
        tuning: SwarmParams.tuning (0 = automatic launch shape; anything else only changes speed, never bits).
        noise: "frozen" (the reference: every step after a reset re-uses noise row N_BURN_IN) or "fresh" (step k of
        an episode uses row N_BURN_IN + k, drawn by Philox inside the step kernel; SWARM_STEP_FRESH_NOISE).
        cluster: None = one CTA per env up to 2048 locusts and a thread-block cluster of the library's size above; an
        integer K = a cluster of K CTAs per env (1..16, for 512 < n_locusts <= 8192; bitwise the same results).
        physics: None (every env uses the class constants), "table" (per-env rows in self.physics, written by the caller)
        or a dict {column: (lo, hi)} (per-env rows redrawn at every reset; unnamed columns stay at the class constant)."""
        self.lib = nat.load()
        if binding not in ("torch", "ctypes"):
            raise ValueError("binding must be 'torch' or 'ctypes'")
        if noise not in ("frozen", "fresh"):
            raise ValueError("noise must be 'frozen' or 'fresh'")
        self.noise = noise
        self._noise_flag = nat.SWARM_STEP_FRESH_NOISE if noise == "fresh" else 0
        self.ops = nat.load_torch_ops() if binding == "torch" else None
        if not torch.cuda.is_available():
            raise nat.SwarmNativeError("BatchedSwarmEnv needs a CUDA device (sm_100a); there is no CPU path")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.E = int(num_envs)
        self.N = int(n_locusts if n_locusts is not None else self.N_LOCUSTS)
        self.A = int(n_agents if n_agents is not None else self.N_AGENTS)
        self.G = int(grid_size)
        tuning = int(tuning)
        if cluster is not None:
            tuning |= nat.tune_cluster(int(cluster))
        elif self.N > nat.MAX_LOCUSTS_ONE_CTA and not tuning & nat.TUNE_CLUSTER_MASK:
            tuning |= nat.TUNE_CLUSTER_AUTO
        self.auto_reset = bool(auto_reset)
        self.rasterize = bool(rasterize)
        self.params = nat.SwarmParams(
            n_envs=self.E, n_locusts=self.N, n_agents=self.A, grid_size=self.G, n_burn_in=self.N_BURN_IN,
            max_episode_steps=int(max_episode_steps), math_mode={"fast": 0, "precise": 1}[math_mode], tuning=tuning,
            noise=self.NOISE, gravity=self.GRAVITY, wind=self.WIND_SPEED, F=self.F, L=self.L, dt=self.dt,
            box_width=3.0, box_height=3.0, seed=int(seed) & (2 ** 64 - 1), env_id_offset=int(env_id_offset))
        nat.check(self.lib.swarm_validate(ctypes.byref(self.params)), "swarm_validate")
        E, N, A, G, d = self.E, self.N, self.A, self.G, self.device
        f64 = torch.float64
        self.x = torch.zeros(E, N, 2, dtype=f64, device=d)
        self.xa = torch.zeros(E, A, 2, dtype=f64, device=d)
        self.noise_x = torch.zeros(E, N, 2, dtype=f64, device=d)
        self.noise_a = torch.zeros(E, A, 2, dtype=f64, device=d)
        self.elapsed = torch.zeros(E, dtype=torch.int32, device=d)
        self.episode = torch.zeros(E, dtype=torch.int32, device=d)      # uint32 on the device side
        self.work = torch.zeros(2 + E, dtype=torch.int32, device=d)     # swarm_step's scratch: queue + per-env ready flags
        self.actions = torch.zeros(E, A, 2, dtype=torch.float32, device=d)
        self.reward = torch.zeros(E, dtype=torch.float32, device=d)
        self.done_u8 = torch.zeros(E, dtype=torch.uint8, device=d)
        self.grid = torch.zeros(E, G, G, 2, dtype=torch.float32, device=d)
        self.positions = torch.zeros(E, A, 2, dtype=torch.uint8, device=d)
        self.state_c = nat.SwarmState(_ptr(self.x), _ptr(self.xa), _ptr(self.noise_x), _ptr(self.noise_a),
                                      _ptr(self.elapsed), _ptr(self.episode), _ptr(self.work), self.work.numel())
        self._io = nat.SwarmStepIO()
        self._io.reward, self._io.done = self.reward.data_ptr(), self.done_u8.data_ptr()
        self._grid_ptr, self._pos_ptr = self.grid.data_ptr(), self.positions.data_ptr()
        self._params_ref, self._state_ref, self._io_ref = (ctypes.byref(self.params), ctypes.byref(self.state_c),
                                                           ctypes.byref(self._io))
        self._done_view = self.done_u8.view(torch.bool)
        self._io_host = None
        self._was_reset = False
        self._blob_bytes, self._blob_t = None, None
        self._ctx = _on(self.device)
        self.final_obs = bool(final_obs)
        self.final_x = self.final_xa = self.terminated = self.truncated = None
        self.final_grid = self.final_positions = None
        if self.final_obs:
            self.final_x = torch.zeros(E, N, 2, dtype=f64, device=d)
            self.final_xa = torch.zeros(E, A, 2, dtype=f64, device=d)
            self.terminated = torch.zeros(E, dtype=torch.uint8, device=d)
            self.truncated = torch.zeros(E, dtype=torch.uint8, device=d)
            if self.rasterize:
                self.final_grid = torch.zeros(E, G, G, 2, dtype=torch.float32, device=d)
                self.final_positions = torch.zeros(E, A, 2, dtype=torch.uint8, device=d)
            self._fin = nat.SwarmStepFinal(_ptr(self.final_x), _ptr(self.final_xa), _ptr(self.terminated),
                                           _ptr(self.truncated), None, None)
            self._fin_ref = ctypes.byref(self._fin)
        self._init_physics(physics)
        self.refresh_params()

    def _init_physics(self, physics):
        self.physics = None
        if physics is None:
            return
        fixed = [float(getattr(self.params, c)) for c in nat.PHYSICS_COLUMNS]
        lo, hi, flags = list(fixed), list(fixed), 0
        if isinstance(physics, dict):
            for name, rng in physics.items():
                if name not in nat.PHYSICS_COLUMNS:
                    raise ValueError("unknown physics column %r (columns: %s)" % (name, ", ".join(nat.PHYSICS_COLUMNS)))
                c = nat.PHYSICS_COLUMNS.index(name)
                lo[c], hi[c] = float(rng[0]), float(rng[1])
            flags = nat.SWARM_PHYSICS_RESAMPLE
        elif physics != "table":
            raise ValueError("physics must be None, 'table' or a dict {column: (lo, hi)}")
        self.physics = torch.tensor([fixed] * self.E, dtype=torch.float64, device=self.device)
        self._phys_flags, self._phys_lo, self._phys_hi = flags, lo, hi
        self._phys_c = nat.SwarmPhysics(self.physics.data_ptr(), flags, 0, (ctypes.c_double * 6)(*lo),
                                        (ctypes.c_double * 6)(*hi))
        self._phys_ref = ctypes.byref(self._phys_c)

    def _phys_args(self):
        return self.physics, self._phys_flags, self._phys_lo, self._phys_hi

    def refresh_params(self):
        self._state_t = (self.x, self.xa, self.noise_x, self.noise_a, self.elapsed, self.episode, self.work)

    @property
    def _blob(self):
        """self.params (which callers may mutate, like the reference's class constants) packed for the torch ops;
        the CPU tensor is rebuilt only when the struct's bytes changed."""
        b = bytes(self.params)
        if b != self._blob_bytes:
            self._blob_bytes, self._blob_t = b, nat.params_blob(self.params)
        return self._blob_t

    # ------------------------------------------------------------------ gym surface
    def reset(self, mask=None, draws=None):
        """SwarmEnv._reset for every env (or those with mask != 0).  draws: InjectedDraws or None
        (None -> device Philox keyed by (seed, global env id, episode))."""
        m = None
        if mask is not None:
            m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        if draws is not None:
            draws.check(self.E, self.N, self.A, self.N_BURN_IN)
        if self.ops is not None:
            dts = draws.tensors() if draws is not None else []
            with torch.cuda.device(self.device):
                if self.physics is not None:
                    self.ops.reset_physics(self._blob, *self._state_t[:6], m, dts, *self._phys_args())
                else:
                    self.ops.reset(self._blob, *self._state_t[:6], m, dts)
            self._was_reset = True
            return self.x, self.xa
        with self._ctx:
            dr = ctypes.byref(draws.c) if draws is not None else None
            if self.physics is not None:
                nat.check(self.lib.swarm_reset_physics(ctypes.byref(self.params), ctypes.byref(self.state_c),
                                                       self._phys_ref, _ptr(m), dr, _stream(self.device)),
                          "swarm_reset_physics")
            else:
                nat.check(self.lib.swarm_reset(ctypes.byref(self.params), ctypes.byref(self.state_c), _ptr(m), dr,
                                               _stream(self.device)), "swarm_reset")
        self._was_reset = True
        return self.x, self.xa

    def step(self, actions, noise_a=None, noise_x=None, clip=False, reset_draws=None, v_out=None,
             rasterize=None, auto_reset=None, grid_out=None, positions_out=None, add_wind=True,
             final_grid_out=None, final_positions_out=None):
        """One env step for the whole batch; a single kernel launch.

        actions: (E,A,2) float32 or float64 CUDA tensor (float32 is the PAAC shared_actions dtype).
        With clip=True actions with |a|>=1 are normalised IN PLACE first (transform_actions_for_env).
        grid_out / positions_out: optional (E,G,G,2) f32 / (E,A,2) u8 tensors that receive the observation
        instead of self.grid / self.positions (e.g. a slot of a rollout ring).
        final_grid_out / final_positions_out: the same for the terminal observation (final_obs=True).
        With final_obs=True the 4th element is the info dict of the terminal outputs (see the class), else {}.
        """
        if not self._was_reset:
            # the reference raises TypeError unpacking self.states=None (multiagent.py:31)
            raise TypeError("step() called before reset()")
        if actions.device != self.device or not actions.is_contiguous() or tuple(actions.shape) != (self.E, self.A, 2):
            raise ValueError("actions must be a contiguous (%d,%d,2) tensor on %s" % (self.E, self.A, self.device))
        rasterize = self.rasterize if rasterize is None else rasterize
        auto_reset = self.auto_reset if auto_reset is None else auto_reset
        flags = (nat.SWARM_STEP_AUTO_RESET if auto_reset else 0) | (nat.SWARM_STEP_CLIP_ACTIONS if clip else 0) | \
                (0 if add_wind else nat.SWARM_STEP_NO_ACTION_WIND) | self._noise_flag
        if self.ops is not None:
            if actions.dtype not in (torch.float32, torch.float64):
                raise ValueError("actions must be float32 or float64")
            g_t = (grid_out if grid_out is not None else self.grid) if rasterize else None
            p_t = (positions_out if positions_out is not None else self.positions) if rasterize else None
            if self.physics is not None:
                dts = reset_draws.tensors() if reset_draws is not None else []
                fin = [None] * 6
                if self.final_obs:
                    fg, fp = self._final_obs_bufs(rasterize, final_grid_out, final_positions_out)
                    fin = [self.final_x, self.final_xa, self.terminated, self.truncated, fg, fp]
                self.ops.step_physics(self._blob, *self._state_t, actions, noise_a, noise_x, self.reward, self.done_u8,
                                      g_t, p_t, v_out, flags, dts, *self._phys_args(), *fin)
                info = self._info(fin[4], fin[5]) if self.final_obs else {}
                return (self.x, self.xa), self.reward, self._done_view, info
            if self.final_obs:
                fg, fp = self._final_obs_bufs(rasterize, final_grid_out, final_positions_out)
                self.ops.step_final(self._blob, *self._state_t, actions, noise_a, noise_x, self.reward, self.done_u8,
                                    g_t, p_t, v_out, flags,
                                    reset_draws.tensors() if reset_draws is not None else [],
                                    self.final_x, self.final_xa, self.terminated, self.truncated, fg, fp)
                return (self.x, self.xa), self.reward, self._done_view, self._info(fg, fp)
            self.ops.step(self._blob, *self._state_t, actions, noise_a, noise_x, self.reward, self.done_u8,
                          g_t, p_t, v_out, flags,
                          reset_draws.tensors() if reset_draws is not None else [])
            return (self.x, self.xa), self.reward, self._done_view, {}
        io = self._io                      # one persistent SwarmStepIO; only the per-call fields change
        if actions.dtype == torch.float32:
            io.actions_f32, io.actions_f64 = actions.data_ptr(), None
        elif actions.dtype == torch.float64:
            io.actions_f32, io.actions_f64 = None, actions.data_ptr()
            flags |= nat.SWARM_STEP_ACTIONS_F64
        else:
            raise ValueError("actions must be float32 or float64")
        io.noise_a = noise_a.data_ptr() if noise_a is not None else None
        io.noise_x = noise_x.data_ptr() if noise_x is not None else None
        if rasterize:
            io.grid = grid_out.data_ptr() if grid_out is not None else self._grid_ptr
            io.positions = positions_out.data_ptr() if positions_out is not None else self._pos_ptr
        else:
            io.grid, io.positions = None, None
        io.v_out = v_out.data_ptr() if v_out is not None else None
        io.flags = flags
        if self.physics is not None:
            fin_ref, info = None, {}
            if self.final_obs:
                fg, fp = self._final_obs_bufs(rasterize, final_grid_out, final_positions_out)
                self._fin.grid, self._fin.positions = _ptr(fg), _ptr(fp)
                fin_ref, info = self._fin_ref, self._info(fg, fp)
            with self._ctx:
                rc = self.lib.swarm_step_physics(self._params_ref, self._state_ref, self._io_ref, fin_ref, self._phys_ref,
                                                 ctypes.byref(reset_draws.c) if reset_draws is not None else None,
                                                 torch.cuda.current_stream(self.device).cuda_stream)
            if rc:
                nat.check(rc, "swarm_step_physics")
            return (self.x, self.xa), self.reward, self._done_view, info
        if self.final_obs:
            fg, fp = self._final_obs_bufs(rasterize, final_grid_out, final_positions_out)
            self._fin.grid, self._fin.positions = _ptr(fg), _ptr(fp)
            with self._ctx:
                rc = self.lib.swarm_step_final(self._params_ref, self._state_ref, self._io_ref, self._fin_ref,
                                               ctypes.byref(reset_draws.c) if reset_draws is not None else None,
                                               torch.cuda.current_stream(self.device).cuda_stream)
            if rc:
                nat.check(rc, "swarm_step_final")
            return (self.x, self.xa), self.reward, self._done_view, self._info(fg, fp)
        with self._ctx:
            rc = self.lib.swarm_step(self._params_ref, self._state_ref, self._io_ref,
                                     ctypes.byref(reset_draws.c) if reset_draws is not None else None,
                                     torch.cuda.current_stream(self.device).cuda_stream)
        if rc:
            nat.check(rc, "swarm_step")
        return (self.x, self.xa), self.reward, self._done_view, {}

    def _final_obs_bufs(self, rasterize, grid_out, positions_out):
        """The terminal observation's targets of one step: the overrides, else the env's own buffers (None, None when the
        step does not rasterise)."""
        if not rasterize:
            return None, None
        E, A, G = self.E, self.A, self.G
        if self.final_grid is None and (grid_out is None or positions_out is None):      # built with rasterize=False
            self.final_grid = torch.zeros(E, G, G, 2, dtype=torch.float32, device=self.device)
            self.final_positions = torch.zeros(E, A, 2, dtype=torch.uint8, device=self.device)
        fg = grid_out if grid_out is not None else self.final_grid
        fp = positions_out if positions_out is not None else self.final_positions
        for t, shape, dt, name in ((fg, (E, G, G, 2), torch.float32, "final_grid_out"),
                                   (fp, (E, A, 2), torch.uint8, "final_positions_out")):
            if t.device != self.device or t.dtype != dt or not t.is_contiguous() or tuple(t.shape) != shape:
                raise ValueError("%s must be a contiguous %s tensor of shape %s on %s" % (name, dt, shape, self.device))
        return fg, fp

    def _info(self, fg, fp):
        return {"terminated": self.terminated.view(torch.bool), "truncated": self.truncated.view(torch.bool),
                "final_x": self.final_x, "final_xa": self.final_xa, "final_grid": fg, "final_positions": fp}

    def stagger_episodes(self, total_envs=None):
        """Opt-in de-synchronisation of the episode boundaries (NOT the reference's behaviour: there every emulator starts
        at elapsed = 0 and all of them hit TimeLimit(128) on the same step, emulator_runner.py:126-132, so every 128th
        batch-step carries the 10 burn-in steps of EVERY env).  Sets env e's TimeLimit counter to
        (global_id * max_episode_steps) // total_envs: from then on E/128 envs end their episode on each step -- their
        first episode is shorter, everything else is unchanged.  Call right after reset()."""
        lim = int(self.params.max_episode_steps)
        if lim <= 0:
            raise ValueError("stagger_episodes needs a TimeLimit (max_episode_steps > 0)")
        total = int(total_envs) if total_envs is not None else self.E
        ids = torch.arange(self.E, device=self.device, dtype=torch.int64) + int(self.params.env_id_offset)
        self.elapsed.copy_(((ids * lim) // max(total, 1) % lim).to(torch.int32))
        return self.elapsed

    def plan(self, rasterize=None):
        """swarm_step_plan: the launch shape step() uses for this batch, as a dict."""
        io = nat.SwarmStepIO()
        io.actions_f32 = self.actions.data_ptr()
        io.reward, io.done = self.reward.data_ptr(), self.done_u8.data_ptr()
        if self.rasterize if rasterize is None else rasterize:
            io.grid, io.positions = self._grid_ptr, self._pos_ptr
        io.flags = nat.SWARM_STEP_AUTO_RESET if self.auto_reset else 0
        out = (ctypes.c_int32 * 8)()
        with self._ctx:
            if self.physics is not None:
                nat.check(self.lib.swarm_step_plan_physics(self._params_ref, self._state_ref, ctypes.byref(io),
                                                           self._phys_ref, out), "swarm_step_plan_physics")
            else:
                nat.check(self.lib.swarm_step_plan(self._params_ref, self._state_ref, ctypes.byref(io), out),
                          "swarm_step_plan")
        keys = ("force_mode", "filler_warp", "raster_place", "threads", "ctas", "smem_bytes", "follower_ctas", "launches")
        d = dict(zip(keys, list(out)))
        cluster = d["raster_place"] == 4
        d["raster_place"] = ("none", "follower kernel", "raster warps in k_step", "k_step's own threads",
                             "the env's cluster")[d["raster_place"]]
        d["layout"] = "cluster" if cluster else "one CTA per env"
        d["cluster_size"] = d["follower_ctas"] if cluster else 1      # out[6] holds K in the cluster layout
        if cluster:
            d["follower_ctas"] = 0
        return d

    # ------------------------------------------------------------------ host-buffer (end-to-end) form
    def step_host(self, host_actions, host_reward, host_done, host_grid=None, host_positions=None):
        """swarm_step_host: actions come from / reward+done go to HOST tensors; the observation stays in HBM
        for the device-resident policy unless host_grid / host_positions are given (then it is also copied back:
        the numpy-out case of the reference's process_state).  Synchronises the stream.  Pinned tensors are read /
        written by the kernel itself over PCIe (zero-copy); self.reward / self.done_u8 are then NOT updated.
        Not available with per-env physics (swarm_step_host takes no SwarmPhysics)."""
        if self.physics is not None:
            raise ValueError("step_host has no per-env physics (swarm_step_host takes no SwarmPhysics); use step()")
        io = self._io_host
        if io is None:
            io = self._io_host = nat.SwarmStepIO()
            io.actions_f32 = self.actions.data_ptr()
            io.reward, io.done = self.reward.data_ptr(), self.done_u8.data_ptr()
            self._io_host_ref = ctypes.byref(io)
        io.grid, io.positions = (self._grid_ptr, self._pos_ptr) if self.rasterize else (None, None)
        io.flags = (nat.SWARM_STEP_AUTO_RESET if self.auto_reset else 0) | self._noise_flag
        with self._ctx:
            rc = self.lib.swarm_step_host(self._params_ref, self._state_ref, self._io_host_ref, host_actions.data_ptr(),
                                          host_reward.data_ptr(), host_done.data_ptr(),
                                          host_grid.data_ptr() if host_grid is not None else None,
                                          host_positions.data_ptr() if host_positions is not None else None,
                                          torch.cuda.current_stream(self.device).cuda_stream)
        if rc:
            nat.check(rc, "swarm_step_host")
        return host_reward, host_done

    # ------------------------------------------------------------------ observation
    def observe(self, box=None):
        """SwarmStateProcessor.process_state of the current state -> (grid, positions)."""
        if self.ops is not None:
            self.ops.rasterize(self._blob, self.x, self.xa, self.grid, self.positions, box)
            return self.grid, self.positions
        with self._ctx:
            nat.check(self.lib.swarm_rasterize(ctypes.byref(self.params), _ptr(self.x), _ptr(self.xa), _ptr(self.grid),
                                               _ptr(self.positions), _ptr(box), _stream(self.device)), "swarm_rasterize")
        return self.grid, self.positions

    def local_states(self, out=None):
        """SwarmRunner.get_local_states for the batch: (E,A,G,G,3) f32 from self.grid/positions."""
        if out is None:
            out = torch.empty(self.E, self.A, self.G, self.G, 3, dtype=torch.float32, device=self.device)
        if self.ops is not None:
            self.ops.expand_obs(self._blob, self.grid, self.positions, out)
            return out
        with self._ctx:
            nat.check(self.lib.swarm_expand_obs(ctypes.byref(self.params), _ptr(self.grid), _ptr(self.positions),
                                                _ptr(out), _stream(self.device)), "swarm_expand_obs")
        return out

    def forces(self, x=None, xa=None, v=None, reward=None):
        """SwarmEnv.v_calculate for the batch -> (v (E,N,2) f32, reward (E,) f32)."""
        x = self.x if x is None else x
        xa = self.xa if xa is None else xa
        if v is None:
            v = torch.empty(self.E, self.N, 2, dtype=torch.float32, device=self.device)
        if reward is None:
            reward = torch.empty(self.E, dtype=torch.float32, device=self.device)
        if self.ops is not None:
            if self.physics is not None:
                self.ops.forces_physics(self._blob, x, xa, v, reward, *self._phys_args())
            else:
                self.ops.forces(self._blob, x, xa, v, reward)
            return v, reward
        if self.physics is not None:
            with self._ctx:
                nat.check(self.lib.swarm_forces_physics(ctypes.byref(self.params), self._phys_ref, _ptr(x), _ptr(xa),
                                                        _ptr(v), _ptr(reward), _stream(self.device)),
                          "swarm_forces_physics")
            return v, reward
        with self._ctx:
            nat.check(self.lib.swarm_forces(ctypes.byref(self.params), _ptr(x), _ptr(xa), _ptr(v), _ptr(reward),
                                            _stream(self.device)), "swarm_forces")
        return v, reward

    def philox_draws(self):
        """The draws the NEXT Philox reset of every env will use, as an InjectedDraws."""
        E, N, A, nb, d = self.E, self.N, self.A, self.N_BURN_IN, self.device
        f64 = torch.float64
        bufs = [torch.empty(E, N, 2, dtype=f64, device=d), torch.empty(E, A, 2, dtype=f64, device=d),
                torch.empty(E, nb, A, 2, dtype=f64, device=d), torch.empty(E, nb + 1, A, 2, dtype=f64, device=d),
                torch.empty(E, nb + 1, N, 2, dtype=f64, device=d)]
        with self._ctx:
            nat.check(self.lib.swarm_philox_draws(ctypes.byref(self.params), ctypes.byref(self.state_c),
                                                  *[_ptr(b) for b in bufs], _stream(self.device)), "swarm_philox_draws")
        return InjectedDraws(*bufs, device=d)

    def philox_noise_rows(self, row0, n_rows):
        """Rows row0 .. row0+n_rows-1 of every env's CURRENT episode's noise tables, as drawn by Philox ->
        (agent_noise (E,n_rows,A,2), particle_noise (E,n_rows,N,2)) f64, unscaled.  Row N_BURN_IN + k is what step k
        of the episode uses with noise="fresh"; rows 0..N_BURN_IN are the ones its reset used."""
        E, N, A, d = self.E, self.N, self.A, self.device
        an = torch.empty(E, int(n_rows), A, 2, dtype=torch.float64, device=d)
        pn = torch.empty(E, int(n_rows), N, 2, dtype=torch.float64, device=d)
        with self._ctx:
            nat.check(self.lib.swarm_philox_noise_rows(ctypes.byref(self.params), ctypes.byref(self.state_c), int(row0),
                                                       int(n_rows), _ptr(an), _ptr(pn), _stream(self.device)),
                      "swarm_philox_noise_rows")
        return an, pn

    # ------------------------------------------------------------------ checkpointing
    def state_dict(self):
        keys = ("x", "xa", "noise_x", "noise_a", "elapsed", "episode") + (("physics",) if self.physics is not None else ())
        return {k: getattr(self, k).clone() for k in keys}

    def load_state_dict(self, sd):
        for k, v in sd.items():
            getattr(self, k).copy_(v)
        self._was_reset = True


class SwarmEnv(object):
    """Drop-in for the reference ``SwarmEnv`` (multiagent.py:7-115): numpy in, numpy out, E=1.

    Like the reference it draws from the GLOBAL numpy RNG in the reference's order
    (multiagent.py:48-56), so ``SwarmEnv(seed=s)`` sees the very same random numbers as the
    reference env -- they are injected into the device reset.  The raw class has no TimeLimit;
    ``make('Swarm-v0')`` adds the 128-step limit the gym registry attaches.
    With ``fresh_noise=True`` it is the reference with SURVEY Q1 fixed: ``self.t`` advances after every step, so
    step k of an episode uses row N_BURN_IN + k of the 138-row noise tables (and step 129 without a TimeLimit
    raises IndexError, as the fixed reference would).
    """
    N_LOCUSTS = 80
    N_AGENTS = 10
    GRID_SIZE = 40
    NOISE = 0.0001
    GRAVITY = -1
    WIND_SPEED = 1
    F = 0.5
    L = 10
    dt = 0.05
    N_BURN_IN = 10

    def __init__(self, seed=None, max_episode_steps=0, math_mode="fast", device=None, fresh_noise=False):
        self.n_seed = seed
        self.states = None
        self.t = 0
        self._max_episode_steps = max_episode_steps
        self._math_mode = math_mode
        self._device = device
        self._fresh = bool(fresh_noise)
        self._tables = None              # fresh noise: the episode's (138,1,A,2) / (138,1,N,2) noise tables on the device
        self._env = None

    def _backend(self):
        if self._env is None or self._env.N != self.N_LOCUSTS or self._env.A != self.N_AGENTS:
            self._env = BatchedSwarmEnv(1, n_locusts=self.N_LOCUSTS, n_agents=self.N_AGENTS, grid_size=84,
                                        max_episode_steps=self._max_episode_steps, device=self._device,
                                        math_mode=self._math_mode, auto_reset=False, rasterize=False,
                                        noise="fresh" if self._fresh else "frozen")
            for k in ("NOISE", "GRAVITY", "WIND_SPEED", "F", "L", "dt"):
                setattr(self._env.params, {"NOISE": "noise", "GRAVITY": "gravity", "WIND_SPEED": "wind",
                                           "F": "F", "L": "L", "dt": "dt"}[k], float(getattr(self, k)))
            self._env.params.n_burn_in = self.N_BURN_IN
            self._env.N_BURN_IN = self.N_BURN_IN
            self._env.refresh_params()
        return self._env

    def _sync_out(self):
        env = self._env
        x = env.x[0].cpu().numpy()
        xa = env.xa[0].cpu().numpy()
        if self.states is None:
            self.states = [x, xa]
        else:                       # the reference mutates its state arrays in place
            self.states[0][...] = x
            self.states[1][...] = xa
        return self.states

    def reset(self):
        return self._reset()

    def step(self, v_action):
        return self._step(v_action)

    def _reset(self):
        env = self._backend()
        if self.n_seed:
            np.random.seed(self.n_seed)
        N, A, nb = self.N_LOCUSTS, self.N_AGENTS, self.N_BURN_IN
        x0 = np.random.rand(N, 2)
        xa0 = np.random.rand(A, 2)
        burn = np.random.normal(size=(nb, A, 2))
        an = np.random.normal(size=(128 + nb, A, 2))
        pn = np.random.normal(size=(128 + nb, N, 2))
        draws = InjectedDraws(x0[None], xa0[None], burn[None], an[None, :nb + 1], pn[None, :nb + 1], env.device)
        env.reset(draws=draws)
        if self._fresh:                   # every row is read, one per step: the step gets it as its override
            self._tables = (torch.as_tensor(an[:, None]).to(env.device), torch.as_tensor(pn[:, None]).to(env.device))
        self.t = nb                       # multiagent.py:59-61 leaves t == N_BURN_IN forever (Q1)
        self.states = None
        return self._sync_out()

    def _step(self, v_action, add_wind=True):
        if self.states is None:
            raise TypeError("cannot unpack non-iterable NoneType object")   # multiagent.py:31 before reset
        env = self._env
        a = torch.as_tensor(np.ascontiguousarray(v_action, dtype=np.float64)[None]).to(env.device)
        if self._fresh:
            an, pn = self._tables
            if self.t >= an.shape[0]:     # multiagent.py:38 indexes agent_noise[self.t] first
                raise IndexError("index %d is out of bounds for axis 0 with size %d" % (self.t, an.shape[0]))
            _, reward, done, _ = env.step(a, noise_a=an[self.t], noise_x=pn[self.t], add_wind=bool(add_wind))
            self.t += 1
        else:
            _, reward, done, _ = env.step(a, add_wind=bool(add_wind))      # multiagent.py:35-36
        self._sync_out()
        return self.states, np.float64(reward[0].item()), np.bool_(done[0].item()), {}

    # ---- static helpers of the reference class, each one kernel through the C ABI
    @staticmethod
    def s(r, F, L):
        lib = nat.load()
        r_t = torch.as_tensor(np.ascontiguousarray(r, dtype=np.float64)).cuda()
        out = torch.empty_like(r_t)
        nat.check(lib.swarm_s_potential(_ptr(r_t), _ptr(out), r_t.numel(), float(F), float(L),
                                        _stream(r_t.device)), "swarm_s_potential")
        return out.cpu().numpy()

    @staticmethod
    def x_update(x, v, dt, noise):
        lib = nat.load()
        x_t = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).cuda()
        v_t = torch.as_tensor(np.ascontiguousarray(v, dtype=np.float64)).cuda()
        n_t = torch.as_tensor(np.array(np.broadcast_to(noise, x.shape), dtype=np.float64)).cuda()
        nat.check(lib.swarm_x_update(_ptr(x_t), _ptr(v_t), _ptr(n_t), x_t.shape[0], float(dt),
                                     _stream(x_t.device)), "swarm_x_update")
        x[...] = x_t.cpu().numpy()
        v[...] = v_t.cpu().numpy()
        return x

    @staticmethod
    def xv_cutoff(x, v):
        lib = nat.load()
        x_t = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).cuda()
        v_t = torch.as_tensor(np.ascontiguousarray(v, dtype=np.float64)).cuda()
        nat.check(lib.swarm_xv_cutoff(_ptr(x_t), _ptr(v_t), x_t.shape[0], _stream(x_t.device)), "swarm_xv_cutoff")
        x[...] = x_t.cpu().numpy()
        v[...] = v_t.cpu().numpy()
        return x, v

    @staticmethod
    def v_calculate(x, xa, F, L, U, G):
        lib = nat.load()
        x_t = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)[None]).cuda()
        xa_t = torch.as_tensor(np.ascontiguousarray(xa, dtype=np.float64)[None]).cuda()
        tuning = nat.TUNE_CLUSTER_AUTO if x_t.shape[1] > nat.MAX_LOCUSTS_ONE_CTA else 0
        p = nat.SwarmParams(n_envs=1, n_locusts=x_t.shape[1], n_agents=xa_t.shape[1], grid_size=84, n_burn_in=10,
                            max_episode_steps=0, math_mode=0, tuning=tuning, noise=1e-4, gravity=float(G),
                            wind=float(U), F=float(F), L=float(L), dt=0.05, box_width=3.0, box_height=3.0,
                            seed=0, env_id_offset=0)
        v = torch.empty(1, x_t.shape[1], 2, dtype=torch.float32, device=x_t.device)
        r = torch.empty(1, dtype=torch.float32, device=x_t.device)
        nat.check(lib.swarm_forces(ctypes.byref(p), _ptr(x_t), _ptr(xa_t), _ptr(v), _ptr(r),
                                   _stream(x_t.device)), "swarm_forces")
        return v[0].double().cpu().numpy(), np.float64(r[0].item())


# fed_gym/__init__.py:21-33 -- the two registered swarm ids and their TimeLimit
REGISTRY = {
    "Swarm-v0": dict(max_episode_steps=128, kwargs={}),
    "Swarm-eval-v0": dict(max_episode_steps=128, kwargs=dict(seed=192)),
}


def make(env_id, **kw):
    """gym.make for the two swarm ids (fed_gym/agents/paac/environment_creator.py:20)."""
    spec = REGISTRY[env_id]
    args = dict(spec["kwargs"])
    args.update(kw)
    return SwarmEnv(max_episode_steps=spec["max_episode_steps"], **args)
