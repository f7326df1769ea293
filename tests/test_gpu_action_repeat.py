"""GPU: action repeat (swarm_step_repeat, BatchedSwarmEnv(action_repeat=K)).

Twin envs from one state: A makes one repeat-K call; B makes K single steps without auto-reset (only the first one
clips) and records every substep; C resets the envs that ended (mask, the same injected draws and physics).  A's
reward is the in-order FP32 sum of B's rewards up to each env's first done; done, terminated, truncated, final_x /
final_xa / final_grid and v_out are B's at that substep; envs that did not end hold B's state after K substeps, the
others C's; grid / positions are the observation of A's returned state.  All bit for bit.  Then repeat 1 against the
existing calls, a real termination inside a repeat, the production shapes under graph replay with an oracle sample,
and PAAC with action_repeat=4.
"""
import numpy as np
import pytest
import torch

from oracle import swarm_oracle as so

from _action_repeat import fold_substeps

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def M(pkg, cuda):
    return pkg.submodule("envs.multiagent")


def bits(t):
    return t.detach().cpu().numpy().tobytes()


def actions(E, A, gen, dtype=torch.float32):
    # a share of the rows beyond |a| = 1, so that clipping changes some of them
    return (1.3 * torch.randn(E, A, 2, device="cuda", generator=gen)).to(dtype).contiguous()


RANGES = {"F": (0.3, 0.7), "L": (5.0, 15.0), "wind": (0.5, 1.5), "gravity": (-1.5, -0.5), "dt": (0.04, 0.06)}
STATE = ("x", "xa", "noise_x", "noise_a", "elapsed", "episode")


def twin_repeat(M, E, N, K, calls=3, draws=False, final_obs=True, dtype=torch.float32, clip=True, add_wind=True,
                override=False, physics=None, **kw):
    """A / B / C twins over `calls` repeat-K calls from staggered episodes (TimeLimit 2K + 1, which K does not divide);
    returns the set of substep indices at which some env ended."""
    limit = 2 * K + 1
    kw.setdefault("binding", "torch")
    mk = lambda **k: M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=limit, seed=77, physics=physics,
                                       **dict(kw, **k))
    A, B, C = mk(final_obs=final_obs, action_repeat=K), mk(auto_reset=False), mk()
    A.reset()
    A.stagger_episodes()
    rd = A.philox_draws() if draws else None
    gen = torch.Generator(device="cuda")
    gen.manual_seed(N + E + K)
    vA = torch.full((E, N, 2), -9.0, device="cuda")
    vB = torch.empty_like(vA)
    if final_obs:
        for k, v in (("final_x", -7.25), ("final_xa", -3.5), ("final_grid", -1.5), ("final_positions", 250)):
            getattr(A, k).fill_(v)
    ended = set()
    for _ in range(calls):
        sd = A.state_dict()
        B.load_state_dict(sd)
        C.load_state_dict(sd)
        before = {k: getattr(A, k).clone() for k in ("final_x", "final_xa", "final_grid", "final_positions")} \
            if final_obs else {}
        a = actions(E, A.A, gen, dtype)
        na = torch.randn(E, A.A, 2, device="cuda", dtype=torch.float64, generator=gen) if override else None
        nx = torch.randn(E, N, 2, device="cuda", dtype=torch.float64, generator=gen) if override else None
        aA, aB = a.clone(), a.clone()
        _, _, _, info = A.step(aA, clip=clip, reset_draws=rd, v_out=vA, add_wind=add_wind, noise_a=na, noise_x=nx)
        rec = {k: [] for k in ("x", "xa", "reward", "done", "elapsed", "v", "grid", "positions")}
        for s in range(K):
            B.step(aB, clip=clip and s == 0, v_out=vB, add_wind=add_wind, noise_a=na, noise_x=nx)
            g, p = B.observe()
            for k, t in (("x", B.x), ("xa", B.xa), ("reward", B.reward), ("done", B.done_u8), ("elapsed", B.elapsed),
                         ("v", vB), ("grid", g), ("positions", p)):
                rec[k].append(t.clone())
        rec = {k: torch.stack(v) for k, v in rec.items()}
        reward, done, last = fold_substeps(rec["reward"].cpu().numpy(), rec["done"].cpu().numpy().astype(bool))
        dm = torch.as_tensor(done, device="cuda")
        idx = torch.as_tensor(last, device="cuda")
        at = lambda k: rec[k][idx, torch.arange(E, device="cuda")]        # B at each env's last stepped substep
        C.reset(mask=dm, draws=rd)
        torch.cuda.synchronize()
        ended |= set(last[done].tolist())
        assert bits(aA) == bits(aB)                                          # clipped once, in place
        assert bits(A.reward) == reward.tobytes()
        assert np.array_equal(A.done_u8.cpu().numpy().astype(bool), done)
        assert bits(vA) == bits(at("v"))
        el_last = at("elapsed")
        if final_obs:
            assert bits(info["terminated"]) == bits(at("reward") >= 0)
            assert bits(info["truncated"]) == bits(el_last >= limit)
            for k, ref in (("final_x", at("x")), ("final_xa", at("xa")), ("final_grid", at("grid")),
                           ("final_positions", at("positions"))):
                assert bits(info[k][dm]) == bits(ref[dm]), k
                assert bits(info[k][~dm]) == bits(before[k][~dm]), k
        # the returned state: B's after K substeps where the env went on, C's where it ended and reset
        live = ~dm
        for k in ("x", "xa", "noise_x", "noise_a") + (("physics",) if physics is not None else ()):
            assert bits(getattr(A, k)[live]) == bits(getattr(B, k)[live]), k
            assert bits(getattr(A, k)[dm]) == bits(getattr(C, k)[dm]), k
        assert bits(A.elapsed[live]) == bits(el_last[live]) and (A.elapsed[dm] == 0).all()
        assert bits(A.episode[live]) == bits(sd["episode"][live])
        assert bits(A.episode[dm]) == bits(C.episode[dm]) and torch.equal(A.episode[dm], sd["episode"][dm] + 1)
        # the observation of the returned state
        g, p = A.grid.clone(), A.positions.clone()
        A.observe()
        assert bits(A.grid) == bits(g) and bits(A.positions) == bits(p)
    return ended


@pytest.mark.parametrize("K", [2, 3, 4, 8])
@pytest.mark.parametrize("N,tuning", [(64, 0), (64, 0x20), (64, 0x30), (80, 0), (80, 0x10), (80, 0x20), (80, 0x30),
                                      (256, 0), (256, 0x10), (256, 0x20), (256, 0x30)])
def test_twins_every_placement(M, K, N, tuning):
    assert twin_repeat(M, 41, N, K, tuning=tuning) == set(range(K))


@pytest.mark.parametrize("math,noise,draws", [("precise", "frozen", False), ("fast", "fresh", False),
                                              ("precise", "fresh", True), ("fast", "frozen", True)])
@pytest.mark.parametrize("N", [64, 80, 256])
def test_twins_math_noise_draws(M, N, math, noise, draws):
    assert twin_repeat(M, 23, N, 3, math_mode=math, noise=noise, draws=draws) == {0, 1, 2}


@pytest.mark.parametrize("physics", ["table", "resample"])
@pytest.mark.parametrize("final_obs", [True, False])
@pytest.mark.parametrize("binding", ["torch", "ctypes"])
def test_twins_physics_final_obs_bindings(M, physics, final_obs, binding):
    phys = RANGES if physics == "resample" else "table"
    assert twin_repeat(M, 23, 80, 4, physics=phys, final_obs=final_obs, binding=binding, noise="fresh") == {0, 1, 2, 3}


@pytest.mark.parametrize("binding", ["torch", "ctypes"])
@pytest.mark.parametrize("dtype,add_wind,override,noise", [(torch.float64, True, False, "frozen"),
                                                           (torch.float32, False, False, "fresh"),
                                                           (torch.float64, False, True, "fresh"),
                                                           (torch.float32, True, True, "frozen")])
def test_twins_actions_wind_overrides(M, binding, dtype, add_wind, override, noise):
    assert twin_repeat(M, 23, 80, 3, dtype=dtype, add_wind=add_wind, override=override, noise=noise,
                       binding=binding) == {0, 1, 2}


@pytest.mark.parametrize("N,cluster,math,noise,physics", [(700, 2, "fast", "frozen", None),
                                                          (700, 2, "precise", "fresh", "resample"),
                                                          (2049, None, "fast", "fresh", "table"),
                                                          (2049, None, "precise", "frozen", None)])
@pytest.mark.parametrize("binding", ["torch", "ctypes"])
def test_twins_cluster(M, N, cluster, math, noise, physics, binding):
    phys = RANGES if physics == "resample" else physics
    assert twin_repeat(M, 9, N, 3, calls=2, cluster=cluster, math_mode=math, noise=noise, physics=phys,
                       binding=binding, draws=binding == "ctypes") == {0, 1, 2}


@pytest.mark.parametrize("binding", ["torch", "ctypes"])
@pytest.mark.parametrize("final_obs,physics", [(False, None), (True, None), (False, "table"), (True, "table")])
@pytest.mark.parametrize("N,tuning", [(80, 0), (256, 0), (256, 0x30), (700, 2 << 8)])
def test_repeat_one_is_the_existing_call(M, binding, final_obs, physics, N, tuning):
    """repeat = 1 through swarm_step_repeat: swarm_step / swarm_step_final / swarm_step_physics in every output, and the
    same plan."""
    mk = lambda **k: M.BatchedSwarmEnv(19, n_locusts=N, max_episode_steps=3, seed=5, tuning=tuning, binding=binding,
                                       final_obs=final_obs, physics=physics, **k)
    A, B = mk(), mk()
    A.reset()
    A.stagger_episodes()
    B.load_state_dict(A.state_dict())
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    plan = A.plan()
    lib, ref = A.lib, B.lib
    calls = []
    for _ in range(4):
        a = actions(19, A.A, gen)
        vA, vB = torch.empty(19, N, 2, device="cuda"), torch.empty(19, N, 2, device="cuda")
        A.action_repeat = 1
        # A through the new entry point (ctypes) or op (torch), B through the existing call
        _step_repeat_one(M, A, a.clone(), vA)
        B.step(a.clone(), clip=True, v_out=vB)
        torch.cuda.synchronize()
        for k in STATE + ("grid", "positions", "reward", "done_u8") + (("physics",) if physics else ()) + \
                (("final_x", "final_xa", "terminated", "truncated", "final_grid", "final_positions") if final_obs else ()):
            assert bits(getattr(A, k)) == bits(getattr(B, k)), k
        assert bits(vA) == bits(vB)
        calls.append(int(A.done_u8.sum()))
    assert sum(calls) > 0
    # the plan of repeat 1 through swarm_step_plan_repeat is swarm_step_plan's / swarm_step_plan_physics'
    import ctypes
    nat = M.nat
    io = nat.SwarmStepIO()
    io.actions_f32 = A.actions.data_ptr()
    io.reward, io.done = A.reward.data_ptr(), A.done_u8.data_ptr()
    io.grid, io.positions = A.grid.data_ptr(), A.positions.data_ptr()
    io.flags = nat.SWARM_STEP_AUTO_RESET
    out = (ctypes.c_int32 * 8)()
    nat.check(lib.swarm_step_plan_repeat(A._params_ref, A._state_ref, ctypes.byref(io),
                                         A._phys_ref if physics else None, 1, out), "plan")
    keys = ("force_mode", "filler_warp", "raster_place", "threads", "ctas", "smem_bytes", "follower_ctas", "launches")
    got = dict(zip(keys, list(out)))
    places = ("none", "follower kernel", "raster warps in k_step", "k_step's own threads", "the env's cluster")
    got["raster_place"] = places[got["raster_place"]]
    if got["raster_place"] == "the env's cluster":                 # out[6] holds K in the cluster layout
        got["follower_ctas"] = 0
    for k in ("force_mode", "filler_warp", "raster_place", "threads", "ctas", "smem_bytes", "follower_ctas", "launches"):
        assert got[k] == plan[k], k


def _step_repeat_one(M, env, a, v):
    """env.step's arguments, sent through swarm_step_repeat / op step_repeat with repeat = 1."""
    import ctypes
    nat = M.nat
    flags = nat.SWARM_STEP_AUTO_RESET | nat.SWARM_STEP_CLIP_ACTIONS
    fin = [None] * 6
    if env.final_obs:
        fin = [env.final_x, env.final_xa, env.terminated, env.truncated, env.final_grid, env.final_positions]
    if env.ops is not None:
        phys = env._phys_args() if env.physics is not None else (None, 0, [0.0] * 6, [0.0] * 6)
        env.ops.step_repeat(env._blob, *env._state_t, a, None, None, env.reward, env.done_u8, env.grid, env.positions,
                            v, flags, [], 1, *phys, *fin)
        return
    io = nat.SwarmStepIO()
    io.actions_f32 = a.data_ptr()
    io.reward, io.done = env.reward.data_ptr(), env.done_u8.data_ptr()
    io.grid, io.positions = env.grid.data_ptr(), env.positions.data_ptr()
    io.v_out = v.data_ptr()
    io.flags = flags
    f = None
    if env.final_obs:
        f = nat.SwarmStepFinal(*[t.data_ptr() for t in fin])
    with env._ctx:
        nat.check(env.lib.swarm_step_repeat(env._params_ref, env._state_ref, ctypes.byref(io),
                                            ctypes.byref(f) if f is not None else None,
                                            env._phys_ref if env.physics is not None else None, 1, None,
                                            torch.cuda.current_stream().cuda_stream), "swarm_step_repeat")


def test_plan_repeat_reports_the_rep_kernels(M):
    env = M.BatchedSwarmEnv(64, n_locusts=80, seed=1)
    env.reset()
    p1 = env.plan()
    env.action_repeat = 4
    p4 = env.plan()
    for k in ("force_mode", "threads", "smem_bytes"):
        assert p1[k] == p4[k], k
    env.action_repeat = 1
    assert env.plan() == p1
    with pytest.raises(ValueError):
        env.action_repeat = 2
        env.step_host(None, None, None)
    # a multi-wave batch with three force warps: raster warps at K = 1, the follower kernel from K = 2 on
    big = M.BatchedSwarmEnv(4096, n_locusts=80, seed=1)
    assert big.plan()["raster_place"] == "raster warps in k_step"
    for k in (2, 4, 8):
        big.action_repeat = k
        assert big.plan()["raster_place"] == "follower kernel", k


@pytest.mark.parametrize("binding", ["torch", "ctypes"])
def test_real_termination_inside_a_repeat(M, binding):
    """One locust, no wind, no gravity, every agent 1e4 away (test_gpu_final_obs.py): every substep has reward 0 >= 0,
    so each env stops at substep 0 with terminated set, auto-resets once, and the TimeLimit at elapsed 2 sets
    truncated as well."""
    E, lim, K = 6, 3, 4
    mk = lambda **k: M.BatchedSwarmEnv(E, n_locusts=1, max_episode_steps=lim, seed=5, binding=binding, **k)
    A, B = mk(final_obs=True, action_repeat=K), mk(auto_reset=False)
    for env in (A, B):
        env.params.wind = 0.0
        env.params.gravity = 0.0
    A.reset()
    A.xa.fill_(1e4)
    A.elapsed.copy_(torch.tensor([0, 1, 2, 2, 1, 0], dtype=torch.int32))
    pre = A.state_dict()
    B.load_state_dict(pre)
    a = torch.zeros(E, A.A, 2, device="cuda")
    _, r, d, info = A.step(a.clone())
    B.step(a.clone())
    gB, pB = B.observe()
    torch.cuda.synchronize()
    assert (r == 0).all() and d.all() and info["terminated"].all()
    assert info["truncated"].cpu().tolist() == [False, False, True, True, False, False]
    assert bits(info["final_x"]) == bits(B.x) and bits(info["final_xa"]) == bits(B.xa)
    assert bits(info["final_grid"]) == bits(gB) and bits(info["final_positions"]) == bits(pB)
    assert (A.elapsed == 0).all() and (A.episode == 2).all()
    # without auto-reset the env stays at its terminal state: one substep, not K
    A2 = mk(final_obs=True, action_repeat=K, auto_reset=False)
    A2.params.wind = A2.params.gravity = 0.0
    A2.load_state_dict(pre)
    A2.step(a.clone())
    torch.cuda.synchronize()
    for k in STATE:
        assert bits(getattr(A2, k)) == bits(getattr(B, k)), k
    assert torch.equal(A2.elapsed, pre["elapsed"] + 1)


@pytest.mark.parametrize("E,N", [(4096, 256), (1024, 64)])
def test_production_shapes_graph_replay_and_oracle(M, E, N):
    """K = 4: a graph-replayed repeat call equals its eager twin in every output.  A sample of envs matches the oracle
    teacher-forced per substep: a single-step twin B (no auto-reset) records every substep, each of B's substeps is
    the oracle's step from B's previous state within the per-step tolerance, and the repeat call returns B's state (or
    terminal state) bit for bit; done / elapsed / episode exact."""
    K, limit = 4, 128
    mk = lambda **k: M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=limit, seed=4242, **k)
    G_, A_ = mk(final_obs=True, action_repeat=K), mk(final_obs=True, action_repeat=K)
    B = mk(auto_reset=False)
    G_.reset()
    G_.stagger_episodes()
    A_.load_state_dict(G_.state_dict())
    gen = torch.Generator(device="cuda")
    gen.manual_seed(7)
    acts = [torch.randn(E, 10, 2, device="cuda", generator=gen).clamp(-0.7, 0.7) for _ in range(4)]
    buf = acts[0].clone()
    G_.step(buf.clone())
    A_.step(acts[0].clone())
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        G_.step(buf)
    sample = torch.as_tensor(np.unique(np.linspace(0, E - 1, 12).astype(int)), device="cuda")
    for s in range(1, 4):
        sd = A_.state_dict()
        B.load_state_dict(sd)
        buf.copy_(acts[s])
        g.replay()
        A_.step(acts[s].clone())
        xs, xas, dones = [sd["x"][sample].clone()], [sd["xa"][sample].clone()], []
        for _ in range(K):
            B.step(acts[s].clone())
            xs.append(B.x[sample].clone())
            xas.append(B.xa[sample].clone())
            dones.append(B.done_u8[sample].clone())
        torch.cuda.synchronize()
        for k in STATE + ("grid", "positions", "reward", "done_u8", "final_x", "final_xa", "terminated", "truncated",
                          "final_grid", "final_positions"):
            assert bits(getattr(G_, k)) == bits(getattr(A_, k)), (s, k)
        xs, xas = [t.cpu().numpy() for t in xs], [t.cpu().numpy() for t in xas]
        dones = torch.stack(dones).cpu().numpy().astype(bool)
        a = acts[s][sample].cpu().numpy().astype(np.float64)
        na, nx = sd["noise_a"][sample].cpu().numpy(), sd["noise_x"][sample].cpu().numpy()
        el0, ep0 = sd["elapsed"][sample].cpu().numpy(), sd["episode"][sample].cpu().numpy()
        for i, e in enumerate(sample.tolist()):
            for sub in range(K):
                x, xa = xs[sub][i][None].copy(), xas[sub][i][None].copy()     # teacher-forced: B's state before
                r, _ = so.step(x, xa, a[i][None], na[i][None], nx[i][None])
                assert np.abs(x[0] - xs[sub + 1][i]).max() <= 1e-5 * np.abs(x[0]).max(), (e, sub)
                assert np.array_equal(xa[0], xas[sub + 1][i]), (e, sub)
                assert dones[sub, i] == (bool(r[0] >= 0) or el0[i] + sub + 1 >= limit), (e, sub)
                if dones[sub, i]:
                    break
            done = bool(dones[sub, i])
            assert bool(A_.done_u8[e]) == done
            if done:
                assert int(A_.elapsed[e]) == 0 and int(A_.episode[e]) == int(ep0[i]) + 1
                assert bits(A_.final_x[e]) == xs[sub + 1][i].tobytes()
            else:
                assert int(A_.elapsed[e]) == int(el0[i]) + K and int(A_.episode[e]) == int(ep0[i])
                assert bits(A_.x[e]) == xs[K][i].tobytes() and bits(A_.xa[e]) == xas[K][i].tobytes()


# ---------------------------------------------------------------------------------------------------- PAAC
def make_learner(pkg, E=4, n_locusts=16, graph=False, K=4):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import train_paac_conv as tp
    args = tp.get_arg_parser().parse_args(["--clip_norm", "1", "-ec", str(E), "--n_locusts", str(n_locusts),
                                           "--action_repeat", str(K)])
    net_creator, env_creator = tp.get_network_and_environment_creator(args)
    paac = pkg.submodule("agents.paac.paac")
    return paac.GridPAACLearner(net_creator, env_creator, args, use_cuda_graph=graph, compact_obs=True)


def test_paac_action_repeat_graph_rollout_equals_eager_env(pkg, M):
    """action_repeat=4 with a TimeLimit of 7 inside the rollout: the graph-replayed updates train (finite loss inputs),
    and the rewards and dones they stored are those of an eager repeat-4 env stepped with the rollout's actions."""
    L = make_learner(pkg, graph=True)
    assert L.env.action_repeat == 4
    L.env.params.max_episode_steps = 7
    L.start()
    E, A, T = L.emulator_counts, L.N_AGENTS, L.max_local_steps
    p = L.env.params
    twin = M.BatchedSwarmEnv(E, n_locusts=16, max_episode_steps=7, seed=int(p.seed), env_id_offset=int(p.env_id_offset),
                             action_repeat=4)
    for _ in range(2):
        twin.load_state_dict(L.env.state_dict())
        L.update()
        torch.cuda.synchronize()
        for t in range(T):
            twin.step(L.actions[t].view(E, A, 2).contiguous())
            assert bits(L.rewards[t, :E]) == bits(twin.reward), t
            assert bits(L.not_over[t].view(E, A)[:, 0]) == bits(1 - twin.done_u8.float()), t
        for k in STATE:
            assert bits(getattr(L.env, k)) == bits(getattr(twin, k)), k
    assert (L.not_over == 0).any() and torch.isfinite(L.y_batch).all()
