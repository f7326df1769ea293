"""GPU: the terminal outputs of swarm_step_final (BatchedSwarmEnv(final_obs=True)).

Twin envs from one state: A keeps the terminal outputs, B is the same env without them, C steps without auto-reset
(reloaded from A before every step, since it does not reset its finished envs).  For every done env A's final_x /
final_xa are C's post-step state and A's final_grid / final_positions are C.observe(), bit for bit; A's every other
output is B's, bit for bit; the rows of envs that are not done keep their (sentinel) bytes.  Then the done split,
the production shapes under CUDA-graph replay, the oracle's process_state, and PAAC's truncation bootstrap.
"""
import numpy as np
import pytest
import torch

from oracle import swarm_oracle as so

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def M(pkg, cuda):
    return pkg.submodule("envs.multiagent")


def bits(t):
    return t.detach().cpu().numpy().tobytes()


def actions(E, A, gen):
    a = torch.randn(E, A, 2, device="cuda", generator=gen)
    n = a.norm(dim=-1, keepdim=True)
    return torch.where(n >= 1.0, a / n, a).contiguous()


SENT = dict(final_x=-7.25, final_xa=-3.5, final_grid=-1.5, final_positions=250)


def twin_run(M, E, N, steps=5, limit=4, draws=False, **kw):
    """Runs the A / B / C twins with staggered episodes; returns the number of done env-steps checked."""
    kw.setdefault("binding", "torch")
    mk = lambda **k: M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=limit, seed=77, **dict(kw, **k))
    A, B, C = mk(final_obs=True), mk(), mk(auto_reset=False)
    A.reset()
    A.stagger_episodes()
    B.load_state_dict(A.state_dict())
    for k, v in SENT.items():
        getattr(A, k).fill_(v)
    rd = A.philox_draws() if draws else None
    gen = torch.Generator(device="cuda")
    gen.manual_seed(N + E)
    n_done = 0
    for _ in range(steps):
        C.load_state_dict(A.state_dict())
        el0 = A.elapsed.clone()
        before = {k: getattr(A, k).clone() for k in SENT}
        a = actions(E, A.A, gen)
        _, rA, dA, info = A.step(a.clone(), reset_draws=rd)
        B.step(a.clone(), reset_draws=rd)
        C.step(a.clone())
        gC, pC = [t.clone() for t in C.observe()]
        torch.cuda.synchronize()
        for k in ("x", "xa", "grid", "positions", "reward", "done_u8", "elapsed", "episode", "noise_x", "noise_a"):
            assert bits(getattr(A, k)) == bits(getattr(B, k)), k
        assert torch.equal(A.reward, C.reward) and torch.equal(A.done_u8, C.done_u8)
        d = dA.clone()
        term = C.reward >= 0
        trunc = (el0 + 1) >= limit
        assert torch.equal(info["terminated"], term) and torch.equal(info["truncated"], trunc)
        assert torch.equal(d, info["terminated"] | info["truncated"])
        for k, ref in (("final_x", C.x), ("final_xa", C.xa), ("final_grid", gC), ("final_positions", pC)):
            got = info[k]
            assert got.data_ptr() == getattr(A, k).data_ptr()
            assert bits(got[d]) == bits(ref[d]), k
            assert bits(got[~d]) == bits(before[k][~d]), k
        n_done += int(d.sum())
    return n_done


@pytest.mark.parametrize("binding", ["torch", "ctypes"])
@pytest.mark.parametrize("N,tuning", [(80, 0x10), (80, 0x20), (80, 0x30), (64, 0x20), (64, 0x30), (256, 0x10),
                                      (256, 0x30), (256, 0)])
def test_twins_every_placement(M, binding, N, tuning):
    assert twin_run(M, 53, N, tuning=tuning, binding=binding) > 0


@pytest.mark.parametrize("math,noise,draws", [("precise", "frozen", False), ("fast", "fresh", False),
                                              ("precise", "fresh", True), ("fast", "frozen", True)])
@pytest.mark.parametrize("N", [64, 80, 256])
def test_twins_math_noise_draws(M, N, math, noise, draws):
    assert twin_run(M, 41, N, math_mode=math, noise=noise, draws=draws) > 0


@pytest.mark.parametrize("N,cluster,math,noise", [(700, 2, "fast", "frozen"), (700, 2, "precise", "fresh"),
                                                  (2049, None, "fast", "frozen"), (2049, None, "precise", "fresh")])
@pytest.mark.parametrize("binding", ["torch", "ctypes"])
def test_twins_cluster(M, N, cluster, math, noise, binding):
    assert twin_run(M, 9, N, steps=4, cluster=cluster, math_mode=math, noise=noise, binding=binding,
                    draws=binding == "ctypes") > 0


def test_without_rasterizer_and_without_auto_reset(M):
    """rasterize=False: state and flags only (final_grid stays None); auto_reset=False: final_x is the returned state."""
    E, N = 16, 80
    env = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=2, seed=3, rasterize=False, auto_reset=False,
                            final_obs=True)
    env.reset()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1)
    for s in range(2):
        _, _, d, info = env.step(actions(E, env.A, gen))
        torch.cuda.synchronize()
        assert info["final_grid"] is None and bool(d.all()) == (s == 1)
    assert torch.equal(info["final_x"], env.x) and torch.equal(info["final_xa"], env.xa)
    assert info["truncated"].all() and not info["terminated"].any()


@pytest.mark.parametrize("binding", ["torch", "ctypes"])
def test_done_split_truncation_count_and_no_limit(M, binding):
    E, N, lim = 32, 80, 5
    env = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=lim, seed=9, final_obs=True, binding=binding)
    env.reset()
    env.stagger_episodes()
    host = env.elapsed.cpu().numpy().astype(np.int64)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2)
    for _ in range(2 * lim):
        _, _, d, info = env.step(actions(E, env.A, gen))
        host += 1
        want = host >= lim
        assert np.array_equal(info["truncated"].cpu().numpy(), want)
        assert np.array_equal(d.cpu().numpy(), want) and not info["terminated"].any()
        host[want] = 0
    free = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=0, seed=9, final_obs=True, binding=binding)
    free.reset()
    free.truncated.fill_(7)
    for _ in range(4):
        _, _, d, info = free.step(actions(E, free.A, gen))
        assert not info["truncated"].any() and not d.any()


@pytest.mark.parametrize("binding", ["torch", "ctypes"])
def test_real_termination_both_flags(M, binding):
    """One locust, no wind, no gravity, every agent 1e4 away: every term of v_calculate underflows to 0 (s(r) =
    F exp(-r / L) - exp(-r) with r ~ 1.4e4), so reward = -mean |v|^2 = 0 >= 0: terminated.  At elapsed == limit both
    flags are set."""
    E, lim = 6, 3
    mk = lambda **k: M.BatchedSwarmEnv(E, n_locusts=1, max_episode_steps=lim, seed=5, binding=binding, **k)
    A, C = mk(final_obs=True), mk(auto_reset=False)
    for env in (A, C):
        env.params.wind = 0.0
        env.params.gravity = 0.0
    A.reset()
    A.xa.fill_(1e4)
    A.elapsed.copy_(torch.tensor([0, 1, 2, 2, 1, 0], dtype=torch.int32))
    C.load_state_dict(A.state_dict())
    a = torch.zeros(E, A.A, 2, device="cuda")
    _, r, d, info = A.step(a.clone())
    C.step(a.clone())
    gC, pC = C.observe()
    torch.cuda.synchronize()
    assert (r == 0).all() and d.all() and info["terminated"].all()
    assert info["truncated"].cpu().tolist() == [False, False, True, True, False, False]
    assert bits(info["final_x"]) == bits(C.x) and bits(info["final_xa"]) == bits(C.xa)
    assert bits(info["final_grid"]) == bits(gC) and bits(info["final_positions"]) == bits(pC)
    assert (A.elapsed == 0).all() and (A.episode == 2).all()         # auto-reset after the termination


@pytest.mark.parametrize("E,N", [(4096, 256), (1024, 64)])
def test_production_shapes_graph_replay(M, E, N):
    """TimeLimit(2): every env ends on alternate steps.  A graph-replayed final_obs env equals its eager twin bit for
    bit (every output, terminal ones included), equals the no-reset twin on the terminal state and observation, and
    sampled terminal grids are the oracle's numpy process_state of final_x / final_xa."""
    mk = lambda **k: M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=2, seed=4242, **k)
    G_, A_, C = mk(final_obs=True), mk(final_obs=True), mk(auto_reset=False)
    G_.reset()
    A_.load_state_dict(G_.state_dict())
    gen = torch.Generator(device="cuda")
    gen.manual_seed(7)
    acts = [actions(E, 10, gen) for _ in range(4)]
    buf = acts[0].clone()
    G_.step(buf.clone())                                # warm-up outside the capture
    A_.step(acts[0].clone())
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        G_.step(buf)
    sample = np.unique(np.linspace(0, E - 1, 24).astype(int))
    for s in range(1, 4):
        C.load_state_dict(A_.state_dict())
        buf.copy_(acts[s])
        g.replay()
        A_.step(acts[s].clone())
        C.step(acts[s].clone())
        gC, pC = C.observe()
        torch.cuda.synchronize()
        for k in ("x", "xa", "grid", "positions", "reward", "done_u8", "elapsed", "episode", "final_x", "final_xa",
                  "terminated", "truncated", "final_grid", "final_positions"):
            assert bits(getattr(G_, k)) == bits(getattr(A_, k)), (s, k)
        d = A_.done_u8.bool()
        assert bool(d.all()) == (s % 2 == 1)
        if not d.any():
            continue
        assert bits(A_.final_x[d]) == bits(C.x[d]) and bits(A_.final_xa[d]) == bits(C.xa[d])
        assert bits(A_.final_grid[d]) == bits(gC[d]) and bits(A_.final_positions[d]) == bits(pC[d])
        fx, fxa = A_.final_x[sample].cpu().numpy(), A_.final_xa[sample].cpu().numpy()
        fg, fp = A_.final_grid[sample].cpu().numpy(), A_.final_positions[sample].cpu().numpy()
        for i in range(len(sample)):
            og, op = so.rasterize(fx[i], fxa[i], 84)
            assert np.array_equal(fg[i], og.astype(np.float32)) and np.array_equal(fp[i], op)


# ---------------------------------------------------------------------------------------------------- PAAC
def make_learner(pkg, E=4, n_locusts=16, graph=False, limit=3, **kw):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import train_paac_conv as tp
    args = tp.get_arg_parser().parse_args(["--clip_norm", "1", "-ec", str(E), "--n_locusts", str(n_locusts)])
    net_creator, env_creator = tp.get_network_and_environment_creator(args)
    paac = pkg.submodule("agents.paac.paac")
    L = paac.GridPAACLearner(net_creator, env_creator, args, use_cuda_graph=graph, **kw)
    L.env.params.max_episode_steps = limit
    return L


@pytest.mark.parametrize("compact", [False, True])
def test_paac_truncation_bootstrap_matches_numpy(pkg, cuda, compact):
    """max_episode_steps = 3 inside T = 5: y_batch is the numpy recomputation of
    ret_t = r_t + g [(1 - done_t) ret_t+1 + truncated_t (1 - terminated_t) V(final_t)] from the recorded rings."""
    L = make_learner(pkg, mask_terminals=True, bootstrap_truncated=True, compact_obs=compact,
                     reward_indexing="per_agent")
    L.start()
    L._rollout()
    with torch.no_grad():
        L._returns()
    torch.cuda.synchronize()
    T, E, A = L.max_local_steps, L.emulator_counts, L.N_AGENTS
    tr, te = L.truncated.cpu().numpy(), L.terminated.cpu().numpy()
    assert tr[2].all() and tr.sum() == tr[2].sum() and not te.any()     # the episode's 3rd step is t = 2
    v_fin = L.network.predict_compact(L.final_grids.view(T * E, *L.final_grids.shape[2:]),
                                      L.final_positions.view(T * E, A, 2))["vs"].float().view(T, -1).cpu().numpy()
    if compact:
        boot = L.network.predict_compact(L.grids[T], L.positions[T])["vs"].cpu().numpy()
    else:
        boot = L.network.predict(L.states[T].view(E * A, *L.states.shape[3:]))["vs"].cpu().numpy()
    r, nov = L.rewards.cpu().numpy(), L.not_over.cpu().numpy()
    g = np.float32(L.gamma)
    ret = boot
    for t in reversed(range(T)):
        ret = r[t] + g * (ret * nov[t] + v_fin[t] * tr[t] * (1 - te[t]))
        assert np.allclose(L.y_batch[t].cpu().numpy(), ret, rtol=1e-5, atol=1e-4), t
    # the truncated step's target really bootstraps: it differs from the masked one
    assert not np.allclose(L.y_batch[2].cpu().numpy(), r[2])


def test_paac_bootstrap_graph_replay_equals_eager(pkg, cuda):
    """The whole update (rollout with the terminal rings, the terminal value forward, returns, Adam) replays as one
    CUDA graph; with the learning rate at 0 the returns it produced equal an eager recomputation from its rings."""
    L = make_learner(pkg, mask_terminals=True, bootstrap_truncated=True, graph=True, compact_obs=True)
    L.initial_lr = 0.0
    L.start()
    for _ in range(2):
        L.update()
    torch.cuda.synchronize()
    assert L._graph is not None and L.truncated.any()
    y = L.y_batch.clone()
    with torch.no_grad():
        L._returns()
    torch.cuda.synchronize()
    assert torch.equal(y, L.y_batch)
