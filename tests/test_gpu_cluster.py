"""The cluster layout on the B200: one env over the K CTAs of a thread-block cluster (tuning bits 8-12).

(a) 512 < N <= 2048: every output bitwise equal to the one-CTA kernels, for every legal K, in both math modes;
(b) N > 2048: the same bits for every K;
(c) against the FP64 oracle: per-locust forces within the bound T_j of test_force_probe_model, teacher-forced steps;
(d) the observation at N > 2048 bit-exact against numpy, fused and standalone, with and without the box;
(e) large batches, graph replay, step_host, shard invariance, torch.ops = ctypes, the SwarmEnv facade, PAAC;
(f) plan() names the layout; refused layouts raise before anything is launched.
"""
import numpy as np
import pytest
import torch

from oracle import swarm_oracle as so

import test_force_probe_model as fp
from test_cluster_layout import step_chunked

pytestmark = pytest.mark.gpu

MATH = ["fast", "precise"]


@pytest.fixture(scope="module")
def M(pkg, cuda):
    return pkg.submodule("envs.multiagent")


@pytest.fixture(scope="module")
def nat(pkg):
    from golds_rl_gym_b200 import _native
    return _native


def force_warps(N):
    T = 2 if N <= 1024 else 4
    return (-(-N // T) + 31) // 32


def legal_k(N):
    nw = force_warps(N)
    return list(range(-(-nw // 32), min(16, nw) + 1))


def new_env(M, N, E, cluster, math="fast", noise="frozen", A=10, G=84, **kw):
    kw.setdefault("binding", "ctypes")
    return M.BatchedSwarmEnv(E, n_locusts=N, n_agents=A, grid_size=G, max_episode_steps=128, seed=11,
                             math_mode=math, noise=noise, cluster=cluster, **kw)


def bits(t):
    a = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
    return a.tobytes()


def scenario(M, N, E, cluster, math, variant, steps=16):
    """Every output of a reset and `steps` steps, as bytes.  The TimeLimit is hit mid-way (auto-reset)."""
    noise = "fresh" if variant == "fresh" else "frozen"
    env = new_env(M, N, E, cluster, math, noise)
    A = env.A
    draws = None
    if variant == "injected":
        ds = [so.draw_reset_numpy(np.random.RandomState(300 + e), N) for e in range(E)]
        draws = M.InjectedDraws(*[np.stack([d[i] for d in ds]) for i in range(5)], device=env.device)
    env.reset(draws=draws)
    env.elapsed.copy_(torch.arange(E, dtype=torch.int32, device=env.device) + 128 - steps // 2)
    rs = np.random.RandomState(N)
    out = [bits(env.x), bits(env.xa), bits(env.noise_x), bits(env.noise_a), bits(env.episode)]
    v = torch.zeros(E, N, 2, dtype=torch.float32, device=env.device)
    for s in range(steps):
        a = torch.as_tensor(rs.normal(scale=1.5, size=(E, A, 2))).to(env.device)
        if variant != "f64":
            a = a.float()
        kw = {}
        if variant == "overrides" and s % 3 == 1:
            kw = dict(noise_a=torch.as_tensor(rs.normal(size=(E, A, 2))).to(env.device),
                      noise_x=torch.as_tensor(rs.normal(size=(E, N, 2))).to(env.device))
        (x, xa), r, d, _ = env.step(a, clip=variant in ("clip", "f64"), v_out=v, add_wind=variant != "nowind",
                                    reset_draws=draws, **kw)
        out += [bits(x), bits(xa), bits(r), bits(d), bits(env.elapsed), bits(env.episode), bits(env.grid),
                bits(env.positions), bits(v), bits(a), bits(env.noise_x), bits(env.noise_a)]
    torch.cuda.synchronize()
    return out


VARIANTS = ["philox", "injected", "fresh", "overrides", "clip", "f64", "nowind"]


# ------------------------------------------------------------------------------------------------ (a)
@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("N", [513, 700, 1024, 1025, 2047, 2048])
def test_bitwise_equal_to_one_cta_every_k(M, N, math):
    ref = scenario(M, N, 3, None, math, "clip")
    for K in legal_k(N):
        got = scenario(M, N, 3, K, math, "clip")
        bad = [i for i, (g, r) in enumerate(zip(got, ref)) if g != r]
        assert not bad, (K, bad[:5])


@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("N", [700, 2047])
def test_bitwise_equal_to_one_cta_every_feature(M, N, math, variant):
    ref = scenario(M, N, 3, None, math, variant)
    ks = legal_k(N)
    for K in sorted({ks[0], 3, ks[-1]} & set(ks)):
        got = scenario(M, N, 3, K, math, variant)
        bad = [i for i, (g, r) in enumerate(zip(got, ref)) if g != r]
        assert not bad, (K, bad[:5])


@pytest.mark.parametrize("math", MATH)
def test_reset_and_forces_equal_one_cta(M, math):
    N, E = 1500, 4
    ref = new_env(M, N, E, None, math)
    ref.reset()
    for K in (1, 5, 12):
        env = new_env(M, N, E, K, math)
        env.reset()
        assert bits(env.x) == bits(ref.x) and bits(env.xa) == bits(ref.xa)
        assert bits(env.noise_x) == bits(ref.noise_x) and bits(env.episode) == bits(ref.episode)
        v0, r0 = ref.forces()
        v1, r1 = env.forces()
        assert bits(v0) == bits(v1) and bits(r0) == bits(r1)


# ------------------------------------------------------------------------------------------------ (b)
@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("N", [2049, 3000, 4096, 8192])
def test_same_bits_for_every_k(M, N, math):
    ks = legal_k(N)
    pick = sorted({ks[0], ks[0] + 1, 3, 5, 8, ks[-1]} & set(ks))
    ref = scenario(M, N, 2, pick[0], math, "philox", steps=8)
    for K in pick[1:]:
        got = scenario(M, N, 2, K, math, "philox", steps=8)
        bad = [i for i, (g, r) in enumerate(zip(got, ref)) if g != r]
        assert not bad, (K, bad[:5])


# ------------------------------------------------------------------------------------------------ (c)
def straddling_state(N, A, K, rs):
    """a dense swarm whose close pairs sit on both sides of every CTA's slice boundary of the virtual targets"""
    x = rs.rand(N, 2) * np.array([3.0, 2.0])
    nf = force_warps(N) * 32
    for r in range(1, K):
        w0 = (r * (nf // 32)) // K * 32            # first virtual target of CTA r (t = 0); t > 0 chunks follow at + t nf
        for t in range(4):
            j = w0 + t * nf
            if 0 < j < N:
                x[j] = x[j - 1] + rs.normal(scale=1e-4, size=2)
    return x, rs.rand(A, 2) * 3.0


@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("N", [2049, 4096, 8192])
@pytest.mark.parametrize("A", [1, 10, 32])
def test_forces_within_the_bound(M, N, A, math):
    rs = np.random.RandomState(N + A)
    K = legal_k(N)[-1]
    x, xa = straddling_state(N, A, K, rs)
    env = new_env(M, N, 1, K, math, A=A)
    env.x.copy_(torch.as_tensor(x[None]))
    env.xa.copy_(torch.as_tensor(xa[None]))
    v, r = env.forces()
    ref = fp.reference_dense(x[None], xa[None])
    q = fp.ratio(v.cpu().numpy().astype(np.float64), ref.v, ref.T(math))
    assert (q <= 1.0).all(), q.max()
    assert abs(float(r.item()) - ref.reward[0]) <= ref.reward_bound(math)[0] + 1e-6 * abs(ref.reward[0])


def force_tolerance(env, math):
    """twice the largest per-locust force bound T_j of env 0's state (the caller scales it by dt): each locust's FP32 chain over N + A
    sources carries up to ~sqrt(N + A) 2^-24 sum |term| (test_force_probe_model), which at N = 8192 exceeds the
    5e-6 max|x| of the smaller swarms"""
    ref = fp.reference_dense(env.x[:1].cpu().numpy(), env.xa[:1].cpu().numpy())
    return 2.0 * float(ref.T(math).max())


@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("N,A", [(2049, 10), (4096, 32), (8192, 1)])
def test_teacher_forced_steps_against_the_oracle(M, N, A, math):
    E, K = 2, legal_k(N)[-1]
    env = new_env(M, N, E, K, math, A=A, auto_reset=False)
    env.reset()
    rs = np.random.RandomState(7)
    nx, na = env.noise_x.cpu().numpy(), env.noise_a.cpu().numpy()
    tol_v = force_tolerance(env, math)
    for s in range(16):
        x, xa = env.x.cpu().numpy(), env.xa.cpu().numpy()
        a = rs.normal(size=(E, A, 2))
        (gx, gxa), r, d, _ = env.step(torch.as_tensor(a).to(env.device))
        rew, done = step_chunked(x, xa, a, na, nx)
        gx = gx.cpu().numpy()
        for e in range(E):
            assert np.abs(gx[e] - x[e]).max() <= 5e-6 * np.abs(x[e]).max() + so.DT * tol_v, (s, e)
        assert np.array_equal(gxa.cpu().numpy(), xa)
        assert np.array_equal(d.cpu().numpy(), done)


# ------------------------------------------------------------------------------------------------ (d)
def edge_state(N, A, G, rs, far=0.0):
    """points exactly on numpy's x edges of the state's own window, 1 ulp beside them, and x == hi"""
    x = rs.rand(N, 2) * np.array([3.0, 5.0]) + np.array([far, 0.0])
    xa = rs.rand(A, 2) * np.array([3.0, 5.0]) + np.array([far, 0.0])
    for it in range(3):       # the mean moves with the pinned points: settle a few times
        m = so.sequential_mean_x(x, xa)
        ex = so.box_edges(m - 1.5, m + 1.5, G)
        for k, i in enumerate(range(0, N, max(1, N // 40))):
            e = ex[k % (G + 1)]
            x[i, 0] = e if k % 3 == 0 else np.nextafter(e, np.inf if k % 3 == 1 else -np.inf)
        xa[0, 0] = ex[G]
    return x, xa


@pytest.mark.parametrize("N,A,G,far", [(2049, 10, 84, 0.0), (4096, 32, 255, 0.0), (8192, 10, 83, 1e4), (3000, 1, 2, 0.0)])
def test_observation_on_edges_is_numpys(M, N, A, G, far):
    rs = np.random.RandomState(N + G)
    E = 3
    xs, xas = zip(*[edge_state(N, A, G, rs, far) for _ in range(E)])
    x, xa = np.stack(xs), np.stack(xas)
    for K in sorted({max(2, legal_k(N)[0]), 3, legal_k(N)[-1]}):
        env = new_env(M, N, E, K, A=A, G=G)
        env.x.copy_(torch.as_tensor(x))
        env.xa.copy_(torch.as_tensor(xa))
        for with_box in (False, True):
            env.grid.fill_(7.0)
            box = torch.empty(E, 4, dtype=torch.float64, device=env.device) if with_box else None
            grid, pos = env.observe(box)
            g, p = grid.cpu().numpy(), pos.cpu().numpy()
            for e in range(E):
                gg, pp = so.rasterize(x[e], xa[e], G)
                assert np.array_equal(g[e], gg.astype(np.float32)) and np.array_equal(p[e], pp), (K, e, with_box)
                if with_box:
                    m = so.sequential_mean_x(x[e], xa[e])
                    assert box[e].tolist() == [m - 1.5, m + 1.5, 0.0, 6.0]
        # fused: the observation of the stepped state
        env.reset()
        env.x.copy_(torch.as_tensor(x))
        env.xa.copy_(torch.as_tensor(xa))
        (gx, gxa), _, _, _ = env.step(torch.zeros(E, A, 2, device=env.device), add_wind=False)
        gx, gxa = gx.cpu().numpy(), gxa.cpu().numpy()
        for e in range(E):
            gg, pp = so.rasterize(gx[e], gxa[e], G)
            assert np.array_equal(env.grid[e].cpu().numpy(), gg.astype(np.float32))
            assert np.array_equal(env.positions[e].cpu().numpy(), pp)


# ------------------------------------------------------------------------------------------------ (e)
@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("E,N", [(64, 8192), (148, 4096)])
def test_large_batches_time_limit_against_the_oracle(M, E, N, math):
    env = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=2, seed=3, math_mode=math, binding="ctypes")
    env.reset()
    rs = np.random.RandomState(1)
    sample = [0, E // 2, E - 1]
    tol_v = force_tolerance(env, math)
    for s in range(3):
        x, xa = env.x[sample].cpu().numpy(), env.xa[sample].cpu().numpy()
        nx, na = env.noise_x[sample].cpu().numpy(), env.noise_a[sample].cpu().numpy()
        a = rs.normal(size=(E, 10, 2)).astype(np.float32)
        (gx, gxa), r, d, _ = env.step(torch.as_tensor(a).cuda())
        done = d.cpu().numpy()
        assert done.all() == (s % 2 == 1)
        if s % 2 == 0:
            rew, _ = step_chunked(x, xa, a[sample].astype(np.float64), na, nx)
            g = gx[sample].cpu().numpy()
            for i in range(len(sample)):
                assert np.abs(g[i] - x[i]).max() <= 5e-6 * np.abs(x[i]).max() + so.DT * tol_v
            assert np.allclose(r[sample].cpu().numpy(), rew, rtol=1e-4)
            assert np.array_equal(gxa[sample].cpu().numpy(), xa)
        else:
            assert (env.elapsed == 0).all() and (env.episode == 2).all()


@pytest.mark.parametrize("math", MATH)
def test_graph_replay_equals_eager(M, math):
    N, E = 4096, 6
    outs = []
    for graph in (False, True):
        env = new_env(M, N, E, 4, math, binding="torch")
        env.reset()
        sd = env.state_dict()
        acts = [torch.as_tensor(np.random.RandomState(s).normal(size=(E, 10, 2)).astype(np.float32)).cuda() for s in range(4)]
        buf = torch.zeros_like(acts[0])
        if graph:
            env.step(buf)                                # warm-up outside the capture
            env.load_state_dict(sd)
            g = torch.cuda.CUDAGraph()
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                with torch.cuda.graph(g, stream=s):
                    env.step(buf)
            torch.cuda.current_stream().wait_stream(s)
            res = []
            for a in acts:
                buf.copy_(a)
                g.replay()
                res += [bits(env.x), bits(env.reward), bits(env.grid)]
        else:
            res = []
            for a in acts:
                env.step(a)
                res += [bits(env.x), bits(env.reward), bits(env.grid)]
        outs.append(res)
    assert outs[0] == outs[1]


def test_torch_ops_equal_ctypes_and_step_host(M):
    N, E = 3000, 4
    res = []
    for binding in ("ctypes", "torch"):
        env = new_env(M, N, E, None, binding=binding)
        env.reset()
        a = torch.as_tensor(np.random.RandomState(0).normal(size=(E, 10, 2)).astype(np.float32)).cuda()
        env.step(a)
        v, r = env.forces()
        res.append([bits(env.x), bits(env.xa), bits(env.grid), bits(env.positions), bits(v), bits(r)])
    assert res[0] == res[1]
    env = new_env(M, N, E, None)
    env.reset()
    ref = new_env(M, N, E, None)
    ref.reset()
    ha = torch.as_tensor(np.random.RandomState(1).normal(size=(E, 10, 2)).astype(np.float32)).pin_memory()
    hr, hd = torch.zeros(E).pin_memory(), torch.zeros(E, dtype=torch.uint8).pin_memory()
    for _ in range(3):
        env.step_host(ha, hr, hd)
        ref.step(ha.cuda())
        torch.cuda.synchronize()
        assert bits(hr) == bits(ref.reward) and bits(env.x) == bits(ref.x) and bits(env.grid) == bits(ref.grid)


def test_shard_invariance(M):
    N = 2500
    whole = new_env(M, N, 6, 3)
    whole.reset()
    halves = [new_env(M, N, 3, 5, env_id_offset=o) for o in (0, 3)]
    for h in halves:
        h.reset()
    a = torch.as_tensor(np.random.RandomState(2).normal(size=(6, 10, 2)).astype(np.float32)).cuda()
    whole.elapsed.fill_(127)
    for h in halves:
        h.elapsed.fill_(127)
    whole.step(a)
    for i, h in enumerate(halves):
        h.step(a[3 * i:3 * i + 3].contiguous())
        assert bits(h.x) == bits(whole.x[3 * i:3 * i + 3]) and bits(h.grid) == bits(whole.grid[3 * i:3 * i + 3])


def test_swarm_env_facade_and_creator_at_4096(M, pkg):
    class Big(M.SwarmEnv):
        N_LOCUSTS = 4096
    env = Big(seed=5, max_episode_steps=128)
    x, xa = env.reset()
    assert x.shape == (4096, 2)
    states, r, d, _ = env.step(np.zeros((10, 2)))
    assert np.isfinite(r) and states[0].shape == (4096, 2)
    v, rew = M.SwarmEnv.v_calculate(states[0], states[1], 0.5, 10, 1, -1)
    assert v.shape == (4096, 2) and np.isfinite(rew)
    ec = pkg.submodule("agents.paac.environment_creator")
    benv = ec.SwarmEnvironmentCreator(n_locusts=4096).create_batched_environment(2)
    assert benv.plan()["layout"] == "cluster"


def test_paac_update_at_4096(M, pkg, cuda):
    import test_paac_gpu as tp
    L = tp.make_learner(pkg, cuda, E=2, n_locusts=4096, compact_obs=False)
    assert L.envs.plan()["layout"] == "cluster" if hasattr(L, "envs") else True
    L.start()
    before = torch.cat([p.detach().flatten().clone() for p in L.network.parameters()])
    L.update()
    torch.cuda.synchronize()
    after = torch.cat([p.detach().flatten() for p in L.network.parameters()])
    assert torch.isfinite(after).all() and not torch.equal(before, after)


# ------------------------------------------------------------------------------------------------ (f)
def test_plan_names_the_cluster_layout(M):
    env = new_env(M, 4096, 4, 3)
    p = env.plan()
    assert p["layout"] == "cluster" and p["cluster_size"] == 3 and p["ctas"] == 12 and p["launches"] == 1
    assert p["raster_place"] == "the env's cluster"
    auto = M.BatchedSwarmEnv(1, n_locusts=8192, binding="ctypes").plan()
    assert auto["layout"] == "cluster" and 2 <= auto["cluster_size"] <= 16
    one = new_env(M, 1024, 4, None).plan()
    assert one["layout"] == "one CTA per env" and one["cluster_size"] == 1


def test_refused_layouts_raise_before_launch(M, nat):
    with pytest.raises(nat.SwarmNativeError):
        new_env(M, 4096, 2, 17)
    with pytest.raises(nat.SwarmNativeError):
        new_env(M, 512, 2, 2)
    with pytest.raises(nat.SwarmNativeError):
        new_env(M, 8193, 2, None)
    env = new_env(M, 8192, 2, 2)
    env.reset()
    x0 = env.x.clone()
    env.params.tuning = nat.tune_cluster(1)          # 2048 threads in one CTA: refused by the call itself
    with pytest.raises(nat.SwarmNativeError):
        env.step(torch.zeros(2, 10, 2, device=env.device))
    torch.cuda.synchronize()
    assert bits(env.x) == bits(x0)
