"""GPU: per-env physics (BatchedSwarmEnv(physics=...), swarm_*_physics).

1. A table whose every row is SwarmParams' gives every output of the calls without a table, bit for bit.
2. An env of a mixed batch gives the bits of a one-env batch whose SwarmParams hold its row (env_id_offset = its id).
3. Teacher-forced steps and forces against the oracle with each env's own constants.
4. Resampling: rows equal the NumPy restatement, the burn-in used them, masks, shards, graph replay, terminal outputs.
5. An edited row changes that env only.  6. Production shapes under graph replay.  7. Facade and PAAC.
"""
import numpy as np
import pytest
import torch

from oracle import swarm_oracle as so

from _env_physics import COLUMNS, DEFAULT_ROW, random_rows, resampled_rows, step_with
from _util import rel_err

pytestmark = pytest.mark.gpu

STEP_TOL, RTOL = 5e-6, 1e-5
OUTPUTS = ("x", "xa", "reward", "done_u8", "elapsed", "episode", "noise_x", "noise_a", "grid", "positions")


@pytest.fixture(scope="module")
def M(pkg, cuda):
    return pkg.submodule("envs.multiagent")


def bits(t):
    return t.detach().cpu().numpy().tobytes()


def actions(E, A, gen):
    a = torch.randn(E, A, 2, device="cuda", generator=gen)
    n = a.norm(dim=-1, keepdim=True)
    return torch.where(n >= 1.0, a / n, a).contiguous()


def gen_of(seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return g


def same_range():
    """A resampling dict whose every range is the class constant: lo == hi, so every draw is exactly SwarmParams'."""
    return {c: (float(v), float(v)) for c, v in zip(COLUMNS, DEFAULT_ROW)}


# ---------------------------------------------------------------------------------------------------- 1. uniform table
def uniform_twins(M, E, N, steps=6, limit=3, draws=False, final_obs=False, physics="table", **kw):
    mk = lambda **k: M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=limit, seed=31, final_obs=final_obs,
                                       **dict(kw, **k))
    A, B = mk(physics=physics), mk()
    assert torch.equal(A.physics, torch.tensor(DEFAULT_ROW, device="cuda").expand(E, 6))
    A.reset()
    B.reset()
    for k in OUTPUTS[:2] + OUTPUTS[4:8]:
        assert bits(getattr(A, k)) == bits(getattr(B, k)), k
    A.stagger_episodes()
    B.stagger_episodes()
    rd = A.philox_draws() if draws else None
    gen = gen_of(N + E)
    vA = torch.zeros(E, N, 2, device="cuda")
    vB = torch.zeros(E, N, 2, device="cuda")
    n_done = 0
    for _ in range(steps):
        a = actions(E, A.A, gen)
        _, _, _, iA = A.step(a.clone(), reset_draws=rd, v_out=vA)
        _, _, d, iB = B.step(a.clone(), reset_draws=rd, v_out=vB)
        torch.cuda.synchronize()
        for k in OUTPUTS:
            assert bits(getattr(A, k)) == bits(getattr(B, k)), k
        assert bits(vA) == bits(vB)
        if final_obs:
            for k in iB:
                assert (iA[k] is None) == (iB[k] is None) and (iB[k] is None or bits(iA[k]) == bits(iB[k])), k
        n_done += int(d.sum())
    fA, rA = A.forces()
    fB, rB = B.forces()
    assert bits(fA) == bits(fB) and bits(rA) == bits(rB)
    assert torch.equal(A.physics, torch.tensor(DEFAULT_ROW, device="cuda").expand(E, 6))
    return n_done


@pytest.mark.parametrize("binding", ["torch", "ctypes"])
@pytest.mark.parametrize("N,tuning", [(64, 0x20), (64, 0x30), (80, 0), (80, 0x10), (80, 0x20), (80, 0x30),
                                      (256, 0), (256, 0x10), (256, 0x30), (700, 0), (1100, 0)])
def test_uniform_table_every_placement(M, binding, N, tuning):
    assert uniform_twins(M, 37, N, tuning=tuning, binding=binding) > 0


@pytest.mark.parametrize("math,noise,draws,final_obs", [("precise", "frozen", False, True), ("fast", "fresh", True, False),
                                                        ("precise", "fresh", True, True), ("fast", "frozen", False, True)])
@pytest.mark.parametrize("N", [64, 80, 256])
def test_uniform_table_math_noise_draws_final(M, N, math, noise, draws, final_obs):
    assert uniform_twins(M, 29, N, math_mode=math, noise=noise, draws=draws, final_obs=final_obs) > 0


@pytest.mark.parametrize("N,cluster,math,noise", [(700, 2, "fast", "frozen"), (700, 2, "precise", "fresh"),
                                                  (2049, None, "fast", "frozen"), (2049, None, "precise", "fresh")])
@pytest.mark.parametrize("binding", ["torch", "ctypes"])
def test_uniform_table_cluster(M, N, cluster, math, noise, binding):
    assert uniform_twins(M, 7, N, steps=4, cluster=cluster, math_mode=math, noise=noise, binding=binding,
                         draws=binding == "ctypes", final_obs=binding == "torch") > 0


@pytest.mark.parametrize("N,kw", [(80, {}), (256, dict(tuning=0x20)), (700, dict(cluster=2))])
def test_resampling_with_fixed_ranges_is_no_table(M, N, kw):
    """lo == hi everywhere: every reset draws exactly SwarmParams' row, so the resampling kernels give the same bits."""
    assert uniform_twins(M, 19, N, physics=same_range(), **kw) > 0


# ------------------------------------------------------------------------------------------------ 2. mixed batch
def single_env(M, row, e, N, **kw):
    env = M.BatchedSwarmEnv(1, n_locusts=N, env_id_offset=e, **kw)
    for c, v in zip(COLUMNS, row):
        setattr(env.params, c, float(v))
    return env


@pytest.mark.parametrize("N,kw", [(80, dict(tuning=0x10)), (80, dict(tuning=0x20)), (80, dict(tuning=0x30)),
                                  (80, {}), (256, {}), (256, dict(tuning=0x20)), (64, dict(tuning=0x30)),
                                  (700, dict(cluster=2)), (2049, {})])
def test_mixed_batch_equals_single_row_batches(M, N, kw):
    E, limit, steps = 24, 4, 9
    rows = random_rows(E, np.random.RandomState(N))
    base = dict(max_episode_steps=limit, seed=5, **kw)
    A = M.BatchedSwarmEnv(E, n_locusts=N, physics="table", **base)
    A.physics.copy_(torch.as_tensor(rows))
    sample = [0, 5, 13, E - 1]
    singles = [single_env(M, rows[e], e, N, **base) for e in sample]
    A.reset()
    for s in singles:
        s.reset()
    gen = gen_of(1)
    n_done = 0
    for step in range(steps):
        a = actions(E, A.A, gen)
        A.step(a.clone())
        for e, s in zip(sample, singles):
            s.step(a[e:e + 1].clone())
        torch.cuda.synchronize()
        for e, s in zip(sample, singles):
            for k in OUTPUTS:
                assert bits(getattr(A, k)[e:e + 1]) == bits(getattr(s, k)), (step, e, k)
        n_done += int(A.done_u8.sum())
    assert n_done > 0 and int(A.episode.max()) >= 3
    v, r = A.forces()
    for e, s in zip(sample, singles):
        vs, rs = s.forces()
        assert bits(v[e:e + 1]) == bits(vs) and bits(r[e:e + 1]) == bits(rs)


# ------------------------------------------------------------------------------------------------ 3. oracle
@pytest.mark.parametrize("math", ["fast", "precise"])
@pytest.mark.parametrize("E,N", [(1, 64), (32, 64), (1, 80), (32, 80), (1, 256), (32, 256)])
def test_teacher_forced_steps_and_forces_vs_oracle(M, E, N, math):
    rows = random_rows(E, np.random.RandomState(E * 1000 + N))
    env = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=0, seed=8, math_mode=math, rasterize=False,
                            physics="table")
    env.physics.copy_(torch.as_tensor(rows))
    env.reset()
    gen = gen_of(3)
    for step in range(16):
        x0, xa0 = env.x.cpu().numpy(), env.xa.cpu().numpy()
        na, nx = env.noise_a.cpu().numpy(), env.noise_x.cpu().numpy()
        a = actions(E, env.A, gen)
        env.step(a)
        gx, gxa, gr = env.x.cpu().numpy(), env.xa.cpu().numpy(), env.reward.cpu().numpy()
        ah = a.cpu().numpy().astype(np.float64)
        for e in range(E):
            x, xa = x0[e:e + 1].copy(), xa0[e:e + 1].copy()
            rew, _ = step_with(x, xa, ah[e:e + 1], na[e:e + 1], nx[e:e + 1], rows[e])
            assert rel_err(gxa[e], xa[0]) <= 1e-12, (step, e)
            assert rel_err(gx[e], x[0]) <= STEP_TOL, (step, e)
            assert abs(gr[e] - rew[0]) <= RTOL * abs(rew[0]), (step, e)
    v, r = env.forces()
    vh, rh = v.cpu().numpy(), r.cpu().numpy()
    xh, xah = env.x.cpu().numpy(), env.xa.cpu().numpy()
    for e in range(E):
        _, _, wind, F, L, _ = rows[e]
        v_ref, r_ref = so.forces(xh[e:e + 1], xah[e:e + 1], F, L, wind, rows[e][1])
        assert np.abs(vh[e] - v_ref[0]).max() <= 1e-5 * np.abs(v_ref[0]).max(), e
        assert abs(rh[e] - r_ref[0]) <= RTOL * abs(r_ref[0]), e


# ------------------------------------------------------------------------------------------------ 4. resampling
RANGES = {"F": (0.2, 0.9), "L": (2.0, 20.0), "wind": (-2.0, 2.0), "gravity": (-2.0, 0.5), "dt": (0.01, 0.1),
          "noise": (0.0, 1e-3)}


def expect_rows(env, ids, episodes):
    lo, hi = np.array(env._phys_lo), np.array(env._phys_hi)
    g = np.asarray(ids) + int(env.params.env_id_offset)
    return resampled_rows(int(env.params.seed), g, episodes, lo, hi)


@pytest.mark.parametrize("N,kw", [(80, {}), (80, dict(tuning=0x20)), (80, dict(tuning=0x30)), (256, {}),
                                  (64, dict(tuning=0x20)), (700, dict(cluster=2)), (2049, {}),
                                  (80, dict(binding="ctypes", noise="fresh"))])
def test_resample_rows_burn_in_and_masks(M, N, kw):
    E, limit = 33, 3
    mk = lambda **k: M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=limit, seed=71, **dict(kw, **k))
    A = mk(physics=dict(RANGES, L=(5.0, 15.0)))
    B = mk(physics="table")                      # resampling off: the reference for the burn-in
    A.reset()
    assert np.array_equal(A.physics.cpu().numpy(), expect_rows(A, range(E), np.zeros(E)))
    A.stagger_episodes()
    gen = gen_of(4)
    for _ in range(5):
        before = A.state_dict()
        a = actions(E, A.A, gen)
        A.step(a)
        d = A.done_u8.bool()
        torch.cuda.synchronize()
        tab, old = A.physics.cpu().numpy(), before["physics"].cpu().numpy()
        dn = d.cpu().numpy()
        assert dn.any()
        assert np.array_equal(tab[dn], expect_rows(A, np.nonzero(dn)[0], before["episode"].cpu().numpy()[dn]))
        assert tab[~dn].tobytes() == old[~dn].tobytes()
        # the auto-reset's burn-in ran with the new row: an explicit reset of the done envs with it preset
        B.load_state_dict(dict(before, physics=A.physics.clone()))
        B.reset(mask=d)
        torch.cuda.synchronize()
        for k in ("x", "xa", "noise_x", "noise_a", "episode"):
            assert bits(getattr(B, k)[d]) == bits(getattr(A, k)[d]), k
    # a masked reset redraws the masked rows only
    mask = torch.zeros(E, dtype=torch.bool, device="cuda")
    mask[::3] = True
    before = A.state_dict()
    A.reset(mask=mask)
    m = mask.cpu().numpy()
    tab, old = A.physics.cpu().numpy(), before["physics"].cpu().numpy()
    assert np.array_equal(tab[m], expect_rows(A, np.nonzero(m)[0], before["episode"].cpu().numpy()[m]))
    assert tab[~m].tobytes() == old[~m].tobytes()
    assert ((tab >= np.array(A._phys_lo)) & (tab <= np.array(A._phys_hi))).all()


@pytest.mark.parametrize("N,kw", [(80, {}), (256, {}), (700, dict(cluster=2))])
def test_resample_shards_equal_whole_batch(M, N, kw):
    E, limit = 40, 3
    base = dict(n_locusts=N, max_episode_steps=limit, seed=12, physics=RANGES, **kw)
    W = M.BatchedSwarmEnv(E, **base)
    S = [M.BatchedSwarmEnv(E // 2, env_id_offset=o, **base) for o in (0, E // 2)]
    W.reset()
    W.stagger_episodes()
    for s in S:
        s.reset()
        s.stagger_episodes(total_envs=E)
    gen = gen_of(6)
    for _ in range(4):
        a = actions(E, W.A, gen)
        W.step(a.clone())
        S[0].step(a[:E // 2].clone())
        S[1].step(a[E // 2:].clone())
    torch.cuda.synchronize()
    assert int(W.episode.max()) >= 2
    for k in OUTPUTS + ("physics",):
        assert bits(getattr(W, k)) == bits(torch.cat([getattr(s, k) for s in S])), k


@pytest.mark.parametrize("N", [80, 256])
def test_resample_graph_replay_equals_eager(M, N):
    E = 48
    base = dict(n_locusts=N, max_episode_steps=2, seed=21, physics=RANGES)
    G, R = M.BatchedSwarmEnv(E, **base), M.BatchedSwarmEnv(E, **base)
    for env in (G, R):
        env.reset()
    a = actions(E, G.A, gen_of(2))
    G.step(a)                                           # warm-up outside the capture
    R.step(a)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        G.step(a)
    for _ in range(4):                                  # every second step auto-resets every env
        g.replay()
        R.step(a)
    torch.cuda.synchronize()
    assert int(R.episode.min()) >= 3
    for k in OUTPUTS + ("physics",):
        assert bits(getattr(G, k)) == bits(getattr(R, k)), k


@pytest.mark.parametrize("N,kw", [(80, {}), (256, {}), (700, dict(cluster=2))])
def test_resample_final_obs_is_old_physics(M, N, kw):
    """The terminal state is the old episode's physics; the table already holds the new row."""
    E, limit = 24, 3
    A = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=limit, seed=4, physics=RANGES, final_obs=True, **kw)
    C = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=limit, seed=4, physics="table", auto_reset=False, **kw)
    A.reset()
    A.stagger_episodes()
    gen = gen_of(9)
    n_done = 0
    for _ in range(4):
        before = A.state_dict()
        C.load_state_dict(before)
        a = actions(E, A.A, gen)
        _, _, d, info = A.step(a.clone())
        C.step(a.clone())
        gC, pC = [t.clone() for t in C.observe()]
        torch.cuda.synchronize()
        d = d.clone()
        for k, ref in (("final_x", C.x), ("final_xa", C.xa), ("final_grid", gC), ("final_positions", pC)):
            assert bits(info[k][d]) == bits(ref[d]), k
        assert torch.equal(A.reward, C.reward)
        dn = d.cpu().numpy()
        assert np.array_equal(A.physics.cpu().numpy()[dn],
                              expect_rows(A, np.nonzero(dn)[0], before["episode"].cpu().numpy()[dn]))
        n_done += int(dn.sum())
    assert n_done > 0


# ------------------------------------------------------------------------------------------------ 5. editable table
@pytest.mark.parametrize("N,kw", [(80, {}), (256, dict(tuning=0x20)), (700, dict(cluster=2))])
def test_edited_row_changes_that_env_only(M, N, kw):
    E = 16
    A, B = [M.BatchedSwarmEnv(E, n_locusts=N, seed=2, physics="table", **kw) for _ in range(2)]
    A.reset()
    B.reset()
    gen = gen_of(5)
    a = actions(E, A.A, gen)
    A.step(a.clone())
    B.step(a.clone())
    A.physics[3, 3] = 0.8                               # F of env 3, between two steps
    A.physics[3, 2] = -0.5                              # and its wind
    a = actions(E, A.A, gen)
    A.step(a.clone())
    B.step(a.clone())
    torch.cuda.synchronize()
    keep = torch.ones(E, dtype=torch.bool, device="cuda")
    keep[3] = False
    for k in ("x", "xa", "reward", "grid", "positions"):
        assert bits(getattr(A, k)[keep]) == bits(getattr(B, k)[keep]), k
    assert not torch.equal(A.x[3], B.x[3]) and not torch.equal(A.xa[3], B.xa[3])


# ------------------------------------------------------------------------------------------------ 6. production shapes
@pytest.mark.parametrize("E,N", [(4096, 256), (1024, 64)])
def test_production_shape_resampling_graph_replay_vs_oracle(M, E, N):
    env = M.BatchedSwarmEnv(E, n_locusts=N, seed=4242, max_episode_steps=2, physics=RANGES)
    env.reset()
    gen = gen_of(7)
    acts = [actions(E, 10, gen) for _ in range(3)]
    env.step(acts[0])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g_reset, g_last = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_reset, stream=side):
        env.step(acts[1])                               # every env ends and redraws its row
    with torch.cuda.graph(g_last, stream=side):
        env.step(acts[2])
    g_reset.replay()
    torch.cuda.synchronize()
    assert env.done_u8.all() and (env.episode == 2).all()
    sample = np.unique(np.linspace(0, E - 1, 32).astype(int))
    rows = env.physics.cpu().numpy()
    assert np.array_equal(rows[sample], expect_rows(env, sample, np.ones(len(sample))))
    x0, xa0 = env.x[sample].cpu().numpy(), env.xa[sample].cpu().numpy()
    na, nx = env.noise_a[sample].cpu().numpy(), env.noise_x[sample].cpu().numpy()
    g_last.replay()
    torch.cuda.synchronize()
    gx, gxa, gr = env.x[sample].cpu().numpy(), env.xa[sample].cpu().numpy(), env.reward[sample].cpu().numpy()
    ah = acts[2][sample].cpu().numpy().astype(np.float64)
    for i, e in enumerate(sample):
        x, xa = x0[i:i + 1].copy(), xa0[i:i + 1].copy()
        rew, _ = step_with(x, xa, ah[i:i + 1], na[i:i + 1], nx[i:i + 1], rows[e])
        assert rel_err(gxa[i], xa[0]) <= 1e-12 and rel_err(gx[i], x[0]) <= STEP_TOL, e
        assert abs(gr[i] - rew[0]) <= RTOL * abs(rew[0]), e
        g, p = so.rasterize(gx[i], gxa[i], 84)
        assert np.array_equal(env.grid[e].cpu().numpy(), g.astype(np.float32)), e
    assert not env.done_u8.any() and int(env.work.sum()) == 0


# ------------------------------------------------------------------------------------------------ 7. facade and PAAC
def test_bindings_state_dict_plan_and_step_host(M):
    E, N = 20, 80
    T, C = [M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=3, seed=6, physics=RANGES, binding=b, final_obs=True)
            for b in ("torch", "ctypes")]
    for env in (T, C):
        env.reset()
    gen = gen_of(8)
    for _ in range(4):
        a = actions(E, T.A, gen)
        _, _, _, iT = T.step(a.clone())
        _, _, _, iC = C.step(a.clone())
        for k in OUTPUTS + ("physics",):
            assert bits(getattr(T, k)) == bits(getattr(C, k)), k
        for k in iT:
            assert bits(iT[k]) == bits(iC[k]), k
    sd = T.state_dict()
    assert "physics" in sd and torch.equal(sd["physics"], T.physics)
    R = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=3, seed=6, physics=RANGES)
    R.load_state_dict(sd)
    a = actions(E, T.A, gen)
    T.step(a.clone())
    R.step(a.clone())
    for k in OUTPUTS + ("physics",):
        assert bits(getattr(T, k)) == bits(getattr(R, k)), k
    # plan(): the PHYS kernels carry a physics row per stage buffer behind their shared memory
    for tuning in (0x20, 0x30):
        pp = M.BatchedSwarmEnv(E, n_locusts=N, physics="table", tuning=tuning).plan()
        p0 = M.BatchedSwarmEnv(E, n_locusts=N, tuning=tuning).plan()
        stages = 2 if tuning == 0x20 else 1
        assert pp["smem_bytes"] == p0["smem_bytes"] + 48 * stages and pp["threads"] == p0["threads"]
    host = [torch.zeros(E, 10, 2).pin_memory(), torch.zeros(E).pin_memory(), torch.zeros(E, dtype=torch.uint8).pin_memory()]
    with pytest.raises(ValueError, match="physics"):
        T.step_host(*host)
    with pytest.raises(ValueError):
        M.BatchedSwarmEnv(4, physics={"G": (0, 1)})
    with pytest.raises(RuntimeError, match="-2"):         # lo > hi: SWARM_ERR_SIZE from the library before any launch
        M.BatchedSwarmEnv(4, physics={"F": (0.7, 0.3)}).reset()


def make_learner(pkg, graph=False, **kw):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import train_paac_conv as tp
    args = tp.get_arg_parser().parse_args(["--clip_norm", "1", "-ec", "8", "--n_locusts", "16",
                                           "--physics", "F=0.3:0.7,L=5:15,wind=0.5:1.5"])
    net_creator, env_creator = tp.get_network_and_environment_creator(args)
    paac = pkg.submodule("agents.paac.paac")
    return paac.GridPAACLearner(net_creator, env_creator, args, use_cuda_graph=graph, **kw)


def test_paac_learner_with_physics_ranges(pkg, cuda):
    L = make_learner(pkg, compact_obs=True)
    L.start()
    rows = L.env.physics.cpu().numpy()
    assert len(np.unique(rows[:, 3])) == len(rows) and (rows[:, 3] >= 0.3).all() and (rows[:, 3] <= 0.7).all()
    assert (rows[:, 0] == so.NOISE).all() and (rows[:, 5] == so.DT).all()
    before = torch.cat([p.detach().flatten().clone() for p in L.network.parameters()])
    for _ in range(2):
        L.update()
    torch.cuda.synchronize()
    after = torch.cat([p.detach().flatten() for p in L.network.parameters()])
    assert torch.isfinite(after).all() and not torch.equal(before, after)
    G = make_learner(pkg, graph=True, compact_obs=True)
    G.initial_lr = 0.0
    G.start()
    for _ in range(2):
        G.update()
    torch.cuda.synchronize()
    assert G._graph is not None
    y = G.y_batch.clone()
    with torch.no_grad():
        G._returns()
    torch.cuda.synchronize()
    assert torch.equal(y, G.y_batch)
