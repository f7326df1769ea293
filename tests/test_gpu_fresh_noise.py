"""GPU tests of fresh per-step noise (SWARM_STEP_FRESH_NOISE; BatchedSwarmEnv(noise="fresh"), SwarmEnv(fresh_noise=True)):
the reference with SURVEY Q1 fixed.  Step k of an episode uses Philox row N_BURN_IN + k of noise streams 3 / 4, drawn in
the step kernel; swarm_philox_noise_rows exports the same rows, and the oracle is fed them.

Tolerances as in test_gpu_parity.py: teacher-forced states within STEP_TOL (max|a-b| <= 5e-6 max|b| per env), agents
exact, rewards rtol 1e-5, done / elapsed / episode exact; every launch shape, sharding and graph replay bitwise."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import swarm_oracle as so

from _fresh_noise import FreshOracleRunner, draw_reset_full, noise_rows
from _util import golden, rel_err

pytestmark = pytest.mark.gpu

RTOL = 1e-5
STEP_TOL = 5e-6
NB = so.N_BURN_IN
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def M(pkg, cuda):
    return pkg.submodule("envs.multiagent")


def clipped(rs, shape):
    a = rs.normal(size=shape).astype(np.float32).astype(np.float64)
    so.clip_actions_(a.reshape(-1, 2))
    return a.astype(np.float32)


def to_dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


def host(*ts):
    return [t.cpu().numpy() for t in ts]


def rows_host(env, row0, n_rows):
    return host(*env.philox_noise_rows(row0, n_rows))


# --------------------------------------------------------------------------------------- export
def test_noise_rows_export_matches_reset_rows_and_restatement(M):
    E, N, seed, off = 8, 80, 4711, 3
    env = M.BatchedSwarmEnv(E, n_locusts=N, seed=seed, env_id_offset=off, noise="fresh")
    for episode in range(2):
        env.reset()
        an, pn = env.philox_noise_rows(0, 128 + NB)
        assert an.shape == (E, 128 + NB, 10, 2) and pn.shape == (E, 128 + NB, N, 2)
        assert torch.equal(an[:, NB], env.noise_a) and torch.equal(pn[:, NB], env.noise_x)    # the frozen row, bitwise
        a2, p2 = env.philox_noise_rows(NB + 7, 3)                                            # any window: same bits
        assert torch.equal(a2, an[:, NB + 7:NB + 10]) and torch.equal(p2, pn[:, NB + 7:NB + 10])
        han, hpn = host(an, pn)
        for e in range(E):
            ra, rp = noise_rows(seed, off + e, episode, 0, 128 + NB, N)
            assert np.abs(han[e] - ra).max() <= 2e-6 and np.abs(hpn[e] - rp).max() <= 2e-6    # FP32 Box-Muller
        tail = hpn[:, NB:]
        assert abs(tail.mean()) < 0.01 and abs(tail.std() - 1.0) < 0.01
        assert abs(han[:, NB:].mean()) < 0.03 and abs(han[:, NB:].std() - 1.0) < 0.03
        if episode == 0:
            first = an.clone()
    assert not torch.equal(first, an)                     # the next episode has its own rows


# --------------------------------------------------------------------------------------- dynamics
@pytest.mark.parametrize("mode", ["fast", "precise"])
@pytest.mark.parametrize("N", [64, 80, 256])
@pytest.mark.parametrize("E", [1, 32])
def test_fresh_step_teacher_forced_16(M, E, N, mode):
    """Every one of 16 fresh-noise steps starts from the ORACLE state; the oracle is fed the exported row 10 + t."""
    env = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=0, math_mode=mode, auto_reset=False, rasterize=False,
                            seed=900 + N, noise="fresh")
    env.reset()
    an, pn = rows_host(env, NB, 16)
    x, xa = host(env.x, env.xa)
    rs = np.random.RandomState(99)
    for t in range(16):
        a = clipped(rs, (E, 10, 2))
        env.x.copy_(to_dev(x)); env.xa.copy_(to_dev(xa))
        (gx, gxa), r, d, _ = env.step(to_dev(a))
        rew, done = so.step(x, xa, a.astype(np.float64), an[:, t], pn[:, t])     # advances the oracle in place
        gx, gxa, r, d = host(gx, gxa, r, d)
        assert np.array_equal(gxa, xa), "agent update is FP64 and must be exact"
        for e in range(E):
            assert rel_err(gx[e], x[e]) <= STEP_TOL, (t, e, rel_err(gx[e], x[e]))
        assert np.all(np.abs(r - rew) <= RTOL * np.abs(rew))
        assert np.array_equal(d, done)
        assert (env.elapsed == t + 1).all()


def test_first_step_equal_then_rows_advance(M):
    """After a Philox reset the first step is bitwise the frozen mode's (both use row 10); the second is not."""
    E, N = 16, 80
    frozen = M.BatchedSwarmEnv(E, n_locusts=N, seed=31)
    fresh = M.BatchedSwarmEnv(E, n_locusts=N, seed=31, noise="fresh")
    frozen.reset(); fresh.reset()
    rs = np.random.RandomState(1)
    acts = [to_dev(clipped(rs, (E, 10, 2))) for _ in range(2)]
    frozen.step(acts[0].clone()); fresh.step(acts[0].clone())
    for k in ("x", "xa", "grid", "positions", "reward", "elapsed", "episode"):
        assert torch.equal(getattr(frozen, k), getattr(fresh, k)), k
    frozen.step(acts[1].clone()); fresh.step(acts[1].clone())
    a, b = host(frozen.x, fresh.x)
    for e in range(E):
        assert rel_err(b[e], a[e]) > 4 * STEP_TOL, e
    assert not torch.equal(frozen.xa, fresh.xa)


@pytest.mark.parametrize("N", [40, 64, 80, 128, 176, 256, 320, 512, 700])
def test_fresh_launch_shapes_bitwise_identical(M, N):
    """Fresh noise in every launch shape (follower kernel, raster warps, the step's own threads, automatic), across an
    auto-reset inside the step kernel (limit 3): the same BITS; sampled envs against the oracle on the last step."""
    nat = M.nat
    E = 21
    ref = None
    rs = np.random.RandomState(N)
    acts = [to_dev(clipped(rs, (E, 10, 2))) for _ in range(5)]
    sample = list(range(0, E, 5))
    for place in (nat.TUNE_RASTER_WARPS, nat.TUNE_RASTER_SELF, nat.TUNE_RASTER_FOLLOW, 0):
        env = M.BatchedSwarmEnv(E, n_locusts=N, seed=77, max_episode_steps=3, tuning=place, noise="fresh")
        env.reset()
        outs = []
        for t in range(5):
            if t == 4:                                  # elapsed 1 of the second episode: row 11 of episode word 1
                x0, xa0, el = host(env.x, env.xa, env.elapsed)
                an, pn = rows_host(env, NB, 3)
            env.step(acts[t].clone())
            outs += [env.x.clone(), env.xa.clone(), env.grid.clone(), env.positions.clone(), env.reward.clone(),
                     env.done_u8.clone(), env.episode.clone(), env.elapsed.clone()]
        torch.cuda.synchronize()
        assert int(env.work.sum()) == 0
        if ref is None:
            ref = outs
            assert (el == 1).all() and (env.episode == 2).all()
            gx, gxa = host(env.x, env.xa)
            a = acts[4].cpu().numpy().astype(np.float64)
            for e in sample:
                x, xa = x0[e:e + 1].copy(), xa0[e:e + 1].copy()
                rew, _ = so.step(x, xa, a[e:e + 1], an[e:e + 1, el[e]], pn[e:e + 1, el[e]])
                assert rel_err(gx[e], x[0]) <= STEP_TOL, (N, e)
                assert np.array_equal(gxa[e], xa[0])
                assert abs(float(env.reward[e]) - rew[0]) <= RTOL * abs(rew[0])
                g, p_ = so.rasterize(gx[e], gxa[e], 84)
                assert np.array_equal(env.grid[e].cpu().numpy(), g.astype(np.float32))
                assert np.array_equal(env.positions[e].cpu().numpy(), p_)
        else:
            for i, (a_, b_) in enumerate(zip(ref, outs)):
                assert torch.equal(a_, b_), (N, place >> 4, i)


def test_fresh_autoreset_timelimit_matches_oracle_runner(M):
    """E=64, N=80, TimeLimit 5, 17 steps with Philox resets inside the step kernel.  Every episode's draws (exported
    with philox_draws before it starts, its noise rows with philox_noise_rows after) are injected into
    FreshOracleRunner; done / elapsed / episode exact on every step, every step teacher-forced."""
    E, N, LIM = 64, 80, 5
    env = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=LIM, seed=2024, noise="fresh")
    table = {}

    def record(inj, ep_before, which):
        an, pn = rows_host(env, 0, NB + LIM)
        for e in which:
            table[(e, int(ep_before[e]))] = (inj[0][e], inj[1][e], inj[2][e], an[e], pn[e])

    inj = host(*env.philox_draws().tensors())
    env.reset()
    record(inj, np.zeros(E, dtype=np.int64), range(E))
    orc = FreshOracleRunner(E, N, lambda e, ep: table[(e, ep)], grid_size=84, max_episode_steps=LIM)
    orc.reset()
    rs = np.random.RandomState(8)
    for t in range(17):
        a = clipped(rs, (E, 10, 2))
        inj = host(*env.philox_draws().tensors())       # what the resets inside this step will draw
        ep_before = env.episode.cpu().numpy().copy()
        orc.x[...], orc.xa[...] = host(env.x, env.xa)   # teacher-forced: the burn-in is free-running and chaotic
        (gx, gxa), r, d, _ = env.step(to_dev(a))
        ep_after = env.episode.cpu().numpy()
        record(inj, ep_before, np.nonzero(ep_after != ep_before)[0])
        rew, done = orc.step(a.astype(np.float64))
        assert np.array_equal(d.cpu().numpy(), done), t
        assert np.array_equal(env.elapsed.cpu().numpy(), orc.elapsed), t
        assert np.array_equal(ep_after, orc.episode), t
        assert np.all(np.abs(r.cpu().numpy() - rew) <= RTOL * np.abs(rew)), t
        gx, gxa = host(gx, gxa)
        for e in np.nonzero(~done)[0]:
            assert rel_err(gx[e], orc.x[e]) <= STEP_TOL, (t, e)
            assert np.array_equal(gxa[e], orc.xa[e]), (t, e)
    assert orc.episode.min() == 4 and (env.elapsed == 2).all()


def test_fresh_noise_after_stagger_episodes(M):
    """stagger_episodes() puts the envs at different points of their episodes: env e's step uses row 10 + elapsed[e]."""
    E, N, LIM = 64, 80, 16
    env = M.BatchedSwarmEnv(E, n_locusts=N, seed=8, max_episode_steps=LIM, noise="fresh")
    env.reset()
    el = env.stagger_episodes().cpu().numpy().copy()
    assert len(set(el.tolist())) == LIM
    an, pn = rows_host(env, NB, LIM)
    x0, xa0 = host(env.x, env.xa)
    a = clipped(np.random.RandomState(4), (E, 10, 2))
    (gx, gxa), r, d, _ = env.step(to_dev(a))
    gx, gxa, r, d = host(gx, gxa, r, d)
    assert np.array_equal(d, el + 1 >= LIM)
    for e in range(E):
        x, xa = x0[e:e + 1].copy(), xa0[e:e + 1].copy()
        rew, _ = so.step(x, xa, a[e:e + 1].astype(np.float64), an[e:e + 1, el[e]], pn[e:e + 1, el[e]])
        assert abs(r[e] - rew[0]) <= RTOL * abs(rew[0]), e
        if not d[e]:
            assert rel_err(gx[e], x[0]) <= STEP_TOL, (e, el[e])
            assert np.array_equal(gxa[e], xa[0]), e


def test_fresh_shard_invariance_bitwise(M):
    """Global env ids key the fresh rows too: 8 envs on one 'rank' == 4+4 envs on two 'ranks', across an auto-reset."""
    N, seed = 64, 77
    whole = M.BatchedSwarmEnv(8, n_locusts=N, seed=seed, noise="fresh")
    parts = [M.BatchedSwarmEnv(4, n_locusts=N, seed=seed, env_id_offset=4 * r, noise="fresh") for r in range(2)]
    whole.reset()
    [p.reset() for p in parts]
    rs = np.random.RandomState(3)
    for t in range(130):                 # crosses the 128-step auto-reset
        a = to_dev(clipped(rs, (8, 10, 2)))
        whole.step(a)
        for r, p in enumerate(parts):
            p.step(a[4 * r:4 * r + 4].contiguous())
    for k in ("x", "xa", "grid", "positions", "reward", "elapsed", "episode"):
        cat = torch.cat([getattr(p, k) for p in parts])
        assert torch.equal(getattr(whole, k), cat), k
    assert whole.episode.cpu().tolist() == [2] * 8 and whole.elapsed.cpu().tolist() == [2] * 8


def test_fresh_step_under_cuda_graph_replay_equals_eager(M):
    """8 captured fresh-noise steps replayed 20 times == 160 eager steps, bitwise: the row comes from the device's
    elapsed counter, so it advances inside the replayed graph (and crosses the 128-step auto-reset)."""
    E, N = 64, 64
    acts = [torch.randn(E, 10, 2, device="cuda").clamp(-0.7, 0.7).contiguous() for _ in range(8)]
    a = M.BatchedSwarmEnv(E, n_locusts=N, seed=21, noise="fresh")
    b = M.BatchedSwarmEnv(E, n_locusts=N, seed=21, noise="fresh")
    a.reset(); b.reset()
    a.step(acts[0]); b.step(acts[0])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for i in range(8):
            a.step(acts[i])
    for _ in range(20):
        g.replay()
    for _ in range(20):
        for i in range(8):
            b.step(acts[i])
    torch.cuda.synchronize()
    for k in ("x", "xa", "elapsed", "episode", "grid", "positions", "reward", "done_u8"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
    assert int(a.episode[0]) == 2


def test_overrides_win_in_fresh_mode(M):
    """io->noise_a / io->noise_x override their own row in either mode: fresh + both overrides == frozen + the same
    overrides, bitwise; an override that repeats the exported fresh row changes nothing, and each override only
    replaces itself."""
    E, N = 16, 80
    gen = torch.Generator(device="cuda"); gen.manual_seed(5)
    envs = {k: M.BatchedSwarmEnv(E, n_locusts=N, seed=13, noise=k.split("_")[0])
            for k in ("frozen_both", "fresh_both", "fresh_none", "fresh_a", "fresh_x")}
    for env in envs.values():
        env.reset()
    for t in range(4):
        act = torch.randn(E, 10, 2, device="cuda", generator=gen).clamp(-0.7, 0.7).contiguous()
        na = torch.randn(E, 10, 2, device="cuda", dtype=torch.float64, generator=gen)
        nx = torch.randn(E, N, 2, device="cuda", dtype=torch.float64, generator=gen)
        envs["frozen_both"].step(act.clone(), noise_a=na, noise_x=nx)
        envs["fresh_both"].step(act.clone(), noise_a=na, noise_x=nx)
        envs["fresh_none"].step(act.clone())
        # the exported rows of the env's own step, given back as overrides, one at a time
        fa = envs["fresh_a"]
        el = int(fa.elapsed[0])
        assert (fa.elapsed == el).all()
        ra, _ = fa.philox_noise_rows(NB + el, 1)
        fa.step(act.clone(), noise_a=ra[:, 0].contiguous())
        fx = envs["fresh_x"]
        _, rx = fx.philox_noise_rows(NB + el, 1)
        fx.step(act.clone(), noise_x=rx[:, 0].contiguous())
        for k in ("x", "xa", "reward", "elapsed"):
            assert torch.equal(getattr(envs["frozen_both"], k), getattr(envs["fresh_both"], k)), (t, k)
            assert torch.equal(getattr(envs["fresh_none"], k), getattr(envs["fresh_a"], k)), (t, k)
            assert torch.equal(getattr(envs["fresh_none"], k), getattr(envs["fresh_x"], k)), (t, k)
    assert not torch.equal(envs["fresh_none"].x, envs["fresh_both"].x)


@pytest.mark.parametrize("pinned", [True, False])
def test_fresh_step_host_matches_device_step(M, pinned):
    """swarm_step_host (pinned: zero-copy, pageable: staged copies) with fresh noise == the device step, across an
    auto-reset (TimeLimit 3); step 2 of the episode differs from the frozen mode."""
    E, N = 300, 64
    a = M.BatchedSwarmEnv(E, n_locusts=N, seed=5, max_episode_steps=3, noise="fresh")
    b = M.BatchedSwarmEnv(E, n_locusts=N, seed=5, max_episode_steps=3, noise="fresh")
    c = M.BatchedSwarmEnv(E, n_locusts=N, seed=5, max_episode_steps=3)
    a.reset(); b.reset(); c.reset()
    pin = (lambda t: t.pin_memory()) if pinned else (lambda t: t)
    h_act = pin(torch.randn(E, 10, 2).clamp_(-0.5, 0.5))
    h_rew = pin(torch.zeros(E))
    h_done = pin(torch.zeros(E, dtype=torch.uint8))
    for t in range(4):                                  # step 3 auto-resets every env
        a.step_host(h_act, h_rew, h_done)
        _, r, d, _ = b.step(h_act.cuda())
        c.step(h_act.cuda())
        torch.cuda.synchronize()
        assert torch.equal(h_rew, r.cpu()) and torch.equal(h_done.bool(), d.cpu())
        assert bool(d.all()) == (t == 2)
        assert torch.equal(a.x, b.x) and torch.equal(a.grid, b.grid)
        assert torch.equal(b.x, c.x) == (t != 1), t    # rows 10 | 11 | reset | 10 of the new episode


# --------------------------------------------------------------------------------------- production shapes
@pytest.mark.parametrize("E,N", [(4096, 256), (1024, 64), (512, 256)])
def test_fresh_production_shape_graph_replay_vs_oracle(M, E, N):
    """Graph-replayed fresh-noise steps of the production batch (automatic launch shape) with TimeLimit 3: a step at
    elapsed 1 (row 11), the auto-reset step, and the first step of the new episode (row 10 of the new episode word),
    32 sampled envs teacher-forced against the oracle with the exported rows."""
    env = M.BatchedSwarmEnv(E, n_locusts=N, seed=4242, max_episode_steps=3, noise="fresh")
    env.reset()
    gen = torch.Generator(device="cuda"); gen.manual_seed(7)
    acts = []
    for _ in range(4):
        a = torch.randn(E, 10, 2, device="cuda", generator=gen)
        n = a.norm(dim=-1, keepdim=True)
        acts.append(torch.where(n >= 1.0, a / n, a).contiguous())
    env.step(acts[0])                                   # warm-up outside the capture; elapsed = 1
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graphs = [torch.cuda.CUDAGraph() for _ in range(3)]
    for g, a in zip(graphs, acts[1:]):
        with torch.cuda.graph(g, stream=side):
            env.step(a)
    sample = np.unique(np.linspace(0, E - 1, 32).astype(int))

    def forced_step(g, a):
        el = env.elapsed[sample].cpu().numpy()
        assert (el == el[0]).all()
        an, pn = env.philox_noise_rows(NB + int(el[0]), 1)
        na, nx = an[sample, 0].cpu().numpy(), pn[sample, 0].cpu().numpy()
        x0, xa0 = host(env.x[sample], env.xa[sample])
        g.replay()
        torch.cuda.synchronize()
        rew, _ = so.step(x0, xa0, a[sample].cpu().numpy().astype(np.float64), na, nx)
        gx, gxa = host(env.x[sample], env.xa[sample])
        assert np.array_equal(gxa, xa0)
        for i in range(len(sample)):
            assert rel_err(gx[i], x0[i]) <= STEP_TOL, sample[i]
            g_, p_ = so.rasterize(gx[i], gxa[i], 84)
            assert np.array_equal(env.grid[sample[i]].cpu().numpy(), g_.astype(np.float32)), sample[i]
            assert np.array_equal(env.positions[sample[i]].cpu().numpy(), p_), sample[i]
        r = env.reward[sample].cpu().numpy()
        assert np.all(np.abs(r - rew) <= RTOL * np.abs(rew))

    forced_step(graphs[0], acts[1])                     # elapsed 1 -> 2: row 11
    assert not env.done_u8.any() and (env.elapsed == 2).all()
    graphs[1].replay()                                  # elapsed 3: done, auto-reset inside the kernel
    torch.cuda.synchronize()
    assert env.done_u8.all() and (env.elapsed == 0).all() and (env.episode == 2).all()
    an, pn = env.philox_noise_rows(NB, 1)
    assert torch.equal(an[:, 0], env.noise_a) and torch.equal(pn[:, 0], env.noise_x)
    forced_step(graphs[2], acts[3])                     # first step of the new episode: row 10
    assert not env.done_u8.any() and (env.elapsed == 1).all() and int(env.work.sum()) == 0


# --------------------------------------------------------------------------------------- facade / PAAC
def test_fresh_facade_matches_fixed_reference(M):
    """make('Swarm-eval-v0', fresh_noise=True) against the reference with its frozen index fixed (the oracle fed row
    10 + t of the same 138-row tables; tests/test_fresh_noise_oracle.py pins that restatement against the reference
    itself), seed 192, the C1 golden actions: steps 1-8 within rtol 1e-5, 9-16 inside the 1e-3 chaos envelope.  The
    frozen facade is off at step 2 by far more, so the check tells the modes apart."""
    d = golden("c1_seed192_n80.npz")
    fresh = M.make("Swarm-eval-v0", fresh_noise=True)
    frozen = M.make("Swarm-eval-v0")
    st = fresh.reset()
    assert fresh.t == NB
    np.random.seed(192)
    draws = draw_reset_full(np.random, 80)
    x, xa = so.reset_injected(*[t[None] for t in draws])
    assert rel_err(st[0], x[0]) <= RTOL and rel_err(st[1], xa[0]) <= 1e-12
    frozen.reset()
    for t in range(16):
        a = d["actions"][t]
        st, r, done, _ = fresh.step(a)
        fst, _, _, _ = frozen.step(a)
        rew, _ = so.step(x, xa, a[None], draws[3][NB + t][None], draws[4][NB + t][None])
        assert fresh.t == NB + t + 1 and frozen.t == NB and not done
        err = rel_err(st[0], x[0])
        assert err <= (RTOL if t < 8 else 1e-3), (t, err)
        if t < 8:
            assert abs(r - rew[0]) <= RTOL * abs(rew[0]), t
        if t == 1:
            assert rel_err(fst[0], x[0]) > RTOL, rel_err(fst[0], x[0])
    raw = M.SwarmEnv(seed=3, fresh_noise=True)
    raw.reset()
    for t in range(128):
        raw.step(np.zeros((10, 2)))
    assert raw.t == 128 + NB
    with pytest.raises(IndexError):
        raw.step(np.zeros((10, 2)))


def test_paac_learner_with_fresh_noise(pkg, cuda):
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import train_paac_conv as tp
    paac = pkg.submodule("agents.paac.paac")
    learners = {}
    for flag in ([], ["--fresh_noise"]):
        args = tp.get_arg_parser().parse_args(["--clip_norm", "1", "-ec", "32", "--n_locusts", "16"] + flag)
        net_creator, env_creator = tp.get_network_and_environment_creator(args)
        torch.manual_seed(0)
        L = paac.GridPAACLearner(net_creator, env_creator, args, use_cuda_graph=False)
        L.start()
        torch.manual_seed(1)
        for _ in range(2):
            L.update()
        torch.cuda.synchronize()
        learners[bool(flag)] = L
    L = learners[True]
    assert L.env.noise == "fresh" and learners[False].env.noise == "frozen"
    assert torch.isfinite(L.global_norm) and float(L.global_norm) > 0
    assert all(torch.isfinite(p).all() for p in L.network.parameters())
    assert (L.env.elapsed == 2 * L.max_local_steps).all()
    assert not torch.equal(L.env.x, learners[False].env.x)
