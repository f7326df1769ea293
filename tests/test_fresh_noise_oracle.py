"""CPU: fresh per-step noise (SWARM_STEP_FRESH_NOISE, SURVEY Q1 fixed) on the oracle side -- the oracle's fresh step
against the reference with `self.t` advanced by hand, the row bookkeeping of FreshOracleRunner, the
Philox row export restatement, and argument checks of swarm_philox_noise_rows that need no GPU."""
import ctypes
import os
import sys

import numpy as np
import pytest

from oracle import philox as ph
from oracle import ref_loader as rl
from oracle import swarm_oracle as so

from _fresh_noise import TABLE_ROWS, FreshOracleRunner, draw_reset_full, noise_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_ref = pytest.mark.skipif(not rl.reference_available(), reason="/root/reference not mounted")


@needs_ref
@pytest.mark.parametrize("seed", [192, 7, 31])
@pytest.mark.parametrize("N", [64, 80])
def test_fresh_step_matches_fixed_reference(N, seed):
    """The reference's SwarmEnv with its frozen index fixed (env.t += 1 after every step) against so.step fed with
    row N_BURN_IN + t at step t, teacher-forced, 16 steps."""
    rl.load_reference()
    np.random.seed(seed)
    draws = draw_reset_full(np.random, N)
    assert draws[3].shape == (TABLE_ROWS, 10, 2) and draws[4].shape == (TABLE_ROWS, N, 2)
    env = rl.make_reference_env(N)
    ref = rl.reference_reset_injected(env, *draws)
    assert env.t == so.N_BURN_IN
    rs = np.random.RandomState(seed + 1)
    for t in range(16):
        a = so.clip_actions_(rs.normal(size=(10, 2)))
        x, xa = ref[0][None].copy(), ref[1][None].copy()
        ref, r, d, _ = env.step(a)
        env.t += 1
        r2, d2 = so.step(x, xa, a[None], draws[3][so.N_BURN_IN + t][None], draws[4][so.N_BURN_IN + t][None])
        assert np.abs(x[0] - ref[0]).max() <= 1e-12 * max(1.0, np.abs(ref[0]).max()), t
        assert np.array_equal(xa[0], ref[1]), t
        assert abs(r - r2[0]) <= 1e-12 * abs(r) and bool(d) == bool(d2[0])
    assert env.t == so.N_BURN_IN + 16


def test_oracle_runner_fresh_rows_over_an_episode(monkeypatch):
    """FreshOracleRunner, TimeLimit 128: the step proper of env e at episode step t gets row 10 + t of that
    env's current tables, for a whole episode and into the next one (the frozen runner keeps row 10)."""
    E, N = 3, 4

    def draws(e, ep):      # recognisable tables: value = 1000 * e + 100 * ep + row
        rows = np.arange(TABLE_ROWS, dtype=np.float64)[:, None, None] + 1000 * e + 100 * ep
        return (np.full((N, 2), 0.5), np.full((10, 2), 0.5), np.zeros((so.N_BURN_IN, 10, 2)),
                np.broadcast_to(rows, (TABLE_ROWS, 10, 2)).copy(), -np.broadcast_to(rows, (TABLE_ROWS, N, 2)).copy())

    calls = []

    def recording_step(x, xa, actions, noise_a, noise_x, add_wind=True):
        calls.append((np.array(noise_a), np.array(noise_x)))
        E_ = x.shape[0]
        return np.full(E_, -1.0), np.zeros(E_, dtype=bool)

    monkeypatch.setattr(so, "step", recording_step)
    for fresh in (True, False):
        runner = FreshOracleRunner if fresh else so.OracleRunner
        run = runner(E, N, draws, grid_size=8, max_episode_steps=128)
        run.reset()
        for t in range(128 + 5):
            del calls[:]
            _, done = run.step(np.zeros((E, 10, 2)))
            na, nx = calls[0]                       # the step proper (burn-in steps of a reset follow it)
            k, ep = t % 128, t // 128
            for e in range(E):
                want = 1000 * e + 100 * ep + (so.N_BURN_IN + k if fresh else so.N_BURN_IN)
                assert (na[e] == want).all() and (nx[e] == -want).all(), (fresh, t, e)
            assert bool(done.all()) == (k == 127)
    # a table that runs out fails like the fixed reference (IndexError), not silently
    run = FreshOracleRunner(1, N, lambda e, ep: tuple(a[:12] if i >= 3 else a for i, a in enumerate(draws(e, ep))),
                            grid_size=8, max_episode_steps=0)
    run.reset()
    run.step(np.zeros((1, 10, 2)))
    run.step(np.zeros((1, 10, 2)))
    with pytest.raises(IndexError):
        run.step(np.zeros((1, 10, 2)))


def test_full_tables_are_the_reference_draw_order():
    """draw_reset_full draws what so.draw_reset_numpy draws (same order), only without cutting the tables."""
    full = draw_reset_full(np.random.RandomState(192), 80)
    cut = so.draw_reset_numpy(np.random.RandomState(192), 80)
    for a, b in zip(full[:3], cut[:3]):
        assert np.array_equal(a, b)
    assert full[3].shape == (TABLE_ROWS, 10, 2) and full[4].shape == (TABLE_ROWS, 80, 2)
    assert np.array_equal(full[3][:11], cut[3]) and np.array_equal(full[4][:11], cut[4])


def test_philox_noise_rows_restate_reset_rows():
    for seed, env_id, episode, N in ((1, 0, 0, 80), (20261018, 5, 3, 64), (2 ** 40 + 9, 77, 1, 17)):
        ref = ph.reset_draws(seed, env_id, episode, N)
        an, pn = noise_rows(seed, env_id, episode, 0, 11, N)
        assert np.array_equal(an, ref[3]) and np.array_equal(pn, ref[4])
        an2, pn2 = noise_rows(seed, env_id, episode, 10, 128, N)
        assert np.array_equal(an2[0], ref[3][10]) and np.array_equal(pn2[0], ref[4][10])
        assert an2.shape == (128, 10, 2) and pn2.shape == (128, N, 2)
        assert abs(pn2.mean()) < 0.1 and abs(pn2.std() - 1.0) < 0.1


def _params(nat, **kw):
    base = dict(n_envs=4, n_locusts=80, n_agents=10, grid_size=84, n_burn_in=10, max_episode_steps=128,
                math_mode=0, tuning=0, noise=1e-4, gravity=-1.0, wind=1.0, F=0.5, L=10.0, dt=0.05,
                box_width=3.0, box_height=3.0, seed=1, env_id_offset=0)
    base.update(kw)
    return nat.SwarmParams(**base)


def test_philox_noise_rows_argument_checks_without_gpu(pkg):
    nat = pkg._native
    lib = nat.load()
    assert nat.SWARM_STEP_FRESH_NOISE == 32
    p = _params(nat)
    fake = ctypes.c_void_p(256)          # never dereferenced: every check below returns before any CUDA call
    st = nat.SwarmState(fake, fake, fake, fake, fake, fake, None, 0)
    f = lib.swarm_philox_noise_rows
    assert f(None, ctypes.byref(st), 0, 11, fake, fake, None) == -1
    assert f(ctypes.byref(p), None, 0, 11, fake, fake, None) == -1
    assert f(ctypes.byref(p), ctypes.byref(nat.SwarmState()), 0, 11, fake, fake, None) == -1
    assert f(ctypes.byref(p), ctypes.byref(st), 0, 11, None, fake, None) == -1
    assert f(ctypes.byref(p), ctypes.byref(st), 0, 11, fake, None, None) == -1
    assert f(ctypes.byref(p), ctypes.byref(st), -1, 11, fake, fake, None) == -2
    assert f(ctypes.byref(p), ctypes.byref(st), 0, 0, fake, fake, None) == -2
    assert f(ctypes.byref(p), ctypes.byref(st), 0, -3, fake, fake, None) == -2
    assert f(ctypes.byref(_params(nat, n_envs=0)), ctypes.byref(st), 0, 11, fake, fake, None) == -2


def test_fresh_noise_options_are_checked_and_plumbed(pkg):
    m = pkg.submodule("envs.multiagent")
    with pytest.raises(ValueError):
        m.BatchedSwarmEnv(4, noise="sometimes")          # refused before any device is needed
    ec = pkg.submodule("agents.paac.environment_creator")
    assert ec.SwarmEnvironmentCreator().noise == "frozen"
    assert ec.SwarmEnvironmentCreator(noise="fresh").noise == "fresh"
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import train_paac_conv as tp
    assert tp.get_arg_parser().parse_args(["--fresh_noise"]).fresh_noise is True
    assert tp.get_arg_parser().parse_args([]).fresh_noise is False
