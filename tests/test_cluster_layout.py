"""The cluster layout (SwarmParams.tuning bits 8-12) without a GPU: what swarm_validate admits and refuses, and a
target-chunked FP64 restatement of the oracle's step for swarms whose dense (N, N) matrices would take gigabytes."""
import ctypes

import numpy as np
import pytest

from oracle import swarm_oracle as so


@pytest.fixture(scope="module")
def nat(pkg):
    pkg.load()
    from golds_rl_gym_b200 import _native
    return _native


def params(nat, **kw):
    d = dict(n_envs=4, n_locusts=4096, n_agents=10, grid_size=84, n_burn_in=10, max_episode_steps=128, math_mode=0,
             tuning=0, noise=1e-4, gravity=-1.0, wind=1.0, F=0.5, L=10.0, dt=0.05, box_width=3.0, box_height=3.0,
             seed=1, env_id_offset=0)
    d.update(kw)
    return nat.SwarmParams(**d)


def validate(nat, **kw):
    return nat.load().swarm_validate(ctypes.byref(params(nat, **kw)))


def force_warps(N):
    T = 2 if N <= 1024 else 4
    return ((-(-N // T) + 31) // 32)


@pytest.mark.parametrize("N,K,want", [
    (4096, None, 0), (4096, 2, 0), (8192, None, 0), (8192, 2, 0), (8192, 16, 0), (513, 1, 0), (2048, 16, 0),
    (8193, None, -2), (8193, 4, -2),              # above the cluster layout's limit
    (512, 2, -4), (300, None, -4),                # unordered pairs below 513: no bitwise twin in a cluster
    (4096, 17, -4), (4096, 30, -4),               # K > 16 (31 = automatic)
    (513, 10, -4),                                # more CTAs than force warps (513 locusts have 9)
    (8192, 1, -2),                                # 2048 virtual threads do not fit one CTA
])
def test_validate_cluster_field(nat, N, K, want):
    assert validate(nat, n_locusts=N, tuning=nat.tune_cluster(K)) == want


def test_validate_without_the_field_is_unchanged(nat):
    assert validate(nat, n_locusts=4096) == -2
    assert validate(nat, n_locusts=2048) == 0
    assert validate(nat, n_locusts=2048, tuning=3 << 4) == 0
    assert validate(nat, n_locusts=80, tuning=1 << 6) == -4      # a bit outside both fields


@pytest.mark.parametrize("place", [1 << 4, 2 << 4, 3 << 4])
def test_placement_bits_with_the_cluster_field_are_refused(nat, place):
    assert validate(nat, n_locusts=4096, tuning=nat.tune_cluster(4) | place) == -4


def test_strerror_names_both_limits(nat):
    msg = nat.load().swarm_strerror(-2).decode()
    assert "2048" in msg and "8192" in msg and "cluster" in msg


def test_force_warps_bound_the_cluster_size(nat):
    for N in (513, 700, 1024, 1025, 2047, 2048, 3000, 8192):
        nw = force_warps(N)
        kmax = min(16, nw)
        assert validate(nat, n_locusts=N, tuning=nat.tune_cluster(kmax)) == 0, N
        if kmax < 16:
            assert validate(nat, n_locusts=N, tuning=nat.tune_cluster(kmax + 1)) == -4, N


# ------------------------------------------------------------------------------------------------ chunked oracle
def v_calculate_chunked(x, xa, chunk=256):
    """so.forces (multiagent.py:88-115) one block of targets at a time: the same FP64 expression per target (locust
    sum over all sources, then the agent sum), memory O(chunk (N + A)) instead of O(N^2)."""
    x = np.asarray(x, dtype=np.float64)
    xa = np.asarray(xa, dtype=np.float64)
    E, N, _ = x.shape
    v = np.empty((E, N, 2), dtype=np.float64)
    base = np.array([so.WIND_SPEED, so.GRAVITY], dtype=np.float64)
    for e in range(E):
        src = np.concatenate([x[e], xa[e]])
        for j0 in range(0, N, chunk):
            xs = x[e, j0:j0 + chunk]
            d = src[None, :, :] - xs[:, None, :]
            r = np.sqrt((d ** 2).sum(axis=-1))
            w = so.s_potential(r)
            vl = ((w[:, :N, None] * d[:, :N]) / (r[:, :N, None] + so.EPS_R)).sum(axis=1)
            va = ((w[:, N:, None] * d[:, N:]) / (r[:, N:, None] + so.EPS_R)).sum(axis=1)
            v[e, j0:j0 + chunk] = (base + vl) + va
    return v, -(v ** 2).sum(axis=-1).mean(axis=-1)


def step_chunked(x, xa, actions, noise_a, noise_x, add_wind=True):
    """so.step with the chunked forces; in place on x, xa; returns (reward, done)"""
    va = np.array(actions, dtype=np.float64, copy=True)
    if add_wind:
        va[..., 0] += so.WIND_SPEED
    so.move_(xa, va, so.NOISE * np.asarray(noise_a, dtype=np.float64))
    v, reward = v_calculate_chunked(x, xa)
    so.move_(x, v, so.NOISE * np.asarray(noise_x, dtype=np.float64))
    return reward, reward >= 0


@pytest.mark.parametrize("N,A", [(1, 1), (37, 10), (300, 32), (600, 1)])
def test_chunked_v_calculate_is_the_oracle(N, A):
    rs = np.random.RandomState(N + A)
    x = rs.rand(2, N, 2) * 3.0
    xa = rs.rand(2, A, 2) * 3.0
    v, r = v_calculate_chunked(x, xa, chunk=64)
    v0, r0 = so.forces(x, xa)
    assert np.allclose(v, v0, rtol=1e-13, atol=1e-13)
    assert np.allclose(r, r0, rtol=1e-13)


def test_chunked_step_is_the_oracle():
    rs = np.random.RandomState(5)
    x, xa = rs.rand(2, 200, 2), rs.rand(2, 10, 2)
    a, na, nx = rs.normal(size=(2, 10, 2)), rs.normal(size=(2, 10, 2)), rs.normal(size=(2, 200, 2))
    x1, xa1 = x.copy(), xa.copy()
    r1, d1 = step_chunked(x1, xa1, a, na, nx)
    r0, d0 = so.step(x, xa, a, na, nx)
    assert np.allclose(x1, x, rtol=1e-13, atol=1e-15) and np.array_equal(xa1, xa)
    assert np.allclose(r1, r0, rtol=1e-13) and np.array_equal(d1, d0)
