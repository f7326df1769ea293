"""The pair forces of every tiling, locust by locust, against FP64 (states and bound: tests/test_force_probe_model.py).

  a. coverage: the round-robin envs put every unordered pair of locusts, and every (agent, locust) pair, in a cluster of
     its own once, at every N of every force mode (MODE 1, MODE 3 with odd and even super-tile counts, MODE 2, MODE 4)
     and A in {1, 10, 32}: a lone locust's force must be (U, G) bit for bit (a misrouted reaction or a pad lane breaks
     it), every cluster member must be within its bound T_j (a missing or doubled pair breaks it);
  b. the pair weight over separations from exactly 0 to 300, below eps, on both sides of the series / MUFU.RCP switch,
     along the axes and at random, at 0, 1e2 and 1e4 from the origin, for four (F, L, U, G);
  c. dense late-episode and synthesised states (grounded layers, duplicates, pairs 1e-5 apart) against the full oracle;
  d. k_step's v_out, reward and new x in every raster placement and both noise modes equal swarm_forces bit for bit;
  e. k_reset equals ten k_step calls bit for bit.
Both math modes throughout; binding="ctypes", so that SWARM_B200_LIB can swap in another build of the library.
"""
import functools

import numpy as np
import pytest
import torch

from oracle import swarm_oracle as so

import test_force_probe_model as fp
from test_gpu_raster_edges import FALLBACK, PLACES

pytestmark = pytest.mark.gpu
MATH = ("fast", "precise")
RATIOS = {}


@pytest.fixture(scope="module")
def M(pkg, cuda):
    yield pkg.submodule("envs.multiagent")
    for k in sorted(RATIOS):
        q = np.concatenate(RATIOS[k])
        print("observed/bound %-9s %-8s n=%-8d q50 %.3g q90 %.3g q99 %.3g max %.3g" % (
            k[0], k[1], q.size, *np.quantile(q, [0.5, 0.9, 0.99]), q.max()))


def new_env(M, E, N, A, math, prm=fp.DEFAULTS, **kw):
    kw.setdefault("rasterize", False)
    env = M.BatchedSwarmEnv(E, n_locusts=N, n_agents=A, max_episode_steps=0, auto_reset=False, binding="ctypes",
                            math_mode=math, **kw)
    env.params.F, env.params.L, env.params.wind, env.params.gravity = prm
    return env


def gpu_forces(env, x, xa):
    dev = env.device
    v, r = env.forces(torch.as_tensor(x).to(dev), torch.as_tensor(xa).to(dev))
    return v.cpu().numpy(), r.cpu().numpy()


def check(family, math, v, r, ref, where, mask=None):
    """every locust (where mask) within T_j; the reward within the bound T_j induces on -mean|v|^2"""
    q = fp.ratio(v.astype(np.float64), ref.v, ref.T(math))
    if mask is not None:
        q = np.where(mask, q, 0.0)
    RATIOS.setdefault((family, math), []).append(q[mask] if mask is not None else q.ravel())
    if q.max() > 1.0:
        e, j = np.unravel_index(int(q.argmax()), q.shape)
        raise AssertionError("%s %s: env %d locust %d off by %.3g = %.3g x T_j; got %s want %s" % (
            where, math, e, j, float(np.sqrt(((v[e, j] - ref.v[e, j]) ** 2).sum())), float(q[e, j]), v[e, j], ref.v[e, j]))
    rb = ref.reward_bound(math)
    bad = np.abs(r - ref.reward) > rb
    assert not bad.any(), (where, math, np.nonzero(bad)[0][:8], r[bad][:4], ref.reward[bad][:4])


# ------------------------------------------------------------------------------------------------ a. coverage
@functools.lru_cache(maxsize=None)
def coverage_ref(N, A):
    return fp.reference_clusters(fp.coverage_layout(N, A))


@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("A", fp.COVER_A)
@pytest.mark.parametrize("N", fp.ALL_N)
def test_coverage_every_pair_once(M, N, A, math):
    lay = fp.coverage_layout(N, A)
    env = new_env(M, lay.E, N, A, math)
    mode = [k for k, ns in fp.MODE_N.items() if N in ns][0]
    assert str(env.plan()["force_mode"]) == mode.split()[0] == str(fp.force_mode(N)), (N, env.plan())
    v, r = gpu_forces(env, lay.x, lay.xa)
    lone = lay.lone()
    want = np.array([so.WIND_SPEED, so.GRAVITY], dtype=np.float32)
    bad = lone & ~(v == want).all(-1)
    assert not bad.any(), ("lone locust not exactly (U, G)", N, A, math, np.argwhere(bad)[:4], v[bad][:4])
    check("coverage", math, v, r, coverage_ref(N, A), (N, A))


# ------------------------------------------------------------------------------------------------ b. pair-weight sweep
@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("prm", fp.PARAMS, ids=lambda p: "F%g_L%g_U%g_G%g" % p)
@pytest.mark.parametrize("N", [2, 64, 600])
def test_pair_weight_sweep(M, N, prm, math):
    F, L, U, G = prm
    A = 10
    for shift in fp.SHIFTS:
        lay = fp.sweep_layout(N, A, L, shift)
        ref = fp.reference_clusters(lay, F, L, U, G)
        env = new_env(M, lay.E, N, A, math, prm)
        v, r = gpu_forces(env, lay.x, lay.xa)
        e, j = np.nonzero(lay.partner >= 0)
        coincident = (lay.x[e, j] == lay.x[e, lay.partner[e, j]]).all(-1)
        assert len(coincident) and coincident.sum() == 8                   # separation 0, 4 directions, both members
        assert (v[e[coincident], j[coincident]] == np.float32([U, G])).all(), (shift, prm, math)
        lone = lay.lone()
        if U != 0 and G != 0:
            assert (v[lone] == np.float32([U, G])).all(), (shift, prm, math)
        check("sweep", math, v, r, ref, (N, prm, shift))
        err = np.sqrt(((v[e, j] - ref.v[e, j]) ** 2).sum(-1))
        print("sweep N=%d %s %s shift %g: probe pair max |dv| %.2e" % (N, prm, math, shift, err.max()))


def test_v_calculate_with_other_parameters(M):
    """the facade's SwarmEnv.v_calculate(x, xa, F, L, U, G) passes every parameter on (fast math)"""
    F, L, U, G = fp.PARAMS[2]
    lay = fp.sweep_layout(64, 10, L, 0.0)
    ref = fp.reference_clusters(lay, F, L, U, G)
    for e in range(0, lay.E, 11):
        v, r = M.SwarmEnv.v_calculate(lay.x[e], lay.xa[e], F, L, U, G)
        vo, ro = so.forces(lay.x[e:e + 1], lay.xa[e:e + 1], F, L, U, G)
        assert np.abs(vo[0] - ref.v[e]).max() < 1e-12
        assert (fp.ratio(v, ref.v[e], ref.T("fast")[e]) <= 1.0).all(), e
        assert abs(r - ro[0]) <= ref.reward_bound("fast")[e], e


# ------------------------------------------------------------------------------------------------ c. dense states
@functools.lru_cache(maxsize=None)
def dense_ref(N, A):
    x, xa = fp.dense_states(N, A)
    return x, xa, fp.reference_dense(x, xa)


@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("N", [64, 80, 256, 513, 1024, 1025, 2047, 2048])
def test_dense_states(M, N, math):
    for A in fp.DENSE_A:
        x, xa, ref = dense_ref(N, A)
        env = new_env(M, len(x), N, A, math)
        v, r = gpu_forces(env, x, xa)
        check("dense", math, v, r, ref, (N, A))


# ------------------------------------------------------------------------------------------------ d. the step's forces
def step_states(N):
    """(x, xa) with y >= 0 everywhere: round-robin envs lifted off the ground, or dense states"""
    if N in (65, 191, 256, 700, 2047):
        lay = fp.coverage_layout(N, 10)
        lift = 1.0 - min(lay.x[..., 1].min(), lay.xa[..., 1].min())
        return lay.x + (0.0, lift), lay.xa + (0.0, lift)
    x, xa = fp.dense_states(N, 10)
    return x, np.maximum(xa, 0.0)


@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("noise", ["frozen", "fresh"])
@pytest.mark.parametrize("N", [65, 191, 256, 700, 2047, 80, 1024])
def test_step_uses_swarm_forces_in_every_placement(M, N, noise, math):
    """actions (-wind, 0) and zero noise keep every agent where it is, so the step's forces are swarm_forces(x, xa) of the
    state before the step, bit for bit, and so is the integration (move_particle rounds like so.move_)"""
    x, xa = step_states(N)
    A = xa.shape[1]
    E = len(x)
    for variant in PLACES:
        env = new_env(M, E, N, A, math, rasterize=True, tuning=PLACES[variant], noise=noise)
        if variant == "warps_static":
            env.state_c.work, env.state_c.work_words = None, 0
        assert env.plan()["raster_place"] in FALLBACK[variant], (variant, env.plan())
        dev = env.device
        x0, xa0 = torch.as_tensor(x).to(dev), torch.as_tensor(xa).to(dev)
        vf, rf = env.forces(x0.clone(), xa0.clone())
        env.x.copy_(x0)
        env.xa.copy_(xa0)
        env.noise_x.zero_()
        env.noise_a.zero_()
        env._was_reset = True
        act = torch.zeros(E, A, 2, dtype=torch.float32, device=dev)
        act[..., 0] = -so.WIND_SPEED
        over = {}
        if noise == "fresh":
            over = dict(noise_a=torch.zeros(E, A, 2, dtype=torch.float64, device=dev),
                        noise_x=torch.zeros(E, N, 2, dtype=torch.float64, device=dev))
        v = torch.full((E, N, 2), np.nan, dtype=torch.float32, device=dev)
        env.step(act, v_out=v, **over)
        torch.cuda.synchronize()
        where = (N, noise, math, variant, env.plan()["raster_place"])
        assert torch.equal(env.xa, xa0), where
        assert torch.equal(v, vf), where
        assert torch.equal(env.reward, rf), where
        want = x.copy()
        so.move_(want, v.double().cpu().numpy(), 0.0)
        assert np.array_equal(env.x.cpu().numpy(), want), where


# ------------------------------------------------------------------------------------------------ e. the reset kernel
@pytest.mark.parametrize("math", MATH)
@pytest.mark.parametrize("N", [65, 192, 700, 1025])
def test_reset_is_ten_steps(M, N, math):
    """k_reset on injected draws whose x0 is a round-robin layout == ten k_step calls with actions burn[k] (f64,
    unclipped) and noise rows k as overrides, bit for bit"""
    A = 10
    lay = fp.coverage_layout(N, A)
    E = lay.E
    rs = np.random.RandomState(N)
    burn = rs.normal(size=(E, so.N_BURN_IN, A, 2)) * 2.0
    an = rs.normal(size=(E, so.N_BURN_IN + 1, A, 2))
    pn = rs.normal(size=(E, so.N_BURN_IN + 1, N, 2))
    env = new_env(M, E, N, A, math)
    dev = env.device
    env.reset(draws=M.InjectedDraws(lay.x, lay.xa, burn, an, pn, device=dev))
    ref = new_env(M, E, N, A, math)
    ref.x.copy_(torch.as_tensor(lay.x).to(dev))
    ref.xa.copy_(torch.as_tensor(lay.xa).to(dev))
    ref._was_reset = True
    for k in range(so.N_BURN_IN):
        ref.step(torch.as_tensor(burn[:, k]).to(dev).contiguous(), noise_a=torch.as_tensor(an[:, k]).to(dev).contiguous(),
                 noise_x=torch.as_tensor(pn[:, k]).to(dev).contiguous())
    torch.cuda.synchronize()
    assert torch.equal(env.x, ref.x) and torch.equal(env.xa, ref.xa), (N, math)
