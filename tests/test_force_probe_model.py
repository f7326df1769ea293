"""State builders and per-locust error bound of the pair-force probes (tests/test_gpu_force_probes.py), proven on the CPU.

The GPU probes check the kernels' forces (csrc/swarm_kernels.cuh: pair_forces in every tiling) locust by locust against
an FP64 reference, with a bound T_j for each locust instead of the parity metric max|dv| / max|v| per env, which hides a
single wrong pair or locust.  This file holds what those checks rest on and proves it without a GPU:

  * isolated-cluster layouts: points grouped in small clusters on a lattice of spacing S = 30 max(L, 1), so that the
    whole far field of a locust, F exp(-S/L) (N + A), is below 2^-25 and a lone locust's FP32 force rounds to exactly
    (U, G); the FP64 forces of such a layout are the per-cluster sums (checked against oracle.swarm_oracle.forces), which
    keeps the reference cheap at N = 2048;
  * the circle-method round robin: round m splits the locusts into N/2 pairs (one bye for odd N), and the N - 1 rounds
    (N for odd N) hold every unordered pair exactly once; agent k of env m sits next to locust (m + k ceil(N/A)) mod N,
    so the N envs hold every (agent, locust) pair;
  * the bound T_j, checked against a NumPy float32 emulation of the precise path.

Per-locust bound.  With d = p_i - p_j, r = |d|, eps = 1e-6 (the reference's "+ 0.000001"):
    M_ij     = (F e^(-r/L) + e^(-r)) r / (r + eps)                  magnitude scale of one contribution
    beta_ij  = (F e^(-r/L) (1 + r/L) + e^(-r) (1 + r)) / (r + eps)  bound on |d c_ij / d d|
    sigma_ij = 2^-46 (|p_i|_inf + |p_j|_inf) log2(e) + 2^-24 r      error of the hi/lo difference
    T_j = sum_i [kappa 2^-23 (4 + r + r/L) M_ij + beta_ij sigma_ij] + K_s 2^-24 sqrt(n_j) sum_i |c_ij| + 2^-23 (|U| + |G|)
with c_ij the reference's contribution, n_j = N + A, and a pair of bitwise equal points left out (its difference is
exactly 0 in the kernel, as is its contribution).  Where the terms come from:
  * sigma: split_hilo rounds p log2(e) to FP64 (2^-53), the hi part to FP32 and the remainder to FP32 (2^-24 of at most
    2^-24 |p|): hi + lo represents each coordinate to 2^-48 |p|, so the difference of two represented points is off by
    up to ~2^-47.5 (|p_i| + |p_j|) in the plane -- however close the two points are.  That is the envelope of the
    kernel far from the origin (DESIGN section 3.1).  The FP32 subtraction and sum add 2^-24 r.
  * kappa 2^-23 (4 + r + r/L) M: the chain r -> s -> w -> w d has four roundings or approximations of relative size
    2^-23 at most: rsqrt.approx (PTX ISA: max relative error 2^-22.9 on the full range), rcp.approx (2^-23; or the
    series 1/(r + eps) = rinv - eps rinv^2, whose dropped term is below 2^-24 where it is used), each ex2.approx
    (2^-22.5 relative on its fraction, fast mode) and the IEEE operations of the precise mode (2^-24 each, exp2f
    within 2 ulp).  ex2 of an argument that carries a relative error e is off by a relative e r ln2 (e r/L ln2 for the
    attraction): hence the r and r/L terms.  kappa = 4 (fast) and 2 (precise) cover the sums of these maxima.
  * K_s 2^-24 sqrt(n_j) sum |c_ij|: the FP32 accumulation over n_j sources.  The rigorous (n_j - 1) 2^-24 sum |c_ij| is
    looser than the parity metric at N >= 256; sqrt(n_j) is the statistical scale of the rounding walk, K_s = 4 covers
    its tail over the probes' 10^5 locusts.
  * 2^-23 (|U| + |G|): adding (U, G) last rounds each component once, by up to 2^-24 of it (the factor 2 keeps that
    rounding alone at half the bound); it also absorbs the far field (< 2^-25).
"""
import functools

import numpy as np
import pytest

from oracle import swarm_oracle as so

EPS = so.EPS_R
LOG2E = 1.4426950408889634
DEFAULTS = (so.F_ATTR, so.L_ATTR, so.WIND_SPEED, so.GRAVITY)       # (F, L, U, G)
PARAMS = [DEFAULTS, (0.2, 3.0, 0.5, -2.0), (2.0, 25.0, 1.0, -1.0), (0.9, 1.5, 0.0, -1.0)]
KAPPA = {"fast": 4.0, "precise": 2.0}
K_S = 4.0
# every tiling of pair_forces, and the sizes that reach it (force_mode in csrc/swarm_b200.cu)
MODE_N = {
    "1": [2, 31, 32, 65, 96, 129, 160, 480],
    "3 odd": [33, 63, 64, 191, 192, 319, 320, 448],         # odd super-tile count: no half passes
    "3 even": [97, 127, 128, 255, 256, 511, 512],           # even super-tile count: a half pass each way
    "2": [513, 700, 1024],
    "4": [1025, 2047, 2048],
}
ALL_N = sorted(n for ns in MODE_N.values() for n in ns)
COVER_A = (1, 10, 32)
DENSE_A = (1, 2, 10, 31, 32)
SHIFTS = (0.0, 1e2, 1e4)
SWITCH = 4096 * EPS       # pairs closer than this take MUFU.RCP for 1/(r + eps) in the unordered-pair modes (inv_r_eps)


def force_mode(N):
    """csrc/swarm_b200.cu force_mode, restated: 1/3 unordered pairs (3: N pads to 64 as well as to 32), 2/4 ordered."""
    if N <= 512:
        return 3 if (N + 63) // 64 * 64 == (N + 31) // 32 * 32 else 1
    return 2 if N <= 1024 else 4


def spacing(L):
    return 30.0 * max(L, 1.0)


def sites(n, sp):
    """n lattice points of spacing sp on an odd-sided square centred on the origin, nearest to the origin first"""
    side = int(np.ceil(np.sqrt(n)))
    side += 1 - side % 2
    k = np.arange(side * side)
    p = np.stack([(k % side - side // 2) * sp, (k // side - side // 2) * sp], axis=1).astype(np.float64)
    return p[np.argsort(np.abs(p).max(1), kind="stable")][:n]


def probe_offsets(rs, n, lo=1e-3, hi=3.0):
    r = np.exp(rs.uniform(np.log(lo), np.log(hi), size=n))
    a = rs.uniform(0.0, 2.0 * np.pi, size=n)
    return np.stack([r * np.cos(a), r * np.sin(a)], axis=1)


class Layout(object):
    """E envs of N locusts and A agents in isolated clusters: partner (E,N) the locust paired with j (-1: none), home (E,A)
    the locust agent k sits next to (-1: a lone agent).  The cluster of locust j is {j, partner j} and the agents at
    home in it; everything else is at least S away."""

    def __init__(self, x, xa, partner, home, S):
        self.x, self.xa, self.partner, self.home, self.S = x, xa, partner, home, S

    @property
    def E(self):
        return self.x.shape[0]

    def shifted(self, dx=0.0, dy=0.0):
        t = np.array([dx, dy])
        return Layout(self.x + t, self.xa + t, self.partner, self.home, self.S)

    def lone(self):
        """(E,N) locusts with no cluster mate"""
        lone = self.partner < 0
        for k in range(self.xa.shape[1]):
            h = self.home[:, k]
            rows = np.nonzero(h >= 0)[0]
            lone[rows, h[rows]] = False
        return lone

    def labels(self):
        """(E, N+A) cluster label of every point (locust j's cluster is min(j, partner j); lone agents get their own)"""
        E, N, A = self.E, self.x.shape[1], self.xa.shape[1]
        j = np.arange(N)[None].repeat(E, 0)
        lab = np.where(self.partner >= 0, np.minimum(j, self.partner), j)
        own = N + np.arange(A)[None].repeat(E, 0)
        hl = np.take_along_axis(lab, np.maximum(self.home, 0), axis=1)
        return np.concatenate([lab, np.where(self.home >= 0, hl, own)], axis=1)


def layout_from(centres, partner, home, rs, S):
    """x of locust j = centres[e, j] (lattice site), partner = site + probe offset, agents next to their home locust"""
    E, N = partner.shape
    x = centres.copy()
    has = (partner >= 0) & (partner > np.arange(N)[None])
    e, j = np.nonzero(has)
    x[e, partner[e, j]] = x[e, j] + probe_offsets(rs, len(e))
    A = home.shape[1]
    xa = np.empty((E, A, 2))
    for k in range(A):
        h = home[:, k]
        xa[:, k] = x[np.arange(E), np.maximum(h, 0)] + probe_offsets(rs, E)
    return Layout(x, xa, partner, home, S)


def round_robin(N):
    """circle-method round robin as arrays (a, b) of shape (rounds, n/2), n = N rounded up to even: round m pairs a[m, k]
    with b[m, k]; for odd N the partner N is the bye"""
    n = N + N % 2
    m = np.arange(n - 1)
    order = np.concatenate([np.full((n - 1, 1), n - 1), (m[:, None] + m[None]) % (n - 1)], axis=1)
    return order[:, :n // 2], order[:, ::-1][:, :n // 2]


@functools.lru_cache(maxsize=None)
def coverage_layout(N, A, seed=0):
    """N envs: env m holds round m mod R of the round robin as pairs and agent k next to locust (m + k ceil(N/A)) mod N"""
    rs = np.random.RandomState(seed + 7919 * N + A)
    a, b = round_robin(N)
    R, h = a.shape
    E = N
    S = spacing(so.L_ATTR)
    ra, rb = a[np.arange(E) % R], b[np.arange(E) % R]
    e = np.arange(E)[:, None]
    partner = np.empty((E, N + 1), dtype=np.int64)
    site = np.empty((E, N + 1), dtype=np.int64)
    partner[e, ra], partner[e, rb] = rb, ra
    site[e, ra] = site[e, rb] = np.arange(h)[None]
    partner, site = partner[:, :N], site[:, :N]
    partner[partner == N] = -1                                         # the bye of odd N
    home = (np.arange(E)[:, None] + -(-N // A) * np.arange(A)[None]) % N
    # a pair with its agents is at most ~12 across: spacing S + 16 keeps other clusters >= S away
    return layout_from(sites(h, S + 16.0)[site], partner, home, rs, S)


def seps():
    """separations of the pair-weight sweep: 0, below eps, a log grid to 300 and the band around the series switch"""
    band = [SWITCH * (1 + s * k * 2.0 ** -20) for k in range(1, 9) for s in (-1, 1)]
    return np.array([0.0, 1e-12, 1e-9, EPS, 10 * EPS] + list(np.logspace(-5, np.log10(300.0), 36)) + band)


@functools.lru_cache(maxsize=None)
def sweep_layout(N, A, L, shift):
    """one probe pair per env near (shift, 0), every other locust and agent lone on the lattice; envs = separations x
    directions (along x with dy == 0, along y with dx == 0, two random)"""
    rs = np.random.RandomState(N + int(L * 10))
    S = spacing(L)
    sp = seps()
    dirs = [(1.0, 0.0), (0.0, 1.0)]
    E = len(sp) * 4
    site = sites(N + A, S + 301.0)
    x = np.empty((E, N, 2))
    xa = np.empty((E, A, 2))
    partner = -np.ones((E, N), dtype=np.int64)
    for e in range(E):
        r, kd = sp[e // 4], e % 4
        if kd < 2:
            u = np.array(dirs[kd])
        else:
            a = rs.uniform(0, 2 * np.pi)
            u = np.array([np.cos(a), np.sin(a)])
        i, j = (0, 1) if N == 2 else rs.choice(N, 2, replace=False)
        perm = rs.permutation(N + A - 1) + 1           # site 0 (the origin) holds the probe pair
        rest = [k for k in range(N) if k not in (i, j)]
        x[e, rest] = site[perm[:len(rest)]]
        xa[e] = site[perm[len(rest):len(rest) + A]]
        x[e, j] = (0.0, 0.0)
        x[e, i] = r * u
        partner[e, i], partner[e, j] = j, i
    lay = Layout(x, xa, partner, -np.ones((E, A), dtype=np.int64), S)
    return lay.shifted(shift)


# ------------------------------------------------------------------------------------------------ dense states
@functools.lru_cache(maxsize=None)
def late_states(N, A):
    """((3,N,2), (3,A,2)) snapshots at steps 32, 96 and 127 of a seeded oracle episode: a grounded layer, dense clusters"""
    rs = np.random.RandomState(4242 + 31 * N + A)
    x0, xa0, burn, an, pn = so.draw_reset_numpy(rs, N, A)
    x, xa = so.reset_injected(x0[None], xa0[None], burn[None], an[None], pn[None])
    out = []
    for t in range(1, 128):
        act = rs.normal(size=(1, A, 2))
        so.clip_actions_(act.reshape(-1, 2))
        so.step(x, xa, act, an[None, 10], pn[None, 10])
        if t in (32, 96, 127):
            out.append((x[0].copy(), xa[0].copy()))
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])


@functools.lru_cache(maxsize=None)
def rolling_swarm(N, A, seed=0):
    """((1,N,2), (1,A,2)) a synthesised rolling swarm: 40 % grounded at y = 0, ~5 % exact duplicates, ~5 % pairs
    1e-5 ... 1e-3 apart, agents inside the swarm"""
    rs = np.random.RandomState(97 * N + A + seed)
    w = 3.0 * np.sqrt(N / 80.0)
    x = np.stack([rs.uniform(0, w, N), rs.exponential(0.6, N)], axis=1)
    x[rs.rand(N) < 0.4, 1] = 0.0
    idx = rs.permutation(N)
    nd = max(1, N // 20)
    x[idx[:nd]] = x[idx[nd:2 * nd]]                                   # exact duplicates
    off = probe_offsets(rs, nd, 1e-5, 1e-3)
    x[idx[2 * nd:3 * nd]] = x[idx[3 * nd:4 * nd]] + off              # close pairs
    x[:, 1] = np.maximum(x[:, 1], 0.0)
    xa = np.stack([rs.uniform(0, w, A), rs.uniform(0, 1.5, A)], axis=1)
    return x[None], xa[None]


def dense_states(N, A):
    """(x, xa, tag) with every snapshot at every shift along x"""
    x, xa = late_states(N, A) if N <= 256 else rolling_swarm(N, A)
    xs = np.concatenate([x + (s, 0.0) for s in SHIFTS])
    xas = np.concatenate([xa + (s, 0.0) for s in SHIFTS])
    return xs, xas


# ------------------------------------------------------------------------------------------------ reference + bound
class Ref(object):
    """FP64 forces v (E,N,2), reward (E,) and the bound's parts: T_j = kappa * a + b + K_S * c + d"""

    def __init__(self, v, a, b, c, d):
        self.v, self.a, self.b, self.c, self.d = v, a, b, c, d
        self.reward = -(v ** 2).sum(-1).mean(-1)

    def T(self, math):
        return KAPPA[math] * self.a + self.b + K_S * self.c + self.d

    def reward_bound(self, math):
        T = self.T(math)
        return (2.0 * np.sqrt((self.v ** 2).sum(-1)) * T + T ** 2).mean(-1) + 2.0 ** -22 * np.abs(self.reward)


def _terms(pt, ps, valid, F, L):
    """targets pt (M,2), sources ps (M,K,2), valid (M,K) -> (sum c (M,2), sum of the a, b and |c| terms (M,))"""
    d = ps - pt[:, None, :]
    r = np.sqrt((d ** 2).sum(-1))
    ok = valid & (r > 0)                        # bitwise equal points contribute exactly 0 in every kernel path
    ea, er = F * np.exp(-r / L), np.exp(-r)
    den = r + EPS
    c = np.where(ok[..., None], ((ea - er) / den)[..., None] * d, 0.0)
    M = (ea + er) * r / den
    beta = (ea * (1 + r / L) + er * (1 + r)) / den
    sig = 2.0 ** -46 * (np.abs(ps).max(-1) + np.abs(pt).max(-1)[:, None]) * LOG2E + 2.0 ** -24 * r
    a = np.where(ok, 2.0 ** -23 * (4 + r + r / L) * M, 0.0).sum(-1)
    b = np.where(ok, beta * sig, 0.0).sum(-1)
    cn = np.sqrt((c ** 2).sum(-1)).sum(-1)
    return c.sum(1), a, b, cn


def _finish(vsum, a, b, cn, n, U, G):
    v = vsum + np.array([U, G])
    return Ref(v, a, b, 2.0 ** -24 * np.sqrt(n) * cn, 2.0 ** -23 * (abs(U) + abs(G)))


def reference_dense(x, xa, F=so.F_ATTR, L=so.L_ATTR, U=so.WIND_SPEED, G=so.GRAVITY, chunk=256):
    """every pair: the oracle's forces (so.forces, restated with the bound's terms), E envs"""
    E, N, _ = x.shape
    A = xa.shape[1]
    out = [np.empty((E, N, 2))] + [np.empty((E, N)) for _ in range(3)]
    for e in range(E):
        src = np.concatenate([x[e], xa[e]])
        for j0 in range(0, N, chunk):
            pt = x[e, j0:j0 + chunk]
            ps = np.broadcast_to(src, (len(pt),) + src.shape)
            valid = np.ones(ps.shape[:2], dtype=bool)
            valid[np.arange(len(pt)), j0 + np.arange(len(pt))] = False
            for o, t in zip(out, _terms(pt, ps, valid, F, L)):
                o[e, j0:j0 + chunk] = t
    return _finish(*out, N + A, U, G)


def reference_clusters(lay, F=so.F_ATTR, L=so.L_ATTR, U=so.WIND_SPEED, G=so.GRAVITY):
    """per-cluster sums: sources of locust j = its partner and the agents at home in {j, partner j}"""
    E, N, _ = lay.x.shape
    A = lay.xa.shape[1]
    te, tj, src = [], [], []
    e, j = np.nonzero(lay.partner >= 0)
    te.append(e), tj.append(j), src.append(lay.x[e, lay.partner[e, j]])
    for k in range(A):
        e = np.nonzero(lay.home[:, k] >= 0)[0]
        h = lay.home[e, k]
        p = lay.partner[e, h]
        for ee, jj in ((e, h), (e[p >= 0], p[p >= 0])):
            te.append(ee), tj.append(jj), src.append(lay.xa[ee, k])
    te, tj, src = np.concatenate(te), np.concatenate(tj), np.concatenate(src)
    out = [np.zeros((E, N, 2))] + [np.zeros((E, N)) for _ in range(3)]
    for i0 in range(0, len(te), 1 << 20):
        sl = slice(i0, i0 + (1 << 20))
        res = _terms(lay.x[te[sl], tj[sl]], src[sl, None], np.ones((len(te[sl]), 1), dtype=bool), F, L)
        for o, t in zip(out, res):
            np.add.at(o, (te[sl], tj[sl]), t)
    return _finish(*out, N + A, U, G)


# ------------------------------------------------------------------------------------------------ float32 emulation
def _fma32(a, b, c):
    return (a.astype(np.float64) * b + c).astype(np.float32)


def split_hilo(p):
    s = p * LOG2E
    hi = s.astype(np.float32)
    return hi, (s - hi).astype(np.float32)


def emulate_precise(x, xa, F, L, U, G):
    """pair_forces<MODE, PRECISE=true> restated in float32 for one env: split_hilo, d = (hi_i - hi_j) + (lo_i - lo_j),
    IEEE sqrt / div, np.exp2 standing in for exp2f; locust sources in order, the agents summed from 0 and added last."""
    f32 = np.float32
    hi, lo = split_hilo(np.asarray(x, np.float64))
    ahi, alo = split_hilo(np.asarray(xa, np.float64))
    Ff, nInvL, eps_s = f32(F), f32(-1.0 / L), f32(EPS * LOG2E)

    def acc(sh, sl, v):
        d = (sh - hi) + (sl - lo)
        dx, dy = d[:, 0], d[:, 1]
        r = np.sqrt(_fma32(dx, dx, dy * dy))
        s = _fma32(np.full_like(r, Ff), np.exp2(r * nInvL), -np.exp2(-r))
        w = s / (r + eps_s)
        v[:, 0] = _fma32(w, dx, v[:, 0])
        v[:, 1] = _fma32(w, dy, v[:, 1])

    v = np.zeros(hi.shape, dtype=np.float32)
    for i in range(len(hi)):
        acc(hi[i], lo[i], v)
    g = np.zeros_like(v)
    for k in range(len(ahi)):
        acc(ahi[k], alo[k], g)
    return (v + g + np.array([U, G], dtype=np.float32)).astype(np.float64)


def ratio(got, ref, T):
    """observed / bound per locust"""
    return np.sqrt(((got - ref) ** 2).sum(-1)) / T


# ------------------------------------------------------------------------------------------------ CPU checks
def test_force_mode_table():
    for mode, ns in MODE_N.items():
        for N in ns:
            assert str(force_mode(N)) == mode.split()[0], N
            if mode.startswith("3"):
                assert ((N + 63) // 64) % 2 == (1 if mode == "3 odd" else 0), N


@pytest.mark.parametrize("N", ALL_N)
def test_round_robin_holds_every_pair_exactly_once(N):
    a, b = round_robin(N)
    assert len(a) == (N - 1 if N % 2 == 0 else N)
    flat = np.concatenate([a, b], axis=1)
    assert (np.sort(flat, axis=1) == np.arange(N + N % 2)[None]).all()          # every locust once per round
    ok = (a < N) & (b < N)
    lo, hi = np.minimum(a, b)[ok], np.maximum(a, b)[ok]
    seen = np.zeros((N, N), dtype=np.int64)
    np.add.at(seen, (lo, hi), 1)
    assert (seen[np.triu_indices(N, 1)] == 1).all() and seen.sum() == N * (N - 1) // 2


@pytest.mark.parametrize("A", COVER_A)
@pytest.mark.parametrize("N", [2, 31, 32, 65, 128, 513])
def test_coverage_layout(N, A):
    """every unordered pair in a cluster of its own exactly once over the N envs, every (agent, locust) pair at least
    once, and other clusters at least S away"""
    lay = coverage_layout(N, A)
    lab = lay.labels()
    pairs = np.zeros((N, N), dtype=np.int64)
    e, j = np.nonzero(lay.partner >= 0)
    np.add.at(pairs, (j, lay.partner[e, j]), 1)
    off = pairs[~np.eye(N, dtype=bool)]
    assert (off >= 1).all() and (off <= 2).all()            # env N - 1 of an even N repeats round 0
    agent_seen = np.zeros((A, N), dtype=bool)
    for k in range(A):
        agent_seen[k, lay.home[:, k]] = True
    assert agent_seen.all()
    pts = np.concatenate([lay.x, lay.xa], axis=1)
    for m in range(0, lay.E, max(1, lay.E // 16)):
        d = np.sqrt(((pts[m, :, None] - pts[m, None]) ** 2).sum(-1))
        other = lab[m, :, None] != lab[m, None, :]
        assert not other.any() or d[other].min() >= lay.S, m
        assert d[~other].max() < 16.0, m


def test_tournament_envs_hold_each_pair_once():
    """the first N - 1 (N for odd N) envs: each unordered pair is a cluster exactly once"""
    for N in (2, 31, 32, 96, 97):
        lay = coverage_layout(N, 10)
        R = len(round_robin(N)[0])
        cnt = np.zeros((N, N), dtype=np.int64)
        e, j = np.nonzero(lay.partner[:R] >= 0)
        np.add.at(cnt, (j, lay.partner[:R][e, j]), 1)
        assert (cnt == 1 - np.eye(N, dtype=np.int64)).all(), N


@pytest.mark.parametrize("N,A", [(2, 1), (2, 10), (5, 3), (8, 10), (7, 1)])
def test_cluster_reference_is_the_full_oracle(N, A):
    """per-cluster sums == so.forces of the whole state within 1e-12 (the far field is below 1e-12 here)"""
    for lay in (coverage_layout(N, A), sweep_layout(N, A, so.L_ATTR, 0.0) if N >= 2 else None):
        ref = reference_clusters(lay)
        v, r = so.forces(lay.x, lay.xa)
        assert np.abs(ref.v - v).max() <= 1e-12
        assert np.abs(ref.reward - r).max() <= 1e-12


def test_dense_reference_is_the_oracle():
    x, xa = dense_states(64, 10)
    ref = reference_dense(x, xa)
    v, r = so.forces(x, xa)
    assert np.abs(ref.v - v).max() <= 1e-12 * np.abs(v).max()
    for F, L, U, G in PARAMS[1:]:
        ref = reference_dense(x[:2], xa[:2], F, L, U, G)
        v, _ = so.forces(x[:2], xa[:2], F, L, U, G)
        assert np.abs(ref.v - v).max() <= 1e-12 * np.abs(v).max()


def test_lone_locusts_far_field_below_half_ulp():
    """F exp(-S/L) (N + A) < 2^-25 for every parameter set and size: a lone locust's FP32 force rounds to (U, G)"""
    for F, L, U, G in PARAMS:
        assert F * np.exp(-spacing(L) / L) * (2048 + 32) < 2.0 ** -25


def test_sweep_layout():
    for N in (2, 64, 600):
        lay = sweep_layout(N, 10, so.L_ATTR, 0.0)
        e, j = np.nonzero(lay.partner >= 0)
        d = lay.x[e, j] - lay.x[e, lay.partner[e, j]]
        r = np.sqrt((d ** 2).sum(-1)).reshape(-1, 2)[:, 0].reshape(-1, 4)
        assert np.array_equal(r[:, 0], seps()) and np.array_equal(r[:, 1], seps())     # the axis-aligned envs, exactly
        assert (d.reshape(-1, 4, 2, 2)[:, 0, :, 1] == 0).all()                         # ... with dy == 0
        near = np.abs(seps() - SWITCH) < 16 * 2.0 ** -20 * SWITCH
        assert (seps()[near] < SWITCH).sum() == 8 and (seps()[near] > SWITCH).sum() == 8
        assert (lay.lone().sum(1) == N - 2).all()
        lab = lay.labels()
        pts = np.concatenate([lay.x, lay.xa], axis=1)
        for m in range(0, lay.E, 37):
            dd = np.sqrt(((pts[m, :, None] - pts[m, None]) ** 2).sum(-1))
            assert dd[lab[m, :, None] != lab[m, None, :]].min() >= lay.S


@pytest.mark.parametrize("shift", SHIFTS)
def test_bound_holds_for_the_precise_emulation(shift):
    """observed / bound <= 0.5 for the float32 emulation of the precise path on probe layouts and dense states"""
    worst = {}
    cases = []
    for N, A in ((2, 10), (31, 1), (64, 32)):
        lay = coverage_layout(N, A).shifted(shift)
        cases.append(("coverage", lay.x, lay.xa, reference_clusters(lay), DEFAULTS))
    for prm in PARAMS:
        lay = sweep_layout(64, 10, prm[1], shift)
        cases.append(("sweep", lay.x, lay.xa, reference_clusters(lay, *prm), prm))
    for N, A in ((80, 10), (256, 2), (513, 31)):
        x, xa = (late_states(N, A) if N <= 256 else rolling_swarm(N, A))
        x, xa = x + (shift, 0.0), xa + (shift, 0.0)
        cases.append(("dense", x, xa, reference_dense(x, xa), DEFAULTS))
    for fam, x, xa, ref, prm in cases:
        T = ref.T("precise")
        for e in range(len(x)):
            got = emulate_precise(x[e], xa[e], *prm)
            q = ratio(got, ref.v[e], T[e])
            worst[fam] = max(worst.get(fam, 0.0), float(q.max()))
            assert q.max() <= 0.5, (fam, e, int(q.argmax()), float(q.max()))
    print("precise emulation, shift %g: worst observed/bound %s" % (shift, worst))
