"""The rasteriser inside the step (env_raster<false> in k_step's raster warps, on k_step's own threads, or in
k_raster_follow) against the oracle, on states built so that its rarely taken branches run.

Fused rasterisation only sees the post-step state, and FP32 forces make that state unpredictable to the last bit.  So the
states here do not move: every locust is grounded and pushed down (v_y <= -0.05 in the oracle, so cutoff zeroes its
velocity), every agent has the action (-1, 0), which the wind turns into v = 0, and both noise rows are zero.  Such a
state is its own next state, bit for bit, in the kernel and in the oracle (both checked), so numpy's window of the
post-step state is known before the step, and points can be put on its edges:
  * locusts and agents exactly on numpy's first, an inner and the last edge (x == hi, the histogram's closed right edge),
    and 1, 2, 3 ulps beside each;
  * agents left of the window, right of it (digitize clamps to G - 1), at y == 6 (closed top edge), just above 6, at 0;
  * windows centred at +-40, +-1e4, +-1e6, and a locust at +-1e13, where the error bound alone (tol >= 0.25) sends the
    whole env to numpy's sequential mean;
  * 255, 256, 257 locusts in one cell (the grid-value look-up table ends at 256 locusts);
  * every locust and agent in one cell (the 16-bit counter half-word at 0xFFFF for N = 2047, A = 31), also with the
    other half of the same 32-bit word occupied by an agent in cell (bx, 1).
The CPU tests prove that each state takes the branch it targets: the acceptance rule of the parallel mean
(test_spec_mean_model.spec_counts) rejects every state built around an edge, so the sequential fall-back runs on it, and
accepts every other one.  The GPU tests force each placement through SwarmParams.tuning, read back which one ran
(plan_step falls back FOLLOW -> WARPS -> SELF when a shape does not fit), size the batch so that every persistent CTA
rasterises several envs, alternate waves of fall-back and fast envs (so the `unsure` flag and the box carry between envs
of one CTA), and compare grid, positions, forces and reward of every env with the oracle over three steps.

Realised on a B200 (148 SMs), as plan() reports it; "16"/"32" is the counter table:
    (48,10,84)    16  WARPS static, SELF filler, FOLLOW -> WARPS, auto WARPS
    (176,10,84)   16  WARPS queue + static, SELF filler, FOLLOW, auto FOLLOW
    (176,10,83)   16  WARPS queue + static, SELF no filler, FOLLOW, auto FOLLOW
    (700,10,84)   16  WARPS queue + static, SELF filler, FOLLOW, auto FOLLOW
    (2047,31,84)  16  WARPS queue + static, SELF filler, FOLLOW, auto FOLLOW
    (2048,10,84)  32  WARPS queue + static, SELF filler, FOLLOW, auto FOLLOW
    (48,32,84)    32  WARPS static, SELF filler, FOLLOW -> WARPS, auto WARPS
    (80,1,2)      16  WARPS static, SELF no filler, FOLLOW -> WARPS, auto WARPS
    (80,10,255)   16  WARPS static, SELF no filler, FOLLOW -> WARPS, auto WARPS
test_launch_matrix_covers_every_branch asserts the parts of this that matter, from plan() on the machine it runs on.
"""
import functools

import numpy as np
import pytest
import torch

from oracle import swarm_oracle as so

from test_spec_mean_model import spec_counts

W, Y_HI = so.BOX_WIDTH, 2.0 * so.BOX_HEIGHT
RTOL = 1e-5
CASES = [(48, 10, 84), (176, 10, 84), (176, 10, 83), (700, 10, 84), (2047, 31, 84), (2048, 10, 84), (48, 32, 84),
         (80, 1, 2), (80, 10, 255)]
LOCAL_CASES = [(G, A) for G in (2, 83, 255) for A in (1, 32)]
REFUSED = [(48, 32, 255)]        # 32 agents need the 32-bit counter table: 255^2 of them do not fit in shared memory
STEPS = 3


# ------------------------------------------------------------------------------------------------ state builders
def window(x, xa, G):
    """numpy's x edges of the state's own observation window."""
    m = so.sequential_mean_x(x, xa)
    return so.box_edges(m - W / 2.0, m + W / 2.0, G)


def edge_distance(p, ex):
    """distance of every p to the nearest of numpy's edges, in bins"""
    i = np.clip(np.searchsorted(ex, p), 1, len(ex) - 1)
    step = (ex[-1] - ex[0]) / (len(ex) - 1)
    return np.minimum(np.abs(p - ex[i - 1]), np.abs(p - ex[i])) / step


def settle(x, xa, G, pins=(), groups=(), margin=0.05):
    """In place: pins [(arr, k, i)] put x of point k of arr (x or xa) exactly on edge i of the state's own window; groups
    [(arr, idx, cell, frac)] put points at lo + (cell + frac) * step of it; every other point is moved to the middle of
    its bin if it is within `margin` bins of an edge.  Every move shifts the window (the mean moves with the points), so
    this iterates to the fixed point."""
    free = {id(x): np.ones(len(x), dtype=bool), id(xa): np.ones(len(xa), dtype=bool)}
    for a, k, _ in pins:
        free[id(a)][k] = False
    for a, idx, _, _ in groups:
        free[id(a)][idx] = False
    for _ in range(400):
        ex = window(x, xa, G)
        lo, step = ex[0], (ex[-1] - ex[0]) / G
        moved = False
        for a, k, i in pins:
            moved |= a[k, 0] != ex[i]
            a[k, 0] = ex[i]
        for a, idx, cell, frac in groups:
            new = lo + (cell + frac) * step
            if np.abs(a[idx, 0] - new).max() > 1e-6 * step:        # (inside a bin: no need to land on the last bit)
                a[idx, 0] = new
                moved = True
        for a in (x, xa):
            t = (a[:, 0] - lo) / step
            fr = t - np.floor(t)
            bad = free[id(a)] & ((fr < margin) | (fr > 1.0 - margin)) & (t > -1.0) & (t < G + 1.0)
            if bad.any():
                a[bad, 0] = lo + (np.floor(t[bad]) + 0.5) * step
                moved = True
        if not moved:
            return
    raise AssertionError("settle did not converge")


def ulps(v, n):
    for _ in range(abs(n)):
        v = np.nextafter(v, np.inf if n > 0 else -np.inf)
    return v


def base_state(rs, N, A, G, centre=0.0, airborne=2, avoid=None):
    """Grounded locusts spread over the middle of a window around `centre`, agents grounded except `airborne` of them."""
    step = W / G
    lo = centre - W / 2.0
    t = rs.uniform(0.1 * G, 0.9 * G, size=N)
    if avoid is not None:                                   # keep the cells [avoid - 1, avoid + 2) free of locusts
        t = np.where((t > avoid - 1) & (t < avoid + 2), t + 4.0 * (1 if avoid < G / 2 else -1), t)
    x = np.stack([lo + t * step, np.zeros(N)], axis=1)
    xa = np.stack([lo + rs.uniform(0.05 * G, 0.95 * G, size=A) * step, np.zeros(A)], axis=1)
    if A > 2 and airborne:
        xa[1:1 + airborne, 1] = rs.uniform(0.3, 5.5, size=airborne)
    return x, xa


def stationary(x, xa, vr=None):
    """-> (v, reward) of the oracle if it keeps (x, xa) exactly where they are under actions (-1, 0) and zero noise with
    every locust pushed down by at least 0.05 (so the FP32 forces of the kernel cannot lift one either), else None.
    so.step, spelled out to keep its forces: the agents move first, the locusts feel the agents' new positions.  vr: the
    oracle's (v, reward) of this state if already known."""
    ya = xa.copy()
    va = np.zeros_like(ya)
    va[:, 0] = -1.0 + so.WIND_SPEED
    so.move_(ya, va, np.zeros_like(ya))
    if not np.array_equal(ya, xa):
        return None
    v, r = so.forces(x[None], ya[None]) if vr is None else (vr[0][None], np.array([vr[1]]))
    y = x.copy()
    so.move_(y, v[0].copy(), np.zeros_like(y))
    if not (np.array_equal(y, x) and (v[0, :, 1] <= -0.05).all()):
        return None
    return v[0], r[0]


class T(object):
    """One state: name, x (N,2), xa (A,2), edge (built so that the parallel mean must be rejected), check ((grid,
    positions, N) -> whether the oracle's observation has the property the state was built for), v / reward (oracle)."""

    def __init__(self, name, x, xa, edge, check, vr):
        self.name, self.x, self.xa, self.edge, self.check = name, x, xa, edge, check
        self.v, self.reward = vr


def pile_check(G, count, cell):
    def check(grid, pos, N):
        return int(round(grid[cell[0], cell[1], 0] * N)) == count
    return check


@functools.lru_cache(maxsize=None)
def templates(N, A, G):
    rs = np.random.RandomState(N * 1000 + A * 10 + G)
    out = []

    def add(name, x, xa, edge, check=None):
        vr = stationary(x, xa)
        if vr is None:                     # an airborne agent pulls too hard: ground it (its cell is not the point)
            xa[:, 1] = np.where(xa[:, 1] > Y_HI, xa[:, 1], 0.0)
            vr = stationary(x, xa)
            assert vr is not None, name
        out.append(T(name, x, xa, edge, check, vr))

    inner = (G // 2 + 3) if G > 4 else 1
    # -- a locust / an agent exactly on numpy's first, an inner and the last edge, and 1..3 ulps beside it
    for who in ("locust", "agent"):
        for i in (0, inner, G):
            x, xa = base_state(rs, N, A, G)
            arr = x if who == "locust" else xa
            k = int(np.argmin(np.abs(arr[:, 0] - window(x, xa, G)[i])))
            if who == "agent":
                xa[k, 1] = 0.0
            settle(x, xa, G, pins=[(arr, k, i)])
            assert arr[k, 0] == window(x, xa, G)[i]
            for n in (0, 1, -1, 2, -2, 3, -3):
                y, ya = x.copy(), xa.copy()
                (y if who == "locust" else ya)[k, 0] = ulps(arr[k, 0], n)
                add("%s_on_edge_%d_%+d_ulp" % (who, i, n), y, ya, True)
    # -- agents outside the window (digitize 0, clamp to G - 1), on / above the closed top edge, on the ground
    for with_edge in (False, True):
        x, xa = base_state(rs, N, A, G, airborne=0)
        k_out = [k for k in range(A)][:5]
        groups = [(xa, np.array(k_out[:1]), -3, 0.5)]                     # left of lo
        if A > 1:
            groups.append((xa, np.array(k_out[1:2]), G + 4, 0.5))       # right of hi
        pins = [(x, 0, inner)] if with_edge else []
        settle(x, xa, G, pins=pins, groups=groups)
        if A > 2:
            xa[2, 1] = Y_HI
        if A > 3:
            xa[3, 1] = np.nextafter(Y_HI, np.inf)
        if A > 4:
            xa[4, 1] = 0.0
        if A == 1:
            xa[0, 1] = Y_HI
        add("agents_outside_top_ground%s" % ("_edge" if with_edge else ""), x, xa, with_edge)
    # -- windows far from the origin, fast and with a locust on an edge
    for c in (40.0, -40.0, 1e4, -1e4, 1e6, -1e6):
        for with_edge in (False, True):
            x, xa = base_state(rs, N, A, G, centre=c)
            settle(x, xa, G, pins=[(x, 1, inner + (1 if c > 0 else -1))] if with_edge else [])
            add("far_%g%s" % (c, "_edge" if with_edge else ""), x, xa, with_edge)
    # -- absurd magnitude: the error bound itself sends the env to the sequential mean
    for s in (1.0, -1.0):
        x, xa = base_state(rs, N, A, G)
        x[0, 0] = s * 1.2345e13
        add("absurd_%+g" % (s * 1.2345e13), x, xa, True)
    # -- pile-ups across the look-up-table boundary (255 / 256 / 257 locusts in one cell)
    if N >= 700:
        pc = G // 4
        for count in (255, 256, 257):
            for with_edge in (False, True):
                x, xa = base_state(rs, N, A, G, avoid=pc)
                idx = np.arange(N - count, N)
                frac = np.sort(rs.uniform(0.3, 0.7, size=count))
                for _ in range(20):        # the window follows the pile: move the other locusts out of its cells
                    settle(x, xa, G, pins=[(x, 0, 3 * G // 4)] if with_edge else [], groups=[(x, idx, pc, frac)])
                    ex = window(x, xa, G)
                    t = (x[:N - count, 0] - ex[0]) / (W / G)
                    clash = np.nonzero((t > pc - 1) & (t < pc + 2))[0]
                    if not len(clash):
                        break
                    x[clash, 0] += 5.0 * W / G
                add("pile_%d%s" % (count, "_edge" if with_edge else ""), x, xa, with_edge,
                    pile_check(G, count, (pc, 0)))
    # -- every point in one cell: the half-word of a 16-bit counter at its maximum for N = 2047, A = 31.  All points share
    #    one x: the mean of the window is inside the pile, so for an even G the pile sits on numpy's middle edge (only
    #    identical points stay in one cell) and the env takes the fall-back; for an odd G it is the middle of a bin.
    X = 0.123456789
    x = np.stack([np.full(N, X), np.zeros(N)], axis=1)
    xa = np.stack([np.full(A, X), np.zeros(A)], axis=1)
    cx = int(np.searchsorted(window(x, xa, G), X, side="right")) - 1
    add("all_in_one_cell", x, xa, G % 2 == 0, pile_check(G, N, (cx, 0)))
    # ... and the other cell of the same 32-bit counter word, (bx, 1), holds the last agent (airborne, above the pile)
    xa = xa.copy()
    xa[-1, 1] = 1.5 * Y_HI / G
    cx = int(np.searchsorted(window(x, xa, G), X, side="right")) - 1
    add("all_in_one_cell_partner_occupied", x, xa, G % 2 == 0, pile_check(G, N, (cx, 0)))
    # -- benign: grounded random states, nowhere near an edge
    for b in range(6):
        x, xa = base_state(rs, N, A, G, centre=rs.uniform(-3.0, 3.0) * b)
        settle(x, xa, G)
        add("benign_%d" % b, x, xa, False)
    return out


@functools.lru_cache(maxsize=None)
def oracle(N, A, G):
    """(grid f32 (T,G,G,2), positions u8 (T,A,2), v f64 (T,N,2), reward f64 (T,)) of every template."""
    ts = templates(N, A, G)
    grids, pos = zip(*[so.rasterize(t.x, t.xa, G) for t in ts])
    return (np.stack(grids).astype(np.float32), np.stack(pos), np.stack([t.v for t in ts]),
            np.array([t.reward for t in ts]))


# ------------------------------------------------------------------------------------------------ CPU checks
@pytest.mark.parametrize("N,A,G", CASES + [(48, A, G) for G, A in LOCAL_CASES])
def test_states_are_stationary_and_hit_their_targets(N, A, G):
    ts = templates(N, A, G)
    names = [t.name for t in ts]
    assert len(names) == len(set(names))
    grids, pos, v, _ = oracle(N, A, G)
    for t, g, p in zip(ts, grids, pos):
        assert t.x.shape == (N, 2) and t.xa.shape == (A, 2)
        assert stationary(t.x, t.xa, (t.v, t.reward)) is not None, t.name
        assert (t.x[:, 1] == 0.0).all(), t.name
        if t.check is not None:
            assert t.check(g, p, N), t.name
        ex = window(t.x, t.xa, G)
        pts = np.concatenate([t.x[:, 0], t.xa[:, 0]])
        if "on_edge" in t.name and t.name.endswith("_+0_ulp"):
            i = int(t.name.split("_")[3])
            assert (pts == ex[i]).any(), t.name                       # exactly on numpy's edge i
        if t.name.startswith("locust_on_edge_%d_" % G) and t.name.endswith("_+0_ulp"):
            assert (t.x[:, 0] == ex[-1]).any()                        # x == hi: the closed right edge
    assert (v[:, :, 1] <= -0.05).all()
    # the classes the GPU tests rely on are all there, each several times
    for prefix, least in (("locust_on_edge", 21), ("agent_on_edge", 21), ("far_", 12), ("absurd", 2),
                          ("all_in_one_cell", 2), ("benign", 6), ("agents_outside", 2)):
        assert sum(n.startswith(prefix) for n in names) >= least, prefix
    if N >= 700:
        assert sum(n.startswith("pile_") for n in names) == 6
    # x == hi appears among the locusts, clamped positions among the agents
    assert any((t.x[:, 0] == window(t.x, t.xa, G)[-1]).any() for t in ts)
    assert (pos[:, :, 0] == G - 1).any() and (pos[:, :, 1] == G - 1).any() and (pos[:, :, 0] == 0).any()


def count_le(p, lo, hi, step, inv_step, G):
    """csrc/swarm_kernels.cuh count_le restated: #{numpy edges <= p}, from a reciprocal-multiply guess that is trusted
    only when its fractional part is further than the guess's error bound from 0 and 1, else from the exact edges."""
    if p == lo:
        return 1
    q = (p - lo) * inv_step
    fl = np.floor(q)
    fr = q - fl
    slack = 1e-9 + 16.0 * max(abs(lo), abs(hi)) * 2.220446049250313e-16 * inv_step
    if 0.0 < q < G and slack < fr < 1.0 - slack:
        return int(fl) + 1
    e = so.box_edges(lo, hi, G)
    return int(np.searchsorted(e, p, side="right"))


@pytest.mark.parametrize("N,A,G", CASES)
def test_count_le_guess_is_never_trusted_wrongly(N, A, G):
    """The fall-back bins x against numpy's exact edges with count_le: its guess must never be trusted when it is wrong,
    also far from the origin, where one ulp of the window's position is several 1e-9 bins (+-1e6: ~3e-9)."""
    for t in templates(N, A, G):
        ex = window(t.x, t.xa, G)
        lo, hi = ex[0], ex[-1]
        step = (hi - lo) / G
        for p in np.concatenate([t.x[:, 0], t.xa[:, 0]]):
            assert count_le(p, lo, hi, step, 1.0 / step, G) == np.searchsorted(ex, p, side="right"), (t.name, p)


@pytest.mark.parametrize("N,A,G", CASES)
def test_acceptance_rule_rejects_every_edge_state_and_accepts_the_rest(N, A, G):
    """env_raster's acceptance rule, restated for any G: each state built around an edge must go to the sequential
    fall-back (else the GPU tests would not run it), each other state must take the fast path, and whatever the rule
    accepts has numpy's own bins.  Two summation orders stand in for the kernel's tree."""
    rs = np.random.RandomState(G)
    ts = templates(N, A, G)
    for t in ts:
        P = N + A
        for order in (np.arange(P), rs.permutation(P)):
            cx, ok = spec_counts(t.x, t.xa, order, G)
            assert ok == (not t.edge), (t.name, ok)
            if ok:
                m = so.sequential_mean_x(t.x, t.xa)
                ex = so.box_edges(m - W / 2.0, m + W / 2.0, G)
                px = np.concatenate([t.x[:, 0], t.xa[:, 0]])
                assert np.array_equal(cx, np.searchsorted(ex, px, side="right")), t.name
                assert edge_distance(px, ex).min() > 0.01, t.name
    assert sum(t.edge for t in ts) >= 40 and sum(not t.edge for t in ts) >= 12


# ------------------------------------------------------------------------------------------------ GPU checks
@pytest.fixture(scope="module")
def M(pkg, cuda):
    return pkg.submodule("envs.multiagent")


PLACES = {"warps": 2 << 4, "warps_static": 2 << 4, "self": 3 << 4, "follow": 1 << 4, "auto": 0}
FALLBACK = {"follow": {"follower kernel", "raster warps in k_step", "k_step's own threads"},
            "warps": {"raster warps in k_step", "k_step's own threads"}, "warps_static": {"raster warps in k_step",
            "k_step's own threads"}, "self": {"k_step's own threads"},
            "auto": {"follower kernel", "raster warps in k_step", "k_step's own threads"}}


def new_env(M, N, A, G, E, variant, **kw):
    env = M.BatchedSwarmEnv(E, n_locusts=N, n_agents=A, grid_size=G, max_episode_steps=0, auto_reset=False,
                            binding="ctypes", tuning=PLACES[variant], **kw)
    if variant == "warps_static":
        env.state_c.work, env.state_c.work_words = None, 0       # static assignment: CTA c takes envs c, c + ctas, ...
    return env


def wave_width(plan):
    """envs per wave: one per persistent CTA of the placement that runs (1 where every env has a CTA of its own)"""
    if plan["raster_place"] == "follower kernel":
        return plan["follower_ctas"]
    if plan["raster_place"] == "raster warps in k_step":
        return plan["ctas"]
    return 1


@functools.lru_cache(maxsize=None)
def sized(N, A, G, variant):
    """(E, wave width): persistent placements get E = 3 x (their CTAs), so that each CTA rasterises several envs; one env
    per CTA placements get every template twice."""
    n = len(templates(N, A, G))
    if variant in ("self", "auto"):
        return 2 * n, None
    import golds_rl_gym_b200 as pkg
    M = pkg.submodule("envs.multiagent")
    probe = new_env(M, N, A, G, 148 * 32, variant)      # more envs than any B200 holds CTAs: ctas = slots
    w = wave_width(probe.plan())
    del probe
    return max(3 * w, 2 * n), w


def dynamic_queue(env, plan, N, A):
    """plan_step's rule for the work queue (raster warps only): a queue in SwarmState, every CTA with >= 3 envs, big envs"""
    return (plan["raster_place"] == "raster warps in k_step" and env.state_c.work is not None and
            env.E >= 3 * plan["ctas"] and N * (N + A) >= 16384)


def assignment(N, A, G, E, w, edge_first):
    """template index of every env: waves of w envs alternate between edge states and the others"""
    ts = templates(N, A, G)
    edge = [i for i, t in enumerate(ts) if t.edge]
    fast = [i for i, t in enumerate(ts) if not t.edge]
    w = w or 1
    idx = np.empty(E, dtype=np.int64)
    for e in range(E):
        kind = ((e // w) % 2 == 0) == edge_first
        pool = edge if kind else fast
        idx[e] = pool[(e // (2 * w) * w + e % w) % len(pool)]
    return idx


def run(M, N, A, G, variant, edge_first=True, math_mode="fast", noise="frozen", unaligned=False, E=None):
    """Three steps of the stationary batch; every env's observation, forces and reward against the oracle.  -> plan()"""
    ts = templates(N, A, G)
    g_ref, p_ref, v_ref, r_ref = oracle(N, A, G)
    if E is None:
        E, w = sized(N, A, G, variant)
    else:
        w = None
    env = new_env(M, N, A, G, E, variant, math_mode=math_mode, noise=noise)
    grid_out = None
    if unaligned:                          # a grid whose data is 8-byte, not 16-byte, aligned: no TMA, no filler warp
        flat = torch.zeros(E * G * G * 2 + 2, dtype=torch.float32, device=env.device)
        grid_out = flat[2:].view(E, G, G, 2)
        assert grid_out.data_ptr() % 16 == 8
        env.grid, env._grid_ptr = grid_out, grid_out.data_ptr()      # plan() reports the shape for this grid
    plan = env.plan()
    assert plan["raster_place"] in FALLBACK[variant], (variant, plan)
    if w is not None:
        assert wave_width(plan) == w, (plan, w)
    idx = assignment(N, A, G, E, wave_width(plan) if w is None else w, edge_first)
    dev = env.device
    x0 = torch.as_tensor(np.stack([ts[i].x for i in idx])).to(dev)
    xa0 = torch.as_tensor(np.stack([ts[i].xa for i in idx])).to(dev)
    env.x.copy_(x0); env.xa.copy_(xa0)
    env.noise_x.zero_(); env.noise_a.zero_()
    env._was_reset = True
    it = torch.as_tensor(idx, device=dev)
    g_want = torch.as_tensor(g_ref).to(dev)[it]
    p_want = torch.as_tensor(p_ref).to(dev)[it]
    v_want = torch.as_tensor(v_ref).to(dev)[it]
    r_want = torch.as_tensor(r_ref).to(dev)[it]
    act = torch.zeros(E, A, 2, dtype=torch.float32, device=dev)
    act[..., 0] = -1.0                                   # + wind 1 = no motion
    v = torch.empty(E, N, 2, dtype=torch.float32, device=dev)
    over = {}
    if noise == "fresh":                                 # the fresh rows are Philox draws: override them with zeros
        over = dict(noise_a=torch.zeros(E, A, 2, dtype=torch.float64, device=dev),
                    noise_x=torch.zeros(E, N, 2, dtype=torch.float64, device=dev))
    for step in range(STEPS):
        env.grid.fill_(np.nan)                           # every cell must be written, zeros included
        env.positions.fill_(255)
        env.step(act, v_out=v, grid_out=grid_out, **over)
        torch.cuda.synchronize()
        where = (variant, (N, A, G), step, plan["raster_place"])
        assert torch.equal(env.x, x0) and torch.equal(env.xa, xa0), where
        bad = ~((env.grid == g_want).flatten(1).all(1) & (env.positions == p_want).flatten(1).all(1))
        assert not bad.any(), (where, sorted({ts[idx[e]].name for e in torch.nonzero(bad)[:, 0].tolist()})[:12])
        rbad = (env.reward.double() - r_want).abs() > RTOL * r_want.abs()
        assert not rbad.any(), (where, sorted({ts[idx[e]].name for e in torch.nonzero(rbad)[:, 0].tolist()})[:12])
        verr = (v.double() - v_want).abs().amax((1, 2)) / v_want.abs().amax((1, 2))
        assert (verr <= RTOL).all(), (where, float(verr.max()), ts[idx[int(verr.argmax())]].name)
        assert int(env.work.sum()) == 0, where
    plan["dynamic"] = dynamic_queue(env, plan, N, A)
    plan["E"] = E
    return plan


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["warps", "warps_static", "self", "follow", "auto"])
@pytest.mark.parametrize("N,A,G", CASES)
def test_fused_rasteriser_on_edges_every_placement(M, N, A, G, variant):
    orders = (True, False) if variant in ("warps", "warps_static", "follow") else (True,)
    for edge_first in orders:
        run(M, N, A, G, variant, edge_first=edge_first)


@pytest.mark.gpu
def test_launch_matrix_covers_every_branch(M):
    """Which (case, placement) pairs the tests above realise, read from plan() for the batch sizes they use: every
    placement with both counter tables, SELF with and without the filler warp, raster warps with the work queue and
    with static assignment."""
    seen = set()
    lines = []
    for N, A, G in CASES:
        for variant in PLACES:
            E, _ = sized(N, A, G, variant)
            env = new_env(M, N, A, G, E, variant)
            plan = env.plan()
            place = {"follower kernel": "FOLLOW", "raster warps in k_step": "WARPS",
                     "k_step's own threads": "SELF"}[plan["raster_place"]]
            t32 = not (N < 2048 and A < 32)
            extra = ("queue" if dynamic_queue(env, plan, N, A) else "static") if place == "WARPS" else \
                    ("filler" if plan["filler_warp"] else "no filler") if place == "SELF" else ""
            seen.add((place, t32, extra))
            seen.add((place, t32))
            lines.append("(%d,%d,%d) %-12s -> %-6s %-9s table %d  E=%d ctas=%d follower_ctas=%d" % (
                N, A, G, variant, place, extra, 32 if t32 else 16, E, plan["ctas"], plan["follower_ctas"]))
            del env
    print("\n".join(lines))
    for place in ("WARPS", "SELF", "FOLLOW"):
        for t32 in (False, True):
            assert (place, t32) in seen, (place, t32, lines)
    for need in (("SELF", False, "filler"), ("SELF", False, "no filler"), ("WARPS", False, "queue"),
                 ("WARPS", False, "static")):
        assert need in seen, (need, lines)


@pytest.mark.gpu
@pytest.mark.parametrize("N,A,G", REFUSED)
def test_unsupported_size_is_refused_at_construction(M, N, A, G):
    with pytest.raises(M.nat.SwarmNativeError, match="unsupported size"):
        M.BatchedSwarmEnv(4, n_locusts=N, n_agents=A, grid_size=G)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["warps", "self", "follow"])
@pytest.mark.parametrize("N,A,G", [(48, 10, 84), (176, 10, 83), (2047, 31, 84)])
@pytest.mark.parametrize("kind", ["precise", "fresh"])
def test_other_step_instantiations(M, N, A, G, variant, kind):
    """math_mode="precise" compiles separate k_step instantiations (each with its own inlined env_raster); noise="fresh"
    takes the step's Philox branch, here overridden by zero rows."""
    if kind == "precise":
        run(M, N, A, G, variant, math_mode="precise")
    else:
        run(M, N, A, G, variant, noise="fresh")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["warps", "self", "follow"])
def test_grid_view_not_16_byte_aligned(M, variant):
    """An observation slot that is only 8-byte aligned: the TMA zero fill and the filler warp are off, the zeros go out
    as plain stores (G = 84 would otherwise always use TMA)."""
    N, A, G = 176, 10, 84
    plan = run(M, N, A, G, variant, unaligned=True, E=2 * len(templates(N, A, G)))
    assert plan["filler_warp"] == 0


@pytest.mark.gpu
def test_grid_not_8_byte_aligned_is_refused(M):
    """A cell's two channels are one float2: a grid that is only 4-byte aligned is refused before anything is launched,
    by the step, the standalone rasteriser and local_states."""
    N, A, G, E = 48, 10, 84, 2
    env = new_env(M, N, A, G, E, "auto")
    env.reset()
    flat = torch.zeros(E * G * G * 2 + 1, dtype=torch.float32, device=env.device)
    bad = flat[1:].view(E, G, G, 2)
    assert bad.data_ptr() % 8 == 4
    act = torch.zeros(E, A, 2, dtype=torch.float32, device=env.device)
    with pytest.raises(M.nat.SwarmNativeError, match="flags"):
        env.step(act, grid_out=bad)
    env.grid = bad
    with pytest.raises(M.nat.SwarmNativeError, match="flags"):
        env.observe()
    with pytest.raises(M.nat.SwarmNativeError, match="flags"):
        env.local_states()
    torch.cuda.synchronize()
    assert (flat == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("N,A,G", [(176, 10, 83), (700, 10, 84), (2047, 31, 84), (80, 1, 2), (80, 10, 255)])
def test_standalone_rasteriser_on_the_same_states(M, N, A, G):
    """observe() (k_rasterize: verified parallel mean, and always sequential when the box is asked for) on every state."""
    ts = templates(N, A, G)
    g_ref, p_ref, _, _ = oracle(N, A, G)
    env = new_env(M, N, A, G, len(ts), "auto")
    env.x.copy_(torch.as_tensor(np.stack([t.x for t in ts])).cuda())
    env.xa.copy_(torch.as_tensor(np.stack([t.xa for t in ts])).cuda())
    for box in (None, torch.zeros(len(ts), 4, dtype=torch.float64, device="cuda")):
        env.grid.fill_(np.nan)
        grid, pos = env.observe(box=box)
        grid, pos = grid.cpu().numpy(), pos.cpu().numpy()
        for e, t in enumerate(ts):
            assert np.array_equal(grid[e], g_ref[e]) and np.array_equal(pos[e], p_ref[e]), (t.name, box is None)


@pytest.mark.gpu
@pytest.mark.parametrize("G,A", LOCAL_CASES)
def test_local_states_of_the_fused_observation(M, G, A):
    """k_expand (local_states) bit-exact against the oracle's get_local_states, on the observations of the edge states:
    several agents in one cell, positions at 0 and clamped to G - 1."""
    N = 48
    if (N, A, G) in REFUSED:
        with pytest.raises(M.nat.SwarmNativeError, match="unsupported size"):
            M.BatchedSwarmEnv(4, n_locusts=N, n_agents=A, grid_size=G)
        return
    ts = templates(N, A, G)
    E = len(ts)
    run(M, N, A, G, "auto", E=E)
    env = new_env(M, N, A, G, E, "auto")
    env.x.copy_(torch.as_tensor(np.stack([t.x for t in ts])).cuda())
    env.xa.copy_(torch.as_tensor(np.stack([t.xa for t in ts])).cuda())
    env._was_reset = True
    act = torch.zeros(E, A, 2, dtype=torch.float32, device=env.device)
    act[..., 0] = -1.0
    env.step(act)
    loc = env.local_states().cpu().numpy()
    grid, pos = env.grid.cpu().numpy(), env.positions.cpu().numpy()
    g_ref, p_ref, _, _ = oracle(N, A, G)
    assert np.array_equal(grid, g_ref) and np.array_equal(pos, p_ref)
    for e in range(E):
        assert np.array_equal(loc[e], so.local_states(g_ref[e], p_ref[e])), ts[e].name
    assert (pos == G - 1).any() and (pos == 0).any()
    if A > 1:
        assert any(len({tuple(p) for p in pos[e]}) < A for e in range(E))      # several agents share a cell
