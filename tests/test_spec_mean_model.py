"""CPU model of the rasteriser's verified parallel mean (csrc/swarm_kernels.cuh, env_raster) against the oracle.

The kernel bins every point against a tree-sum mean and accepts the result only if each point is further from the nearest
bin edge than a rigorous bound on everything that can separate that computation from numpy's (sequential mean, linspace
edges, searchsorted).  This test restates the acceptance rule in NumPy, arithmetic operation for arithmetic operation, and
checks the two properties the kernel relies on, on random and adversarial states:
  (1) soundness: whenever the rule accepts an env, the speculative x counts equal numpy's own (oracle) for EVERY point;
  (2) usefulness: random states are practically always accepted, states with a point on / next to an edge never are.
The CUDA path itself is compared with the oracle on such states in tests/test_gpu_parity.py
(test_rasterizer_verified_parallel_mean_next_to_edges: the standalone rasteriser behind observe()) and in
tests/test_gpu_raster_edges.py (the rasteriser inside the step, in every launch shape; it uses spec_counts to prove that
its states take the branch each of them targets).
"""
import numpy as np

from oracle import swarm_oracle as so

G, W = 84, so.BOX_WIDTH
EPS = 2.220446049250313e-16


def spec_counts(x, xa, order, G=G):
    """(#edges <= p for every point, accepted?) the way env_raster's speculative phase computes them for a G x G grid.
    `order` permutes the points before a pairwise sum: any summation order stands in for the kernel's warp-shuffle tree."""
    inv_x = G / W                                        # KP.inv_x (make_kp)
    px = np.concatenate([x[:, 0], xa[:, 0]])
    P = px.size
    tot = float(np.sum(px[order]))                       # pairwise, not sequential
    xmax = float(np.max(np.abs(px)))
    lo_s = tot * (1.0 / P) - W / 2.0
    tol = 1e-9 + 2.0 * ((P + 16) * xmax + 32.0 * (W / 2.0)) * EPS * inv_x
    qs = (px - lo_s) * inv_x
    fl = np.floor(qs)
    fr = qs - fl
    ok = bool(tol < 0.25) and bool(np.all((fr > tol) & (fr < 1.0 - tol)))
    cx = (np.minimum(np.maximum(fl, -1.0), float(G)) + 1).astype(np.int64)
    return cx, ok


def oracle_counts(x, xa):
    m = so.sequential_mean_x(x, xa)
    ex = so.box_edges(m - W / 2.0, m + W / 2.0, G)
    px = np.concatenate([x[:, 0], xa[:, 0]])
    return np.searchsorted(ex, px, side="right"), ex


def test_accepted_envs_have_numpys_bins():
    rs = np.random.RandomState(3)
    accepted = total = 0
    for trial in range(3000):
        N = int(rs.choice([5, 33, 64, 80, 256, 700]))
        shift = rs.uniform(-300.0, 300.0) if trial % 3 else 0.0
        x = rs.rand(N, 2) * [rs.uniform(0.5, 5.0), 2.0] + [shift, 0.0]
        xa = rs.rand(10, 2) * [4.0, 3.0] + [shift - 0.5, 0.0]
        cx, ok = spec_counts(x, xa, rs.permutation(N + 10))
        ref, _ = oracle_counts(x, xa)
        total += 1
        if ok:
            accepted += 1
            assert np.array_equal(cx, ref), trial
    assert accepted >= 0.99 * total, (accepted, total)      # random states: the sequential chain is practically never needed


def test_points_next_to_an_edge_are_never_accepted():
    rs = np.random.RandomState(4)
    for trial in range(400):
        N = int(rs.choice([33, 64, 80, 256]))
        x = rs.rand(N, 2) * [2.5, 1.5] + [rs.uniform(-60.0, 60.0), 0.0]
        xa = rs.rand(10, 2) * [3.4, 3.0] + [x[:, 0].mean() - 1.7, 0.0]
        j, i = rs.randint(N), (0, G, rs.randint(1, G))[trial % 3]
        for _ in range(40):                  # fixed point: the window moves with the point that is put on its edge
            _, ex = oracle_counts(x, xa)
            x[j, 0] = ex[i]
        for ulps in (0, 1, -1, 4, -7):
            y = x.copy()
            for _ in range(abs(ulps)):
                y[j, 0] = np.nextafter(y[j, 0], np.inf if ulps > 0 else -np.inf)
            cx, ok = spec_counts(y, xa, rs.permutation(N + 10))
            ref, ex = oracle_counts(y, xa)
            near = np.min(np.abs(ex - y[j, 0])) < 1e-10
            if near:                         # (the fixed point converged onto the edge: always, except for tiny P)
                assert not ok, (trial, ulps)
            if ok:
                assert np.array_equal(cx, ref), (trial, ulps)


def test_bound_dominates_the_difference_of_the_means():
    """The first term of the bound: |sequential mean - any-order mean| <= (P + 1) 2^-52 max|x|, observed with two orders
    of magnitude to spare."""
    rs = np.random.RandomState(5)
    worst = 0.0
    for trial in range(2000):
        N = int(rs.choice([64, 80, 256, 2048]))
        x = rs.rand(N, 2) * 3.0 + [rs.uniform(-100.0, 100.0), 0.0]
        xa = rs.rand(10, 2) * 3.0 + [x[0, 0], 0.0]
        px = np.concatenate([x[:, 0], xa[:, 0]])
        m_seq = so.sequential_mean_x(x, xa)
        m_par = float(np.sum(px[rs.permutation(px.size)])) * (1.0 / px.size)
        bound = (px.size + 1) * 2.0 ** -52 * np.max(np.abs(px))
        assert abs(m_seq - m_par) <= bound
        worst = max(worst, abs(m_seq - m_par) / bound)
    assert worst < 0.1
