"""Times the cluster layout (one env over the K CTAs of a thread-block cluster) against itself and the one-CTA kernels.

For each (N, E, layout) it replays a CUDA graph of 8 batch-steps (auto-reset, fused observation, fast math) and reports
the device time per batch-step (CUDA events) in steady state and with every env at its episode boundary (TimeLimit
reached: 10 burn-in steps follow), locust-updates/s, and ordered pairs/s against the 4-MUFU XU ceiling of ordered
pairs (2.33e12 pairs/s on a B200, DESIGN 3.1).  Layouts are timed in alternation, round by round, so that a drift of
the shared machine hits all of them alike; the median over rounds is reported.

    python scripts/cluster_bench.py --out profiles/r04_cluster
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

XU_PAIRS = 2.33e12


def force_warps(N):
    T = 2 if N <= 1024 else 4
    return (-(-N // T) + 31) // 32


def legal_k(N):
    nw = force_warps(N)
    return list(range(-(-nw // 32), min(16, nw) + 1))


def make(M, N, E, layout):
    """layout: 0 = one CTA per env, "auto" = the cluster layout at the library's K, K = a cluster of K CTAs"""
    from golds_rl_gym_b200 import _native as nat
    tuning = nat.TUNE_CLUSTER_AUTO if layout == "auto" else 0
    env = M.BatchedSwarmEnv(E, n_locusts=N, max_episode_steps=128, seed=1, binding="torch", tuning=tuning,
                            cluster=layout if isinstance(layout, int) and layout > 0 else None)
    env.reset()
    return env


class Case(object):
    def __init__(self, M, N, E, layout, steps=8):
        self.N, self.E, self.layout = N, E, layout
        self.env = env = make(M, N, E, layout)
        self.plan = env.plan()
        self.acts = torch.randn(E, env.A, 2, device=env.device).clamp_(-1, 1)
        env.step(self.acts)                                     # warm-up + caches, outside the capture
        self.g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            with torch.cuda.graph(self.g, stream=s):
                for _ in range(steps):
                    env.step(self.acts)
        torch.cuda.current_stream().wait_stream(s)
        self.steps = steps

    def time(self, boundary, reps):
        """us per batch-step: `reps` replays of the graph; boundary = every env hits its TimeLimit on the first step"""
        env, out = self.env, []
        st, en = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(reps):
            env.elapsed.fill_(127 if boundary else 8)
            st.record()
            self.g.replay()
            en.record()
            en.synchronize()
            out.append(st.elapsed_time(en) * 1e3 / self.steps)
        out.sort()
        return out[len(out) // 2] if not boundary else out[len(out) // 2] * self.steps - 7 * self.steady

    def free(self):
        del self.g
        del self.env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write OUT.json and OUT.md")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="a few shapes only (rehearsal)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cluster_bench.py needs a CUDA device")
    import golds_rl_gym_b200 as pkg
    M = pkg.submodule("envs.multiagent")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    groups = []
    if a.quick:
        groups.append([(4096, 1, k) for k in (1, 4, "auto")] + [(1024, 8, 0), (1024, 8, 2)])
    else:
        for N in (4096, 8192):
            for E in (1, 16, 148):
                groups.append([(N, E, k) for k in legal_k(N)] + [(N, E, "auto")])
        for N in (1024, 2048):
            for E in (1, 8, 32, 148, 1024):
                groups.append([(N, E, 0)] + [(N, E, k) for k in sorted({1, 2, 4, 8, legal_k(N)[-1]})] + [(N, E, "auto")])
    rows = []
    for grp in groups:
        cases = []
        for (N, E, k) in grp:
            try:
                cases.append(Case(M, N, E, k))
            except Exception as ex:          # a layout the device refuses (shared memory, unschedulable cluster)
                rows.append(dict(N=N, E=E, K=k, refused=str(ex).splitlines()[0]))
        res = {id(c): ([], []) for c in cases}
        for _ in range(a.rounds):
            for c in cases:
                c.steady = c.time(False, a.reps)
                res[id(c)][0].append(c.steady)
                res[id(c)][1].append(c.time(True, a.reps))
        for c in cases:
            s, b = sorted(res[id(c)][0]), sorted(res[id(c)][1])
            us, ub = s[len(s) // 2], b[len(b) // 2]
            pairs = c.E * c.N * (c.N + c.env.A)
            rows.append(dict(N=c.N, E=c.E, K=c.plan["cluster_size"], layout=c.plan["layout"],
                             requested={0: "one CTA"}.get(c.layout, c.layout), ctas=c.plan["ctas"],
                             threads=c.plan["threads"], us_step=round(us, 2), us_boundary_step=round(ub, 2),
                             locust_updates_per_s=c.E * c.N / (us * 1e-6), pairs_per_s=pairs / (us * 1e-6),
                             xu_share=pairs / (us * 1e-6) / XU_PAIRS))
            print(json.dumps(rows[-1]), flush=True)
            c.free()
        torch.cuda.empty_cache()
        if a.out:
            write(a.out, gpu, rows)


def write(out, gpu, rows):
    """OUT.json and OUT.md of the rows so far"""
    if out:
        with open(out + ".json", "w") as f:
            json.dump(dict(gpu=gpu, rows=rows), f, indent=1)
        with open(out + ".md", "w") as f:
            f.write("# Cluster layout: us per batch-step (%s)\n\n" % gpu)
            f.write("| N | E | requested | layout | K | CTAs | threads | us/step | us at the boundary | locust-upd/s | pairs/s | of XU ceiling |\n")
            f.write("|---|---|---|---|---|---|---|---|---|---|---|---|\n")
            for r in rows:
                if "refused" in r:
                    f.write("| %d | %d | %s | refused: %s |||||||||\n" % (r["N"], r["E"], r["K"], r["refused"][:80]))
                    continue
                f.write("| %d | %d | %s | %s | %d | %d | %d | %.2f | %.2f | %.3g | %.3g | %.1f %% |\n" % (
                    r["N"], r["E"], r["requested"], r["layout"], r["K"], r["ctas"], r["threads"], r["us_step"],
                    r["us_boundary_step"], r["locust_updates_per_s"], r["pairs_per_s"], 100 * r["xu_share"]))


if __name__ == "__main__":
    main()
