#!/usr/bin/env python
"""Cost of action repeat (BatchedSwarmEnv(action_repeat=K), swarm_step_repeat) against what a caller can build today.

    python scripts/action_repeat_ab.py [--shapes 4096x256 1024x64 ...] [--ks 1 2 4 8] [--rounds 5] [--out FILE.json]
    python scripts/action_repeat_ab.py --sass PARENT.so NEW.so        # CPU: SASS of the existing kernels unchanged?
    python scripts/action_repeat_ab.py --spills LIB.so                  # CPU: where the REP kernels spill

Microseconds per decision (one step() of the learner) and per physics step (decision / K), for three arms:
  fused     one repeat-K call (swarm_step_repeat);
  last_obs  K single steps, only the last one rasterises (the best a caller can do without the call; correct only when
            no episode ends inside the K steps);
  every_obs K single steps, each with an observation;
  fin_null  (K = 1 only) swarm_step_final with every terminal output NULL: the FIN kernel the REP kernels are built on,
            against the plain step (fused at K = 1) -- what the REP kernels' null-fin code costs per decision.
Each arm is a CUDA graph of 4 decisions, replayed; the arms (and the fused call in each forced raster placement, tuning
0x10 / 0x20 / 0x30) are timed in alternation, in one process, over several rounds (the order rotates every round).
Two windows:
  steady    no TimeLimit: no episode ends;
  boundary  TimeLimit K: every env ends on the decision's last physics step and auto-resets (10 burn-in steps).
The GPU's name and power limit are read in the same run and stored with the numbers.

--sass compares `cuobjdump -sass` of two builds of libswarm_b200.so: every kernel of PARENT must have the same
instructions in NEW (names matched after dropping the REP template argument and the repeat parameter).
"""
import argparse
import json
import os
import re
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

from env_physics_ab import sass_functions, spill_sites    # noqa: E402

SHAPES = ["4096x256", "1024x256", "512x256", "4096x80", "1024x80", "1024x64"]
KS = [1, 2, 4, 8]
ARMS = ("fused", "last_obs", "every_obs")
PLACES = {"follow": 0x10, "warps": 0x20, "self": 0x30}
DECISIONS = 4
SWARM_STEP_AUTO_RESET = 1


def sass_compare(parent, new):
    """-> (identical, differing names, missing names, count of REP kernels in new)."""
    old, cur = sass_functions(parent), sass_functions(new)
    strip, n_rep = {}, 0
    for name, body in cur.items():
        m = re.match(r"(.*)<(.*), \(bool\)([01])>\((.*), int\)$", name)
        if m and ("k_step" not in m.group(1)):
            m = None
        if m and m.group(3) == "1":
            n_rep += 1
            continue
        strip[(m.group(1) + "<" + m.group(2) + ">(" + m.group(4) + ")") if m else name] = body
    same, diff, missing = 0, [], []
    for name, body in old.items():
        if name not in strip:
            missing.append(name)
        elif strip[name] == body:
            same += 1
        else:
            diff.append(name)
    return same, diff, missing, n_rep


def is_rep(name):
    return bool(re.search(r"k_step(_cluster)?<.*, \(bool\)1>\(.*, int\)$", name))


def decision(env, a, K, arm):
    if arm == "fused":
        env.action_repeat = K
        env.step(a)
        return
    if arm == "fin_null":      # K = 1: the FIN kernel of swarm_step_final with every terminal output NULL
        env.action_repeat = 1
        env.ops.step_final(env._blob, *env._state_t, a, None, None, env.reward, env.done_u8, env.grid, env.positions,
                           None, SWARM_STEP_AUTO_RESET | env._noise_flag, [], None, None, None, None, None, None)
        return
    env.action_repeat = 1
    for s in range(K):
        env.step(a, rasterize=arm == "every_obs" or s == K - 1)


def graph_of(env, acts, K, arm):
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):               # warm-up outside the capture
        for a in acts:
            decision(env, a, K, arm)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for a in acts:
            decision(env, a, K, arm)
    return g


def timed_us_per_decision(env, g, replays):
    import torch
    env.elapsed.zero_()                         # stream-ordered before the first event: not timed
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (DECISIONS * replays)


def shape_rows(M, shape, ks, rounds):
    import torch
    E, N = (int(v) for v in shape.split("x"))
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1234)
    acts = []
    for _ in range(DECISIONS):
        a = torch.randn(E, 10, 2, device="cuda", generator=gen)
        n = a.norm(dim=-1, keepdim=True)
        acts.append(torch.where(n >= 1.0, a / n, a).contiguous())
    rows = []
    for K in ks:
        runs, plans = {}, {}
        for win, limit in (("steady", 0), ("boundary", K)):
            variants = [(arm, 0) for arm in ARMS] + ([("fused@" + p, t) for p, t in PLACES.items()] if win == "steady" else [])
            if K == 1:
                variants.append(("fin_null", 0))
            for name, tuning in variants:
                env = M.BatchedSwarmEnv(E, n_locusts=N, seed=1234, max_episode_steps=limit, tuning=tuning)
                env.reset()
                env.action_repeat = K if name.startswith("fused") else 1     # the kernels the arm launches
                plans[win, name] = env.plan()["raster_place"]
                runs[win, name] = (env, graph_of(env, acts, K, name.split("@")[0]), [])
        for r in range(rounds):
            keys = list(runs)
            keys = keys[r % len(keys):] + keys[:r % len(keys)]
            for key in keys:
                env, g, t = runs[key]
                timed_us_per_decision(env, g, 1)      # back in cache / clocks after the switch
                t.append(timed_us_per_decision(env, g, 4))
        env = runs["boundary", "fused"][0]
        torch.cuda.synchronize()
        assert bool(env.done_u8.all())                 # the boundary window really ends every env
        row = {"shape": shape, "E": E, "N": N, "K": K, "launch": plans["steady", "fused"]}
        for win in ("steady", "boundary"):
            row[win] = {}
            for (w, name), (_, _, t) in runs.items():
                if w != win:
                    continue
                med = statistics.median(t)
                row[win][name] = {"us_per_decision": med, "us_per_physics_step": med / K, "us_spread": max(t) - min(t),
                                  "place": plans[w, name]}
        rows.append(row)
        print(json.dumps(row), flush=True)
        del runs
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--shapes", nargs="+", default=SHAPES)
    ap.add_argument("--ks", nargs="+", type=int, default=KS)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="JSON file for the table (default: print only)")
    ap.add_argument("--sass", nargs=2, metavar=("PARENT_LIB", "NEW_LIB"))
    ap.add_argument("--spills", metavar="LIB", help="CPU: spill sites (STL / LDL) of every REP kernel by source line")
    args = ap.parse_args()
    if args.spills:
        bad = 0
        for name, st in sorted(spill_sites(args.spills).items()):
            if not is_rep(name) or not st:
                continue
            locs = sorted(set(l for _, l, _, _ in st))
            inloop = sorted(set(l for _, l, _, p in st if p))
            bad += len(inloop)
            print("%s: %d STL / %d LDL at %s%s" % (re.sub(r"\(swarm::KP.*", "", name).replace("void <unnamed>::", ""),
                                                  sum(k == "STL" for k, _, _, _ in st), sum(k == "LDL" for k, _, _, _ in st),
                                                  ", ".join(locs), ("  IN A PAIR LOOP: " + ", ".join(inloop)) if inloop else ""))
        raise SystemExit(1 if bad else 0)
    if args.sass:
        same, diff, missing, n_rep = sass_compare(*args.sass)
        print("existing kernels with identical SASS: %d; different: %d; missing: %d; REP kernels: %d"
              % (same, len(diff), len(missing), n_rep))
        for name in diff + missing:
            print("  ", name)
        raise SystemExit(1 if diff or missing else 0)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("action_repeat_ab.py measures the GPU: no CUDA device")
    import golds_rl_gym_b200 as pkg
    from fresh_noise_ab import gpu_info
    M = pkg.submodule("envs.multiagent")
    info = gpu_info()
    rows = []
    for shape in args.shapes:
        rows += shape_rows(M, shape, args.ks, args.rounds)
    result = dict(info, rounds=args.rounds, decisions_per_graph=DECISIONS,
                  method="CUDA graph of 4 decisions replayed; median over rounds, arms and forced placements rotated in "
                         "one process; steady = no TimeLimit, boundary = TimeLimit K (every env ends on the decision's "
                         "last physics step and auto-resets)", rows=rows)
    print("| shape | K | window | fused us/decision | last_obs | every_obs | fused us/physics step |")
    print("|---|---|---|---|---|---|---|")
    for row in rows:
        for win in ("steady", "boundary"):
            w = row[win]
            f = w["fused"]["us_per_decision"]
            print("| %s | %d | %s | %.2f | %.2f (%+.1f %%) | %.2f (%+.1f %%) | %.2f |" % (
                row["shape"], row["K"], win, f, w["last_obs"]["us_per_decision"],
                100.0 * (f / w["last_obs"]["us_per_decision"] - 1.0), w["every_obs"]["us_per_decision"],
                100.0 * (f / w["every_obs"]["us_per_decision"] - 1.0), w["fused"]["us_per_physics_step"]))
    print("| shape | K | automatic (place) | follow | warps | self |")
    print("|---|---|---|---|---|---|")
    for row in rows:
        w = row["steady"]
        print("| %s | %d | %.2f (%s) | %s |" % (row["shape"], row["K"], w["fused"]["us_per_decision"], w["fused"]["place"],
                                             " | ".join("%.2f (%s)" % (w["fused@" + p]["us_per_decision"],
                                                                       w["fused@" + p]["place"]) for p in PLACES)))
    print("| shape | window | plain step us | FIN kernel, fin all NULL, us (delta) |")
    print("|---|---|---|---|")
    for row in rows:
        if row["K"] != 1:
            continue
        for win in ("steady", "boundary"):
            f, n = row[win]["fused"]["us_per_decision"], row[win]["fin_null"]["us_per_decision"]
            print("| %s | %s | %.2f | %.2f (%+.2f us, %+.1f %%) |" % (row["shape"], win, f, n, n - f, 100.0 * (n / f - 1.0)))
    print("(%s, power limit %s)" % (info["gpu"], info["power_limit"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
