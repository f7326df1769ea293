#!/usr/bin/env python
"""Cost of fresh per-step noise (BatchedSwarmEnv(noise="fresh"), SWARM_STEP_FRESH_NOISE) against the frozen row.

    python scripts/fresh_noise_ab.py [--shapes 4096x256 512x256 ...] [--rounds 7] [--out profiles/r03_fresh_noise_ab.json]

Steady-state microseconds per batch-step as in DESIGN.md section 5: a CUDA graph of 8 steps, replayed.  For every shape
a frozen and a fresh env (same seed, automatic launch shape, TimeLimit 128) are timed in alternation, in one process,
over several rounds (the order flips every round), in two windows:
  steady    8 replays = 64 steps inside an episode (elapsed set to 0 first: no boundary in the window);
  episode   16 replays = 128 steps from elapsed 0: the last one auto-resets every env (10 burn-in steps each).
The GPU's name and power limit are read in the same run and stored with the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES = ["4096x256", "1024x256", "512x256", "4096x80", "1024x80", "1024x64"]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clock = [s.strip() for s in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:                     # the numbers still carry the device name torch reports
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % exc}


def graph_of(env, acts):
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):               # warm-up outside the capture
        for a in acts:
            env.step(a)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for a in acts:
            env.step(a)
    return g


def timed_us_per_step(env, g, replays):
    import torch
    env.elapsed.zero_()                         # stream-ordered before the first event: not timed
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (8 * replays)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--shapes", nargs="+", default=SHAPES)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None, help="JSON file for the table (default: print only)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("fresh_noise_ab.py measures the GPU: no CUDA device")
    import golds_rl_gym_b200 as pkg
    M = pkg.submodule("envs.multiagent")
    info = gpu_info()
    rows = []
    for shape in args.shapes:
        E, N = (int(v) for v in shape.split("x"))
        gen = torch.Generator(device="cuda"); gen.manual_seed(1234)
        acts = []
        for _ in range(8):
            a = torch.randn(E, 10, 2, device="cuda", generator=gen)
            n = a.norm(dim=-1, keepdim=True)
            acts.append(torch.where(n >= 1.0, a / n, a).contiguous())
        runs = {}
        for mode in ("frozen", "fresh"):
            env = M.BatchedSwarmEnv(E, n_locusts=N, seed=1234, max_episode_steps=128, noise=mode)
            env.reset()
            runs[mode] = (env, graph_of(env, acts), {"steady": [], "episode": []})
        plan = runs["frozen"][0].plan()
        for r in range(args.rounds):
            for mode in (("frozen", "fresh") if r % 2 == 0 else ("fresh", "frozen")):
                env, g, t = runs[mode]
                timed_us_per_step(env, g, 2)                                  # back in cache / clocks after the switch
                t["steady"].append(timed_us_per_step(env, g, 8))
                t["episode"].append(timed_us_per_step(env, g, 16))
        row = {"shape": shape, "E": E, "N": N, "launch": plan["raster_place"], "ctas": plan["ctas"]}
        for win in ("steady", "episode"):
            fz, fr = runs["frozen"][2][win], runs["fresh"][2][win]
            row[win] = {"frozen_us_median": statistics.median(fz), "fresh_us_median": statistics.median(fr),
                        "frozen_us_min": min(fz), "fresh_us_min": min(fr),
                        "frozen_us_spread": max(fz) - min(fz), "fresh_us_spread": max(fr) - min(fr),
                        "delta_us": statistics.median(fr) - statistics.median(fz),
                        "delta_pct": 100.0 * (statistics.median(fr) / statistics.median(fz) - 1.0)}
        rows.append(row)
        print(json.dumps(row), flush=True)
        del runs
        torch.cuda.empty_cache()
    result = dict(info, rounds=args.rounds, method="CUDA graph of 8 steps replayed; median over rounds, frozen/fresh "
                  "alternated in one process; steady = 64 steps inside an episode, episode = 128 steps incl. the "
                  "lock-step auto-reset", rows=rows)
    print("| shape | launch | window | frozen us/step | fresh us/step | delta us | delta % |")
    print("|---|---|---|---|---|---|---|")
    for row in rows:
        for win in ("steady", "episode"):
            w = row[win]
            print("| %s | %s | %s | %.2f | %.2f | %+.2f | %+.1f |" % (row["shape"], row["launch"], win, w["frozen_us_median"],
                                                                    w["fresh_us_median"], w["delta_us"], w["delta_pct"]))
    print("(%s, power limit %s)" % (info["gpu"], info["power_limit"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
