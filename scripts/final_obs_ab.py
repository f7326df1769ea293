#!/usr/bin/env python
"""Cost of the terminal outputs (BatchedSwarmEnv(final_obs=True), swarm_step_final) against the plain step.

    python scripts/final_obs_ab.py [--shapes 4096x256 64x8192 ...] [--rounds 7] [--paac 32 1024] [--out FILE.json]

Microseconds per batch-step, as in DESIGN.md section 5: a CUDA graph of 8 steps, replayed.  For every shape an env
without and one with the terminal outputs (same seed, automatic launch shape) are timed in alternation, in one
process, over several rounds (the order flips every round), in two windows:
  steady    TimeLimit 128, 8 replays = 64 steps inside an episode (elapsed set to 0 first): no env is done, the extra
            cost is the masked rasteriser launch whose CTAs all leave after reading one byte;
  boundary  TimeLimit 1: every step ends (and auto-resets) every env, so every step also copies the terminal state out
            and rasterises the terminal observation of the whole batch.
PAAC: frames/s of the graph-replayed update (mask_terminals=True) with and without bootstrap_truncated.
The GPU's name and power limit are read in the same run and stored with the numbers.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

from fresh_noise_ab import gpu_info, graph_of, timed_us_per_step      # noqa: E402

SHAPES = ["4096x256", "1024x256", "512x256", "4096x80", "1024x80", "1024x64", "64x8192"]


def shape_rows(M, shape, rounds):
    import torch
    E, N = (int(v) for v in shape.split("x"))
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1234)
    acts = []
    for _ in range(8):
        a = torch.randn(E, 10, 2, device="cuda", generator=gen)
        n = a.norm(dim=-1, keepdim=True)
        acts.append(torch.where(n >= 1.0, a / n, a).contiguous())
    runs = {}
    for win, limit in (("steady", 128), ("boundary", 1)):
        for mode in ("off", "on"):
            env = M.BatchedSwarmEnv(E, n_locusts=N, seed=1234, max_episode_steps=limit, final_obs=mode == "on")
            env.reset()
            runs[win, mode] = (env, graph_of(env, acts), [])
    plan = runs["steady", "off"][0].plan()
    for r in range(rounds):
        for win in ("steady", "boundary"):
            for mode in (("off", "on") if r % 2 == 0 else ("on", "off")):
                env, g, t = runs[win, mode]
                timed_us_per_step(env, g, 2)                # back in cache / clocks after the switch
                t.append(timed_us_per_step(env, g, 8))
    row = {"shape": shape, "E": E, "N": N, "launch": plan["raster_place"], "layout": plan["layout"]}
    for win in ("steady", "boundary"):
        off, on = runs[win, "off"][2], runs[win, "on"][2]
        row[win] = {"off_us_median": statistics.median(off), "on_us_median": statistics.median(on),
                    "off_us_spread": max(off) - min(off), "on_us_spread": max(on) - min(on),
                    "delta_us": statistics.median(on) - statistics.median(off),
                    "delta_pct": 100.0 * (statistics.median(on) / statistics.median(off) - 1.0)}
    done = runs["boundary", "on"][0]
    torch.cuda.synchronize()
    assert bool(done.done_u8.all()) and bool(done.truncated.all())        # the boundary window really ends every env
    return row


def paac_fps(pkg, E, bootstrap, updates=8, rounds=3):
    import torch
    import train_paac_conv as tp
    args = tp.get_arg_parser().parse_args(["-ec", str(E)])
    net_creator, env_creator = tp.get_network_and_environment_creator(args)
    paac = pkg.submodule("agents.paac.paac")
    L = paac.GridPAACLearner(net_creator, env_creator, args, use_cuda_graph=True, mask_terminals=True,
                             bootstrap_truncated=bootstrap)
    L.start()
    for _ in range(2):
        L.update()                                      # capture + one replay
    torch.cuda.synchronize()
    out = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        for _ in range(updates):
            L.update()
        torch.cuda.synchronize()
        out.append(updates * L.max_local_steps * L.total_emulators / (time.perf_counter() - t0))
    del L
    torch.cuda.empty_cache()
    return statistics.median(out)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--shapes", nargs="+", default=SHAPES)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--paac", nargs="*", type=int, default=[32, 1024], help="emulators per GPU of the PAAC figure")
    ap.add_argument("--out", default=None, help="JSON file for the table (default: print only)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("final_obs_ab.py measures the GPU: no CUDA device")
    import golds_rl_gym_b200 as pkg
    M = pkg.submodule("envs.multiagent")
    info = gpu_info()
    rows = []
    for shape in args.shapes:
        rows.append(shape_rows(M, shape, args.rounds))
        print(json.dumps(rows[-1]), flush=True)
        torch.cuda.empty_cache()
    paac_rows = []
    for E in args.paac:
        fps = {b: paac_fps(pkg, E, b) for b in (False, True)}
        paac_rows.append({"emulators": E, "fps_masked": fps[False], "fps_bootstrap_truncated": fps[True],
                          "delta_pct": 100.0 * (fps[True] / fps[False] - 1.0)})
        print(json.dumps(paac_rows[-1]), flush=True)
    result = dict(info, rounds=args.rounds, method="CUDA graph of 8 steps replayed; median over rounds, off/on "
                  "alternated in one process; steady = 64 steps inside an episode (TimeLimit 128), boundary = "
                  "TimeLimit 1 (every env ends and auto-resets on every step)", rows=rows, paac=paac_rows)
    print("| shape | launch | window | off us/step | on us/step | delta us | delta % | spread off / on |")
    print("|---|---|---|---|---|---|---|---|")
    for row in rows:
        for win in ("steady", "boundary"):
            w = row[win]
            print("| %s | %s | %s | %.2f | %.2f | %+.2f | %+.1f | %.2f / %.2f |" % (
                row["shape"], row["launch"], win, w["off_us_median"], w["on_us_median"], w["delta_us"], w["delta_pct"],
                w["off_us_spread"], w["on_us_spread"]))
    for r in paac_rows:
        print("PAAC %d emulators: %.0f frames/s masked, %.0f with bootstrap_truncated (%+.1f %%)" % (
            r["emulators"], r["fps_masked"], r["fps_bootstrap_truncated"], r["delta_pct"]))
    print("(%s, power limit %s)" % (info["gpu"], info["power_limit"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
