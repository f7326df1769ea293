#!/usr/bin/env python
"""Cost of per-env physics (BatchedSwarmEnv(physics=...), swarm_step_physics) against the plain step.

    python scripts/env_physics_ab.py [--shapes 4096x256 1024x64 ...] [--rounds 7] [--out FILE.json]
    python scripts/env_physics_ab.py --sass PARENT.so NEW.so        # CPU: SASS of the default kernels unchanged?
    python scripts/env_physics_ab.py --spills LIB.so                  # CPU: where the PHYS kernels spill

Microseconds per batch-step, as in DESIGN.md section 5: a CUDA graph of 8 steps, replayed.  For every shape three envs
(same seed, automatic launch shape) are timed in alternation, in one process, over several rounds (the order rotates
every round): the default step, the PHYS kernels with a fixed table ("table") and the PHYS kernels redrawing each env's
row at every reset ("resample", F / L / wind / gravity / dt / noise ranges).  Two windows:
  steady    TimeLimit 128, 8 replays = 64 steps inside an episode (elapsed set to 0 first);
  boundary  TimeLimit 1: every step ends and auto-resets every env (10 burn-in steps each; "resample" also draws rows).
The GPU's name and power limit are read in the same run and stored with the numbers.

--sass compares `cuobjdump -sass` of two builds of libswarm_b200.so: every kernel of PARENT must have the same
instructions in NEW (names matched after dropping the PHYS template argument and the SwarmPhysics parameter).
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

SHAPES = ["4096x256", "1024x256", "4096x80", "512x256", "1024x80", "1024x64"]
VARIANTS = ("default", "table", "resample")
RANGES = {"F": (0.3, 0.7), "L": (5.0, 15.0), "wind": (0.5, 1.5), "gravity": (-1.5, -0.5), "dt": (0.04, 0.06),
          "noise": (5e-5, 2e-4)}


def sass_functions(lib):
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    out = subprocess.run([os.path.join(cuda, "bin", "cuobjdump"), "-sass", lib], capture_output=True, text=True,
                         check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur is not None:
            funcs[cur].append(" ".join(line.split()))
    names = list(funcs)
    dem = subprocess.run([os.path.join(cuda, "bin", "cu++filt")], input="\n".join(names), capture_output=True,
                         text=True, check=True).stdout.split("\n")
    return {d: "\n".join(funcs[n]) for n, d in zip(names, dem)}


def sass_compare(parent, new):
    """-> (identical, differing names, missing names, count of PHYS kernels in new)."""
    old, cur = sass_functions(parent), sass_functions(new)
    strip = {}
    n_phys = 0
    for name, body in cur.items():
        m = re.match(r"(.*)<(.*), \(bool\)([01])>\((.*), SwarmPhysics\)$", name)
        if m and m.group(3) == "1":
            n_phys += 1
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
    return same, diff, missing, n_phys


# swarm_kernels.cuh lines of the pair loops (inv_r_eps .. forces_ordered): a spill site whose innermost source line
# falls in here counts as "in a pair loop"
PAIR_LOOP_MARKERS = ("__device__ __forceinline__ float inv_r_eps(", "__device__ __forceinline__ void pair_forces(")


def spill_sites(lib):
    """-> {demangled kernel: [(STL/LDL, innermost 'file:line', inlined-at chain, in_pair_loop)]} from nvdisasm's
    inline line info of the library's cubin."""
    import tempfile
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    src = open(os.path.join(ROOT, "golds-rl-gym_b200", "csrc", "swarm_kernels.cuh")).read().splitlines()
    lo = next(i for i, l in enumerate(src) if l.startswith(PAIR_LOOP_MARKERS[0])) + 1
    hi = next(i for i, l in enumerate(src) if l.startswith(PAIR_LOOP_MARKERS[1])) + 1
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([os.path.join(cuda, "bin", "cuobjdump"), "-xelf", "all", os.path.abspath(lib)], cwd=tmp,
                       check=True, capture_output=True)
        cubin = [f for f in os.listdir(tmp) if f.endswith(".cubin")][0]
        dis = subprocess.run([os.path.join(cuda, "bin", "nvdisasm"), "-gi", "-c", os.path.join(tmp, cubin)],
                             capture_output=True, text=True, check=True).stdout
    sites, cur, loc = {}, None, ""
    for line in dis.splitlines():
        m = re.match(r"\.text\.(\S+):", line.strip())
        if m:
            cur, loc = m.group(1), ""
            sites[cur] = []
            continue
        m = re.search(r'//## File "([^"]+)", line (\d+)(.*)', line)
        if m:
            loc = (os.path.basename(m.group(1)), int(m.group(2)), m.group(3).strip())
            continue
        m = re.search(r"\b(STL|LDL)(\.\S+)?\s", line)
        if m and cur and loc:
            f, ln, chain = loc
            sites[cur].append((m.group(1), "%s:%d" % (f, ln), chain, f == "swarm_kernels.cuh" and lo <= ln < hi))
    names = list(sites)
    dem = subprocess.run([os.path.join(cuda, "bin", "cu++filt")], input="\n".join(names), capture_output=True,
                         text=True, check=True).stdout.split("\n")
    return {d: sites[n] for n, d in zip(names, dem)}


def shape_rows(M, shape, rounds):
    import torch
    from fresh_noise_ab import graph_of, timed_us_per_step
    E, N = (int(v) for v in shape.split("x"))
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1234)
    acts = []
    for _ in range(8):
        a = torch.randn(E, 10, 2, device="cuda", generator=gen)
        n = a.norm(dim=-1, keepdim=True)
        acts.append(torch.where(n >= 1.0, a / n, a).contiguous())
    phys = {"default": None, "table": "table", "resample": RANGES}
    runs = {}
    for win, limit in (("steady", 128), ("boundary", 1)):
        for v in VARIANTS:
            env = M.BatchedSwarmEnv(E, n_locusts=N, seed=1234, max_episode_steps=limit, physics=phys[v])
            env.reset()
            runs[win, v] = (env, graph_of(env, acts), [])
    plans = {v: runs["steady", v][0].plan() for v in VARIANTS}
    for r in range(rounds):
        for win in ("steady", "boundary"):
            order = VARIANTS[r % 3:] + VARIANTS[:r % 3]
            for v in order:
                env, g, t = runs[win, v]
                timed_us_per_step(env, g, 2)                # back in cache / clocks after the switch
                t.append(timed_us_per_step(env, g, 8))
    row = {"shape": shape, "E": E, "N": N, "launch": plans["default"]["raster_place"],
           "smem_bytes": {v: plans[v]["smem_bytes"] for v in VARIANTS}, "ctas": {v: plans[v]["ctas"] for v in VARIANTS}}
    for win in ("steady", "boundary"):
        base = statistics.median(runs[win, "default"][2])
        row[win] = {}
        for v in VARIANTS:
            t = runs[win, v][2]
            med = statistics.median(t)
            row[win][v] = {"us_median": med, "us_spread": max(t) - min(t), "delta_us": med - base,
                           "delta_pct": 100.0 * (med / base - 1.0)}
    env = runs["boundary", "resample"][0]
    torch.cuda.synchronize()
    assert bool(env.done_u8.all())                          # the boundary window really ends every env
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--shapes", nargs="+", default=SHAPES)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None, help="JSON file for the table (default: print only)")
    ap.add_argument("--sass", nargs=2, metavar=("PARENT_LIB", "NEW_LIB"))
    ap.add_argument("--spills", metavar="LIB", help="CPU: spill sites (STL / LDL) of every PHYS kernel by source line")
    args = ap.parse_args()
    if args.spills:
        bad = 0
        for name, st in sorted(spill_sites(args.spills).items()):
            if "SwarmPhysics" not in name or not re.search(r"\(bool\)1>\(", name) or not st:
                continue
            locs = sorted(set(l for _, l, _, _ in st))
            inloop = sorted(set(l for _, l, _, p in st if p))
            bad += len(inloop)
            print("%s: %d STL / %d LDL at %s%s" % (re.sub(r"\(swarm::KP.*", "", name).replace("void <unnamed>::", ""),
                                                  sum(k == "STL" for k, _, _, _ in st), sum(k == "LDL" for k, _, _, _ in st),
                                                  ", ".join(locs), ("  IN A PAIR LOOP: " + ", ".join(inloop)) if inloop else ""))
        raise SystemExit(1 if bad else 0)
    if args.sass:
        same, diff, missing, n_phys = sass_compare(*args.sass)
        print("default kernels with identical SASS: %d; different: %d; missing: %d; PHYS kernels: %d"
              % (same, len(diff), len(missing), n_phys))
        for name in diff + missing:
            print("  ", name)
        raise SystemExit(1 if diff or missing else 0)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("env_physics_ab.py measures the GPU: no CUDA device")
    import golds_rl_gym_b200 as pkg
    from fresh_noise_ab import gpu_info
    M = pkg.submodule("envs.multiagent")
    info = gpu_info()
    rows = []
    for shape in args.shapes:
        rows.append(shape_rows(M, shape, args.rounds))
        print(json.dumps(rows[-1]), flush=True)
        torch.cuda.empty_cache()
    result = dict(info, rounds=args.rounds, ranges=RANGES,
                  method="CUDA graph of 8 steps replayed; median over rounds, default / table / resample rotated in one "
                         "process; steady = 64 steps inside an episode (TimeLimit 128), boundary = TimeLimit 1 (every env "
                         "ends and auto-resets on every step)", rows=rows)
    print("| shape | launch | window | default us/step | table us/step (delta) | resample us/step (delta) |")
    print("|---|---|---|---|---|---|")
    for row in rows:
        for win in ("steady", "boundary"):
            w = row[win]
            print("| %s | %s | %s | %.2f | %.2f (%+.2f us, %+.1f %%) | %.2f (%+.2f us, %+.1f %%) |" % (
                row["shape"], row["launch"], win, w["default"]["us_median"],
                w["table"]["us_median"], w["table"]["delta_us"], w["table"]["delta_pct"],
                w["resample"]["us_median"], w["resample"]["delta_us"], w["resample"]["delta_pct"]))
    print("(%s, power limit %s)" % (info["gpu"], info["power_limit"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
