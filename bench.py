#!/usr/bin/env python
"""Benchmark of the swarm hot path (BASELINE.json metric: swarm env-steps/s & locust-updates/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c2|n80|paac3|paac5] [--scaling strong|weak]
                    [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one batch-step: every env of the rank's shard advances once through the fused kernel
(SwarmEnv._step + TimeLimit + SwarmRunner auto-reset + 84x84 compact rasterise).

Scaling (BASELINE.json configs[3]: "4096 envs x 256 locusts ... sharded across 1/2/4/8 B200"): the default is STRONG
scaling -- the named batch is split over the ranks like the reference splits its emulators over workers
(fed_gym/agents/paac/runners.py:18-19,65-66), global env ids keep the Philox streams shard-invariant and there is no
data-path collective.  `--scaling weak` gives every GPU the whole named batch; at N > 1 the default line carries that
figure too (secondary.weak).  Rank 0 prints ONE JSON line.

The timed region is exactly --steps batch-steps and starts 8 steps into a fresh episode, so it holds (K + 8) // 128
lock-step auto-reset boundaries (every env runs the reset's 10 burn-in steps inside one batch-step).

--dump-outputs DIR writes what the last timed step returned to its caller (see dump_outputs).  Inputs are seeded, so two
builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[3]: the configuration the metric's target is quoted on
    "c4": dict(E=4096, N=256, name="C4 large-swarm stress: 4096 envs x 256 locusts, all-pairs forces"),
    # BASELINE.json configs[1]
    "c2": dict(E=1024, N=64, name="C2 batched swarm env: 1024 envs x 64 locusts"),
    # the reference's default swarm size (fed_gym/envs/multiagent.py:8-9) at the C2 batch size
    "n80": dict(E=1024, N=80, name="1024 envs x 80 locusts (reference default N_LOCUSTS; every PAAC config's swarm)"),
}
PAAC = {
    # BASELINE.json configs[2] / configs[4]
    "paac3": dict(E=32, name="C3 PAAC conv training as in scripts/train_paac_conv.py (--height=84 --clip_norm=1), 32 emulators"),
    "paac5": dict(E=8192, name="C5 PAAC conv training, 8192 emulators sharded over the GPUs, NCCL gradient all-reduce"),
}
A, G = 10, 84
FLOPS_PER_PAIR = 18            # SURVEY.md 8(d)
MUFU_PER_CLK_SM = 15.93        # measured, scripts/microbench.cu (profiles/r01_microbench.jsonl)
MIN_STEPS = 256                # end-to-end (host-buffer) figure
DUMP_ENVS = 512                # --dump-outputs: at most this many envs (a seeded sample), about 31 MB at 84x84 and N = 256


def ncu_traffic(workload):
    """dram read+write bytes per batch-step of the step kernel(s), from the newest committed ncu --set full summary
    (profiles/rNN_summary.json: {"traffic_bytes_per_step": {workload: bytes}})."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    try:
        for name in sorted(os.listdir(pdir)):
            if name.endswith("_summary.json"):
                with open(os.path.join(pdir, name)) as f:
                    summ = json.load(f)
                t = summ.get("traffic_bytes_per_step", {}).get(workload)
                if t:
                    best = float(t)
                elif workload == "c4" and "k_step" in summ:       # round-1 layout
                    tot = 0.0
                    for k in ("k_step", "k_raster_follow"):
                        d = summ.get(k, {})
                        if "dram__bytes_read.sum" in d:
                            tot += (float(d["dram__bytes_read.sum"]) + float(d["dram__bytes_write.sum"])) * 1e6
                    best = tot or best
    except Exception:
        pass
    return best


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm_gbs=float(p["hbm_gbs"]), sm_max_mhz=float(p["sm_max_mhz"]), source="measured")
    except Exception:
        return dict(hbm_gbs=6650.0, sm_max_mhz=1965.0, source="fallback")


class ClockSampler(object):
    """nvidia-smi polled every 20 ms from BEFORE the warm-up (it needs ~0.2 s to start); only the samples whose
    timestamps fall inside the timed region count."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self, t_begin, t_end):
        import datetime
        if self.proc is None:
            return None
        time.sleep(0.06)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            return None
        rows, mx = [], 0.0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [s.strip() for s in line.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), [n for n, v in zip(names, f[4:8]) if v.lower().startswith("active")]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
        if not rows:
            return None
        inside = [r for r in rows if t_begin - 0.02 <= r[0] <= t_end + 0.02]
        where = "timed region"
        if not inside:                      # a short timed region can fall between two 20 ms samples
            inside = sorted(rows, key=lambda r: r[1])[len(rows) // 2:]
            where = "whole run (no sample inside the timed region)"
        reasons = sorted({n for r in inside for n in r[2]})
        return dict(sm_mhz=statistics.median([r[1] for r in inside]), sm_max_mhz=mx, reasons=reasons,
                    samples=len(inside), sampled="nvidia-smi -lms 20, " + where)


def cpu_baseline_block(N, seconds, name):
    """The reference itself (oracle/_ref, staged by oracle/make_ref.py) on every host core, the faster NumPy port
    beside it.  Bounded samples: about `seconds` of wall time for the reference, a third of that for the port."""
    from oracle import cpu_baseline as cb
    model = cb.cpu_model()
    port = None
    probe = cb.time_port(N, steps=4, warmup=1, envs_per_proc=2)
    steps_p = int(max(8, min(20000, (seconds / 3.0) * probe["steps"] / max(probe["seconds"], 1e-6))))
    res = cb.time_port(N, steps=steps_p, warmup=1, envs_per_proc=2)
    port = {"value": res["env_steps_per_s"] * N, "unit": "locust-updates/s", "cores": res["procs"], "kind": "port",
            "env_steps_per_sec": res["env_steps_per_s"],
            "sample": "%d envs (2 per core) x %d steps, vectorised NumPy FP64 restatement (oracle/swarm_oracle.py) of "
                      "SwarmEnv.step + process_state; %.1f s" % (res["envs"], res["steps"], res["seconds"])}
    if not cb.reference_staged():
        port["cpu_model"] = model
        port["note"] = "oracle/_ref is not staged on this box: the port stands in for the reference"
        return port
    probe = cb.time_reference(N, steps=2, warmup=1, envs_per_proc=1)
    steps_r = int(max(4, min(5000, seconds * probe["steps"] / max(probe["seconds"], 1e-6))))
    res = cb.time_reference(N, steps=steps_r, warmup=1, envs_per_proc=1)
    return {"value": res["env_steps_per_s"] * N, "unit": "locust-updates/s", "cores": res["procs"], "kind": "reference",
            "cpu_model": model, "env_steps_per_sec": res["env_steps_per_s"],
            "sample": "%s: %d envs (1 per core) x %d steps of the UNMODIFIED reference (fed_gym SwarmEnv.step + "
                      "SwarmStateProcessor.process_state(84), staged under oracle/_ref), one process per core, "
                      "OMP_NUM_THREADS=1, clipped N(0,1) actions, reset excluded; %.1f s"
                      % (name, res["envs"], res["steps"], res["seconds"]),
            "port": port}


def run_reference(args, wl):
    """--impl reference: the reference's own CPU implementation of the path on all host cores, on the same workload
    shape; each step is a bounded sample (1 env per core)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_baseline as cb
    N = wl["N"]
    # One "step" of this arm = one pass of every host core over its own envs.  How many envs a core owns is sized from a
    # one-env calibration so that the K timed steps take about 20 s in total (1..64 envs per core): a 0.2 s sample -- what
    # 20 steps of one env per core would be -- measured anywhere between 2.7e5 and 4.9e5 on the same box.
    steps, warm = max(1, args.steps), max(1, min(args.warmup, 3))
    if cb.reference_staged():
        t_env = cb.time_reference(N, steps=2, warmup=1, envs_per_proc=1, procs=1)["seconds"] / 2.0
        per = int(max(1, min(64, round(20.0 / (steps * max(t_env, 1e-6))))))
        res = cb.time_reference(N, steps=steps, warmup=warm, envs_per_proc=per)
        kind, what = "reference", "the UNMODIFIED reference (oracle/_ref: fed_gym SwarmEnv.step + SwarmStateProcessor.process_state)"
    else:
        t_env = cb.time_port(N, steps=2, warmup=1, envs_per_proc=1, procs=1)["seconds"] / 2.0
        per = int(max(2, min(64, round(20.0 / (steps * max(t_env, 1e-6))))))
        res = cb.time_port(N, steps=steps, warmup=warm, envs_per_proc=per)
        kind, what = "port", "NumPy FP64 port (oracle/_ref not staged on this box)"
    value = res["env_steps_per_s"] * N
    unit = "locust-updates/s"
    sample = "%d envs (%d per core) x %d steps of %s, %s, reset excluded" % (
        res["envs"], res["envs"] // max(1, res["procs"]), res["steps"], wl["name"], what)
    print(json.dumps({
        "impl": "reference", "metric": "locust_updates_per_sec", "value": value, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * res["seconds"] / max(1, res["steps"]), "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"] + " (bounded sample)", "envs_timed": res["envs"], "n_locusts": N,
                   "n_agents": A, "grid": G},
        "env_steps_per_sec": res["env_steps_per_s"],
        "cpu_baseline": {"value": value, "unit": unit, "cores": res["procs"], "kind": kind, "sample": sample,
                         "cpu_model": cb.cpu_model()},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def paac_frames_per_sec(E_total, updates, warmup_updates, world, rank, local, seconds_cap=None, net_precision="fp32"):
    """PAAC frames/s (= T*E / loop time, paac.py:397-401) of the device-resident learner, CUDA-event timed.
    E_total emulators are sharded over the ranks.  seconds_cap bounds the timed region (updates are reduced, never
    below 50, and the figure says how many ran)."""
    import torch
    import golds_rl_gym_b200 as pkg
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import train_paac_conv as tp
    args = tp.get_arg_parser().parse_args(["--height=84", "--clip_norm=1", "-ec", str(E_total)])
    net_creator, env_creator = tp.get_network_and_environment_creator(args)
    learner = pkg.submodule("agents.paac.paac").GridPAACLearner(net_creator, env_creator, args, net_precision=net_precision)
    learner.start()
    sh = pkg.submodule("sharding")
    dev = torch.device("cuda", local)
    for _ in range(warmup_updates):
        learner.update()
    torch.cuda.synchronize()
    if seconds_cap:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            learner.update()
        e1.record()
        torch.cuda.synchronize()
        per = sh.max_over_ranks(e0.elapsed_time(e1) / 4.0, device=dev) * 1e-3
        updates = int(max(50, min(updates, seconds_cap / max(per, 1e-6))))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(updates):
        learner.update()
    e1.record()
    torch.cuda.synchronize()
    ms = sh.max_over_ranks(e0.elapsed_time(e1), device=dev)
    frames = updates * learner.max_local_steps * learner.total_emulators
    net_dtype = {"fp32": "fp32 (cuDNN / cuBLAS TF32 disabled: torch.backends.cudnn.allow_tf32 = cuda.matmul.allow_tf32 = False)",
                 "tf32": "tf32 (EXTRA, not the reference's precision: TF32 tensor cores for convolutions and matmuls)",
                 "bf16": "bf16 autocast (EXTRA, not the reference's precision)"}[net_precision]
    res = dict(frames_per_sec=frames / (ms * 1e-3), ms_per_update=ms / updates, updates=updates,
                emulators=learner.total_emulators, emulators_per_gpu=learner.emulator_counts,
                local_steps=learner.max_local_steps, policy_batch=learner.real_batch_size,
                observation="compact (grid + positions; conv1 factorised over the shared channels)" if learner.compact_obs
                else "expanded (E,A,84,84,3)", net_dtype=net_dtype,
                launch="one CUDA graph per update (rollout + returns + backward + all-reduce + Adam)")
    del learner
    torch.cuda.empty_cache()
    return res


def run_paac(args, wl, key):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    updates = max(args.steps, 500) if key == "paac3" else max(args.steps, 50)
    res = paac_frames_per_sec(wl["E"], updates, max(args.warmup, 3), world, rank, local,
                              seconds_cap=None if key == "paac3" else 60.0)
    if rank == 0:
        print(json.dumps({
            "metric": "paac_frames_per_sec", "value": res["frames_per_sec"], "unit": "frames/s", "n_gpus": world,
            "steps": res["updates"], "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_update"],
            "higher_is_better": True, "scaling": "strong" if key == "paac5" else "weak", "vs_baseline": None,
            "dtype": res["net_dtype"], "data": "synthetic",
            "config": {"workload": wl["name"], "emulators": wl["E"], "emulators_per_gpu": res["emulators_per_gpu"],
                       "n_locusts": 80, "n_agents": A, "grid": G, "local_steps": res["local_steps"],
                       "parallelism": "env-sharded x%d, flat-gradient NCCL all-reduce" % world},
            "paac": res, "gpu_launches": res["updates"] * res["local_steps"]}))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, env):
    """Writes what the last step returned to its caller -- the state (x, xa), reward, done and the observation (grid,
    positions) -- as out_dir/<name>.npy, the state in float64 and the rest in float32.  Batches of more than DUMP_ENVS
    envs keep a fixed seeded sample of DUMP_ENVS of them; env_index.npy lists which (local env ids)."""
    import numpy as np
    import torch
    E = env.E
    idx = np.arange(E) if E <= DUMP_ENVS else np.sort(np.random.RandomState(0).choice(E, DUMP_ENVS, replace=False))
    sel = torch.as_tensor(idx, device=env.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    for name, t in (("x", env.x), ("xa", env.xa), ("reward", env.reward), ("done", env.done_u8), ("grid", env.grid),
                    ("positions", env.positions)):
        a = t.index_select(0, sel).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def measure_env(M, torch, dist, dev, world, rank, E, N, first_id, K, W, math_mode, use_graph, sampler=None,
                want_extras=True, dump_dir=None):
    """Times K device-resident batch-steps of E envs x N locusts on this rank.  Returns a dict of measurements;
    every time is the MAX over ranks.  dump_dir: where to write the last timed step's outputs (dump_outputs)."""
    env = M.BatchedSwarmEnv(E, n_locusts=N, n_agents=A, grid_size=G, max_episode_steps=128, seed=1234,
                            env_id_offset=first_id, device=dev, math_mode=math_mode, auto_reset=True, rasterize=True)
    env.reset()
    plan = env.plan()
    # inputs resident in HBM: a ring of pre-clipped N(0,1) actions (seeded per rank)
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    ring = []
    for _ in range(8):
        a = torch.randn(E, A, 2, device=dev, generator=gen)
        n = a.norm(dim=-1, keepdim=True)
        ring.append(torch.where(n >= 1.0, a / n, a).contiguous())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(v):
        if world > 1:
            t = torch.tensor([v], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return float(v)

    wall = [0.0, 0.0]

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        wall[0] = time.time()
        e0.record()
        for i in range(k):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        wall[1] = time.time()
        barrier()
        return rank_max(e0.elapsed_time(e1))

    step = lambda i: env.step(ring[i & 7])
    for i in range(W):
        step(i)
    # The device-resident rollout replays a CUDA graph of 8 consecutive steps (one per action tensor of
    # the ring): same kernels, same arguments, no per-step host work.
    graph = None
    if use_graph:
        torch.cuda.synchronize()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for i in range(8):
                step(i)
        torch.cuda.current_stream(dev).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for i in range(8):
                step(i)
    run8 = (lambda i: graph.replay()) if graph is not None else (lambda i: [step(j) for j in range(8)])
    # untimed: the first replays upload the graph.  Ending them in a synchronise (timed() does) before the reset below
    # measured 0.1 % faster timed steps than letting the reset queue behind them.
    timed(run8, 8)
    env.reset()                             # start the timed region in a fresh episode (elapsed = 8 everywhere)
    for i in range(8):
        step(i)
    # K steps in order ring[0], ring[1], ...: whole 8-step replays, then the remainder launched one by one
    t_ms = timed(lambda i: run8(i) if i < K // 8 else step(i - K // 8), K // 8 + K % 8)
    clocks = sampler.stop(wall[0], wall[1]) if sampler else None
    if dump_dir is not None:
        dump_outputs(dump_dir, env)
    out = dict(E=E, N=N, K=K, ms=t_ms, ms_per_step=t_ms / K, plan=plan, clocks=clocks, region_s=wall[1] - wall[0])
    # per-8-step latencies over one episode: the lock-step boundary (10 burn-in steps inside one step) shows as the max
    env.reset()
    lat = []
    for r in range(17):
        lat.append(timed(run8, 1) / 8.0)
    out["replay8_ms_per_step"] = dict(median=statistics.median(lat), max=max(lat),
                                      note="8-step graph replays across one 128-step episode boundary, per-step average of each")
    if want_extras:
        # force kernel alone (swarm_forces = SwarmEnv.v_calculate for the batch)
        v = torch.empty(E, N, 2, dtype=torch.float32, device=dev)
        r = torch.empty(E, dtype=torch.float32, device=dev)
        force = lambda i: env.forces(v=v, reward=r)
        for i in range(3):
            force(i)
        nf = max(20, K // 16)
        out["ms_forces"] = timed(force, nf) / nf
        rast = lambda i: env.observe()
        for i in range(3):
            rast(i)
        out["ms_raster"] = timed(rast, nf) / nf
    # end to end through the host-buffer C-ABI call: actions from pinned host memory, reward/done back
    h_act = [a.cpu().pin_memory() for a in ring]
    h_rew = torch.zeros(E, dtype=torch.float32).pin_memory()
    h_done = torch.zeros(E, dtype=torch.uint8).pin_memory()
    e2e_step = lambda i: env.step_host(h_act[i & 7], h_rew, h_done)
    for i in range(16):          # every host buffer of the ring once or more (the library caches a graph per argument set)
        e2e_step(i)
    Ke = max(MIN_STEPS, min(K, 2048))
    barrier()
    w0 = time.perf_counter()
    for i in range(Ke):
        e2e_step(i)
    torch.cuda.synchronize()
    out["e2e_ms_per_step"] = rank_max((time.perf_counter() - w0) * 1e3) / Ke
    out["e2e_steps"] = Ke
    if want_extras and world == 1:
        # ... and with the compact observation copied back to pinned host memory as well (the numpy-out facade case)
        h_grid = torch.zeros(E, G, G, 2, dtype=torch.float32).pin_memory()
        h_pos = torch.zeros(E, A, 2, dtype=torch.uint8).pin_memory()
        full = lambda i: env.step_host(h_act[i & 7], h_rew, h_done, h_grid, h_pos)
        for i in range(10):
            full(i)
        Kf = 64
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        for i in range(Kf):
            full(i)
        torch.cuda.synchronize()
        out["e2e_full_obs_ms_per_step"] = (time.perf_counter() - w0) * 1e3 / Kf
        out["e2e_full_obs_steps"] = Kf
        del h_grid, h_pos
    del env
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1024)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS) + sorted(PAAC))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): the named env batch is sharded over the GPUs; weak: every GPU gets the whole batch")
    ap.add_argument("--math", default="fast", choices=["fast", "precise"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary figures (C2, N=80, weak scaling, PAAC C5)")
    ap.add_argument("--no-paac", action="store_true", help="skip the secondary PAAC frames/s figure (config 3)")
    ap.add_argument("--no-graph", action="store_true", help="launch every step from Python instead of replaying a CUDA graph")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target wall time of the CPU-baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0's envs; --impl ours, c4/c2/n80)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS):
        ap.error("--dump-outputs needs --impl ours and one of the workloads %s" % "/".join(sorted(WORKLOADS)))
    if args.workload in PAAC:
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the reference learner needs TensorFlow 1.4 (not in this image)"}))
            return
        return run_paac(args, PAAC[args.workload], args.workload)
    wl = WORKLOADS[args.workload]
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args, wl)

    import torch
    import torch.distributed as dist
    import golds_rl_gym_b200 as pkg
    M = pkg.submodule("envs.multiagent")
    sh = pkg.submodule("sharding")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N = wl["N"]
    if args.scaling == "strong":
        first, E = sh.shard_envs(wl["E"], world, rank)       # np.split semantics: E_total % world == 0
    else:
        first, E = rank * wl["E"], wl["E"]
    E_total = E * world
    sampler = ClockSampler(local) if rank == 0 else None      # started early: nvidia-smi takes a moment to come up
    m = measure_env(M, torch, dist, dev, world, rank, E, N, first, args.steps, args.warmup, args.math, not args.no_graph,
                    sampler=sampler, want_extras=True, dump_dir=args.dump_outputs if rank == 0 else None)
    K, ms_step = m["K"], m["ms_per_step"]
    env_steps = E_total / (ms_step * 1e-3)
    pairs_per_launch = E * N * (N + A)                        # per rank: what ONE launch of the dominant kernel does
    pk = peaks()
    fp32_peak = 148 * 128 * 2 * pk["sm_max_mhz"] * 1e6 / 1e12          # TFLOP/s
    achieved = pairs_per_launch * FLOPS_PER_PAIR / (ms_step * 1e-3) / 1e12
    xu_peak = 148 * MUFU_PER_CLK_SM * pk["sm_max_mhz"] * 1e6
    # algorithmic HBM bytes of the fused launch (SURVEY 8d): state r/w + frozen noise + actions + obs
    bytes_per_env = (N + A) * 16 * 3 + A * 8 + 5 + 8 + (G * G * 2 * 4 + A * 2)
    hbm = E * bytes_per_env / (ms_step * 1e-3) / 1e9

    weak = None
    if world > 1 and args.scaling == "strong" and not args.no_secondary:
        mw = measure_env(M, torch, dist, dev, world, rank, wl["E"], N, rank * wl["E"], 256, args.warmup, args.math,
                         not args.no_graph, sampler=None, want_extras=False)
        weak = {"scaling": "weak", "envs_per_gpu": wl["E"], "ms_per_step": mw["ms_per_step"], "steps": mw["K"],
                "value": world * wl["E"] * N / (mw["ms_per_step"] * 1e-3), "unit": "locust-updates/s",
                "e2e": world * wl["E"] * N / (mw["e2e_ms_per_step"] * 1e-3)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_block(N, args.cpu_seconds, wl["name"])

    paac = None
    if world == 1 and not args.no_paac and args.workload == "c4":
        try:
            paac = paac_frames_per_sec(PAAC["paac3"]["E"], 500, 20, 1, 0, local)
            paac["config"] = PAAC["paac3"]["name"]
            extra = paac_frames_per_sec(PAAC["paac3"]["E"], 500, 20, 1, 0, local, net_precision="tf32")
            paac["extra_tf32"] = {k: extra[k] for k in ("frames_per_sec", "ms_per_update", "updates", "net_dtype")}
        except Exception as exc:      # the secondary figure must never take the headline down
            paac = {"error": repr(exc)}
    paac5 = None
    if world > 1 and not args.no_paac and not args.no_secondary and args.workload == "c4":
        try:
            paac5 = paac_frames_per_sec(PAAC["paac5"]["E"], 500, 5, world, rank, local, seconds_cap=70.0)   # 500 updates fit at 8 GPUs
            paac5["config"] = PAAC["paac5"]["name"]
            extra = paac_frames_per_sec(PAAC["paac5"]["E"], 200, 5, world, rank, local, seconds_cap=15.0, net_precision="tf32")
            paac5["extra_tf32"] = {k: extra[k] for k in ("frames_per_sec", "ms_per_update", "updates", "net_dtype")}
        except Exception as exc:
            paac5 = {"error": repr(exc)}

    # BASELINE.json configs[1] (C2) and the reference's default swarm size next to the headline workload: measured by
    # child processes of this very script, each with its own roofline and CPU baseline
    secondary = None
    if world == 1 and rank == 0 and args.workload == "c4" and not args.no_secondary:
        secondary = {}
        for key in ("c2", "n80"):
            try:
                res = subprocess.run([sys.executable, os.path.abspath(__file__), "--workload", key, "--steps", "512", "--warmup",
                                      str(args.warmup), "--no-paac", "--no-secondary", "--cpu-seconds", "4"],
                                     capture_output=True, text=True, timeout=400)
                d = json.loads(res.stdout.strip().splitlines()[-1])
                secondary[key] = {k: d[k] for k in ("value", "unit", "ms_per_step", "steps", "env_steps_per_sec", "e2e", "config",
                                                    "roofline", "roofline_hbm", "cpu_baseline", "launch_shape") if k in d}
            except Exception as exc:
                secondary[key] = {"error": repr(exc)}
    # BASELINE.json configs[0] (C1): the single-env gym facade (numpy in / numpy out, one host round trip per step) next to
    # the reference's own single-process rate on this box's CPU
    if world == 1 and rank == 0 and args.workload == "c4" and not args.no_secondary:
        try:
            import numpy as np
            fenv = M.make("Swarm-eval-v0")
            fenv.reset()
            rs = np.random.RandomState(0)
            acts = rs.normal(size=(400, 10, 2)) * 0.5
            for t in range(50):
                fenv.step(acts[t])
            t0 = time.perf_counter()
            for t in range(50, 350):
                _, _, dn, _ = fenv.step(acts[t])
                if dn:
                    fenv.reset()
            c1 = {"facade_steps_per_sec": 300.0 / (time.perf_counter() - t0),
                  "config": "C1: SwarmEnv (N=80, seed 192, TimeLimit 128) through the numpy-in / numpy-out gym facade, 300 steps incl. "
                            "two resets; one kernel launch + host round trip per step"}
            if not args.no_cpu_baseline:
                from oracle import cpu_baseline as cb
                if cb.reference_staged():
                    r1 = cb.time_reference(80, steps=200, warmup=2, envs_per_proc=1, procs=1)
                    c1["reference_steps_per_sec_one_process"] = r1["env_steps_per_s"]
            secondary = dict(secondary or {}, c1=c1)
        except Exception as exc:
            secondary = dict(secondary or {}, c1={"error": repr(exc)})
    if weak is not None:
        secondary = dict(secondary or {}, weak=weak)
    if paac5 is not None:
        secondary = dict(secondary or {}, paac5=paac5)

    if rank == 0:
        # MUFU per UNORDERED pair: rsq + 2 ex2 + rcp; the unordered-pair modes (force_mode 1 and 3: N <= 512) take 1/(r+eps) from
        # the rsq by a one-term series instead of the rcp (fast math): 3
        mufu_pair = 3.0 if (m["plan"]["force_mode"] in (1, 3) and args.math == "fast") else 4.0
        xu_ach = 0.5 * mufu_pair * pairs_per_launch / (ms_step * 1e-3)
        e2e_val = E_total * N / (m["e2e_ms_per_step"] * 1e-3)
        out = {
            "metric": "locust_updates_per_sec", "value": env_steps * N, "unit": "locust-updates/s",
            "n_gpus": world, "steps": K, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32 pair forces / f64 integrator state", "data": "synthetic",
            "config": {"workload": wl["name"] + "; fused step + TimeLimit(128) + auto-reset + 84x84 compact rasterise",
                       "envs_total": E_total, "envs_per_gpu": E, "n_locusts": N, "n_agents": A, "grid": G, "math": args.math,
                       "actions": "N(0,1) clipped to unit norm, 8 pre-generated device tensors",
                       "launch": "python per step" if args.no_graph else "CUDA graph of 8 steps replayed",
                       "timed_region": "%d steps from step 8 of an episode, %d lock-step auto-reset boundaries included, %.2f s"
                                       % (K, (K + 8) // 128, m["region_s"]),
                       "l2": ("no explicit flush: each step streams %.0f MB of observations per GPU, more than the 126 MB L2"
                              if E * G * G * 8 > 126e6 else
                              "no explicit flush: each step streams %.0f MB of observations per GPU (smaller than the 126 MB "
                              "L2, which may absorb part of the write-back)") % (E * G * G * 2 * 4 / 1e6),
                       "parallelism": "env-sharded x%d (%s scaling), no collective" % (world, args.scaling)},
            "launch_shape": m["plan"],
            "env_steps_per_sec": env_steps, "pairs_per_sec": env_steps * N * (N + A),
            "roofline": {"bound": "fp32", "kernel": "k_step (fused step" + (" + k_raster_follow" if m["plan"]["launches"] == 2 else " + rasterise") + ")",
                         "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak,
                         # the same with (a) only the steady-state steps (median 8-step replay: no episode boundary inside) and
                         # (b) the pair work of the auto-resets counted too: every 128th step also runs the reset's 10
                         # burn-in steps (multiagent.py:59-61) for every env, 138 force evaluations per 128 counted steps
                         "frac_steady_state": pairs_per_launch * FLOPS_PER_PAIR / (m["replay8_ms_per_step"]["median"] * 1e-3) / 1e12 / fp32_peak,
                         "frac_counting_reset_burn_in": achieved / fp32_peak * (128.0 + 10.0) / 128.0,
                         "traffic": ncu_traffic(args.workload) if world == 1 else None,
                         "xu_pipe": {"achieved_mufu_per_s": xu_ach, "peak_mufu_per_s": xu_peak, "frac": xu_ach / xu_peak,
                                     "mufu_per_unordered_pair": mufu_pair,
                                     "note": "the busiest pipe: %.0f MUFU per UNORDERED pair = %.1f per ordered pair; "
                                             "%.2f MUFU/clk/SM measured (scripts/microbench.cu)" % (mufu_pair, mufu_pair / 2, MUFU_PER_CLK_SM)},
                         "note": "compute-bound kernel (190 flop/B at N=256): algorithmic 18 flop/pair x %d ordered pairs per launch "
                                 "(this rank's shard) over the mean launch duration of the timed region; peak = 148 SM x 128 lanes x 2 "
                                 "x %.0f MHz (%s clock); traffic = ncu dram read+write bytes per launch (profiles/)"
                                 % (pairs_per_launch, pk["sm_max_mhz"], pk["source"])},
            "roofline_hbm": {"bound": "hbm", "achieved": hbm, "peak": pk["hbm_gbs"], "unit": "GB/s",
                             "frac": hbm / pk["hbm_gbs"], "bytes_per_launch": E * bytes_per_env, "peak_source": pk["source"]},
            "force_kernel": {"ms": m["ms_forces"], "pairs_per_sec": pairs_per_launch / (m["ms_forces"] * 1e-3),
                             "tflops_algorithmic": pairs_per_launch * FLOPS_PER_PAIR / (m["ms_forces"] * 1e-3) / 1e12,
                             "frac_fp32_peak": pairs_per_launch * FLOPS_PER_PAIR / (m["ms_forces"] * 1e-3) / 1e12 / fp32_peak,
                             "frac_xu_ceiling": 0.5 * mufu_pair * pairs_per_launch / (m["ms_forces"] * 1e-3) / xu_peak},
            "raster_kernel": {"ms": m["ms_raster"], "gbs": E * (G * G * 2 * 4 + A * 2 + (N + A) * 16) / (m["ms_raster"] * 1e-3) / 1e9,
                              "frac_hbm_peak": E * (G * G * 2 * 4 + A * 2 + (N + A) * 16) / (m["ms_raster"] * 1e-3) / 1e9 / pk["hbm_gbs"]},
            "step_latency": m["replay8_ms_per_step"],
            "e2e": {"value": e2e_val, "unit": "locust-updates/s", "h2d_bytes_per_step": E_total * A * 2 * 4,
                    "d2h_bytes_per_step": E_total * 5, "ms_per_step": m["e2e_ms_per_step"], "steps": m["e2e_steps"],
                    "note": "swarm_step_host with pinned HOST buffers, one call + stream sync per step, wall clock: the kernel "
                            "reads the step's actions from host memory over PCIe (cp.async prefetch, zero-copy) and posts "
                            "reward+done into host memory; observations stay in HBM for the device-resident policy"},
            "gpu_launches": K * m["plan"]["launches"] * world,
            "clocks": m["clocks"],
        }
        if "e2e_full_obs_ms_per_step" in m:
            out["e2e_full_obs"] = {"value": E_total * N / (m["e2e_full_obs_ms_per_step"] * 1e-3), "unit": "locust-updates/s",
                                   "ms_per_step": m["e2e_full_obs_ms_per_step"], "steps": m["e2e_full_obs_steps"],
                                   "h2d_bytes_per_step": E * A * 2 * 4, "d2h_bytes_per_step": E * 5 + E * (G * G * 2 * 4 + A * 2),
                                   "note": "as e2e, plus the compact observation (grid + positions) copied back to pinned host memory "
                                           "every step: the numpy-out case of process_state; PCIe-bound"}
        if cpu:
            out["cpu_baseline"] = cpu
        if paac is not None:
            out["paac"] = paac
        if secondary is not None:
            out["secondary"] = secondary
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
