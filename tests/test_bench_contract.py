"""bench.py contract checks: the reference arm (CPU port on the host cores) prints ONE JSON line with the keys a caller
reads, non-zero ranks stay silent; on the GPU, --steps sets the timed steps and --dump-outputs is reproducible."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          env=e, timeout=300)


def test_reference_arm_prints_one_json_line():
    res = run(["--impl", "reference", "--workload", "c2", "--steps", "3", "--warmup", "3"])
    assert res.returncode == 0, res.stderr
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert KEYS <= set(d), KEYS - set(d)
    assert d["impl"] == "reference" and d["metric"] == "locust_updates_per_sec" and d["unit"] == "locust-updates/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    # oracle/_ref is staged in the build container (oracle/make_ref.py) and travels to the GPU box: the arm then
    # times the unmodified reference; without it (a bare checkout) the NumPy port stands in
    from oracle import make_ref
    assert d["cpu_baseline"]["kind"] == ("reference" if make_ref.staged() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"] and d["cpu_baseline"]["cpu_model"]
    assert d["scaling"] in ("strong", "weak")
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_are_silent():
    res = run(["--impl", "reference", "--workload", "c2", "--steps", "3", "--warmup", "3", "--gpus", "2"],
              env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_dump_outputs_only_for_the_gpu_env_path(tmp_path):
    for args in (["--impl", "reference"], ["--workload", "paac3"], ["--steps", "0"]):
        res = run(args + ["--dump-outputs", str(tmp_path / "out")])
        assert res.returncode == 2 and "usage" in res.stderr, args
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_reproducible(tmp_path):
    """Exactly --steps steps are timed (not a multiple of the 8-step graph); the dump is float32/float64, at most 64 MB,
    a seeded sample of the 1024 envs, self-consistent (grid and positions rasterise the dumped state bit for bit) and
    identical on a second run with the same arguments."""
    from oracle import swarm_oracle as so
    args = ["--workload", "c2", "--steps", "13", "--warmup", "3", "--no-cpu-baseline", "--no-secondary", "--no-paac"]
    dumps = []
    for k in range(2):
        out = tmp_path / str(k)
        res = run(args + ["--dump-outputs", str(out)])
        assert res.returncode == 0, res.stderr
        assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == 13
        files = sorted(out.glob("*.npy"))
        assert sum(p.stat().st_size for p in files) <= 64 << 20
        d = {p.stem: np.load(p) for p in files}
        assert set(d) == {"env_index", "x", "xa", "reward", "done", "grid", "positions"}
        assert all(a.dtype in (np.float32, np.float64) for a in d.values())
        assert d["x"].shape == (512, 64, 2) and d["x"].dtype == np.float64 and d["grid"].shape == (512, 84, 84, 2)
        assert len(set(d["env_index"].tolist())) == 512 and d["env_index"].max() < 1024
        for e in (0, 255, 511):
            g, p = so.rasterize(d["x"][e], d["xa"][e], 84)
            assert np.array_equal(d["grid"][e], g.astype(np.float32)) and np.array_equal(d["positions"][e], p)
        dumps.append(d)
    for name, a in dumps[0].items():
        assert np.array_equal(a, dumps[1][name]), name


def test_strong_scaling_is_the_default_and_shards_like_np_split(pkg):
    """`--gpus N` runs BASELINE.json configs[3] as written: 4096 envs TOTAL split over the ranks (np.split semantics of
    fed_gym/agents/paac/runners.py:18-19), global env ids as RNG keys."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'ap.add_argument("--scaling", default="strong"' in src
    sh = pkg.submodule("sharding")
    for world in (1, 2, 4, 8):
        parts = [sh.shard_envs(4096, world, r) for r in range(world)]
        assert [p[1] for p in parts] == [4096 // world] * world
        assert [p[0] for p in parts] == [r * (4096 // world) for r in range(world)]
    with pytest.raises(ValueError):
        sh.shard_envs(4096, 3, 0)


def test_reference_staging_recipe(tmp_path):
    """oracle/make_ref.py copies exactly the two NumPy-only reference files of the path, byte for byte, and records
    their SHA-256; the staged tree is git-ignored."""
    from oracle import make_ref
    gi = open(os.path.join(ROOT, ".gitignore")).read()
    assert "oracle/_ref/" in gi
    assert make_ref.FILES == ["fed_gym/envs/multiagent.py", "fed_gym/agents/state_processors.py"]
    if not os.path.isdir("/root/reference"):
        pytest.skip("reference not mounted")
    assert make_ref.stage(quiet=True) and make_ref.staged()
    import hashlib
    man = json.load(open(os.path.join(make_ref.REF, "MANIFEST.json")))
    for rel in make_ref.FILES:
        a = open(os.path.join("/root/reference", rel), "rb").read()
        b = open(os.path.join(make_ref.REF, rel), "rb").read()
        assert a == b and man["sha256"][rel] == hashlib.sha256(a).hexdigest()
