"""CPU: the terminal outputs of swarm_step_final -- SwarmStepFinal has the C layout (checked with gcc), its argument
errors are returned before anything touches a GPU, the torch op is registered and GridPAACLearner refuses
bootstrap_truncated without mask_terminals."""
import ctypes
import os
import subprocess
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_step_final_struct_matches_c_layout(pkg, tmp_path):
    nat = pkg._native
    cls = nat.SwarmStepFinal
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "swarm_b200.h"', "int main(void){",
             'printf("size %zu\\n", sizeof(SwarmStepFinal));']
    for f, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(SwarmStepFinal, %s));' % (f, f))
    lines.append("return 0;}")
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(out["size"]) == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(out[f]) == getattr(cls, f).offset, f
    assert [f for f, _ in cls._fields_] == ["x", "xa", "terminated", "truncated", "grid", "positions"]


def _params(nat, **kw):
    base = dict(n_envs=4, n_locusts=80, n_agents=10, grid_size=84, n_burn_in=10, max_episode_steps=128,
                math_mode=0, tuning=0, noise=1e-4, gravity=-1.0, wind=1.0, F=0.5, L=10.0, dt=0.05,
                box_width=3.0, box_height=3.0, seed=1, env_id_offset=0)
    base.update(kw)
    return nat.SwarmParams(**base)


def test_step_final_argument_errors_without_gpu(pkg):
    """Inconsistent terminal buffers are SWARM_ERR_FLAGS and missing required ones SWARM_ERR_NULL, returned before any
    CUDA call (the pointers below are never dereferenced)."""
    nat = pkg._native
    lib = nat.load()
    p = _params(nat)
    st, io = nat.SwarmState(), nat.SwarmStepIO()
    X, XA, G, P = 0x10000, 0x20000, 0x30000, 0x40000
    bad = [dict(grid=G),                                  # grid without positions
           dict(x=X, xa=XA, positions=P),                 # positions without grid
           dict(xa=XA, grid=G, positions=P),              # grid without x (the rasteriser's source)
           dict(x=X, grid=G, positions=P),                # grid without xa
           dict(x=X, xa=XA, grid=G + 4, positions=P)]     # grid not 8-byte aligned
    for kw in bad:
        fin = nat.SwarmStepFinal(**kw)
        assert lib.swarm_step_final(ctypes.byref(p), ctypes.byref(st), ctypes.byref(io), ctypes.byref(fin), None,
                                    None) == -4, kw
    # NULL: params, state, io -- with and without terminal buffers
    fin = nat.SwarmStepFinal(x=X, xa=XA, terminated=P, truncated=P + 8, grid=G, positions=P)
    assert lib.swarm_step_final(None, ctypes.byref(st), ctypes.byref(io), ctypes.byref(fin), None, None) == -1
    assert lib.swarm_step_final(ctypes.byref(p), None, None, ctypes.byref(fin), None, None) == -1
    assert lib.swarm_step_final(ctypes.byref(p), ctypes.byref(st), None, None, None, None) == -1
    assert lib.swarm_step_final(ctypes.byref(p), ctypes.byref(st), ctypes.byref(io), ctypes.byref(fin), None, None) == -1
    # sizes are validated first, like swarm_step
    assert lib.swarm_step_final(ctypes.byref(_params(nat, n_envs=0)), ctypes.byref(st), ctypes.byref(io),
                                ctypes.byref(nat.SwarmStepFinal()), None, None) == -2


def test_step_final_torch_op_registered(pkg):
    ops = pkg.load_torch_ops()
    assert hasattr(ops, "step_final")
    schema = str(ops.step_final.default._schema)
    for name in ("final_x", "final_xa", "terminated", "truncated", "final_grid", "final_positions"):
        assert name in schema, name


def test_bootstrap_truncated_needs_mask_terminals(pkg):
    paac = pkg.submodule("agents.paac.paac")
    args = types.SimpleNamespace(max_local_steps=5, num_actions=2, initial_lr=1e-3, lr_annealing_steps=1,
                                 max_global_steps=1, gamma=0.99, clip_norm=3.0, clip_norm_type="global",
                                 emulator_counts=4)
    with pytest.raises(ValueError, match="mask_terminals"):
        paac.GridPAACLearner(None, None, args, mask_terminals=False, bootstrap_truncated=True)
