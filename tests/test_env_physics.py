"""CPU: per-env physics (SwarmPhysics) -- the struct has the C layout (checked with gcc), every argument error of the
*_physics calls is returned before any CUDA call, the NumPy restatement of a resampled row behaves as documented, the
oracle step with explicit constants is so.step at the default constants, and the training script parses --physics."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import swarm_oracle as so

from _env_physics import DEFAULT_ROW, resampled_row, step_with

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_physics_struct_matches_c_layout(pkg, tmp_path):
    nat = pkg._native
    cls = nat.SwarmPhysics
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "swarm_b200.h"', "int main(void){",
             'printf("size %zu\\n", sizeof(SwarmPhysics));',
             'printf("resample %u\\n", (unsigned)SWARM_PHYSICS_RESAMPLE);']
    for f, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(SwarmPhysics, %s));' % (f, f))
    lines.append("return 0;}")
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(out["size"]) == ctypes.sizeof(cls) == 112
    for f, _ in cls._fields_:
        assert int(out[f]) == getattr(cls, f).offset, f
    assert int(out["resample"]) == nat.SWARM_PHYSICS_RESAMPLE
    assert nat.PHYSICS_COLUMNS == ("noise", "gravity", "wind", "F", "L", "dt")


def _params(nat, **kw):
    base = dict(n_envs=4, n_locusts=80, n_agents=10, grid_size=84, n_burn_in=10, max_episode_steps=128,
                math_mode=0, tuning=0, noise=1e-4, gravity=-1.0, wind=1.0, F=0.5, L=10.0, dt=0.05,
                box_width=3.0, box_height=3.0, seed=1, env_id_offset=0)
    base.update(kw)
    return nat.SwarmParams(**base)


def _phys(nat, table=0x10000, flags=0, reserved=0, lo=None, hi=None):
    lo = list(DEFAULT_ROW) if lo is None else lo
    hi = list(DEFAULT_ROW) if hi is None else hi
    return nat.SwarmPhysics(table, flags, reserved, (ctypes.c_double * 6)(*lo), (ctypes.c_double * 6)(*hi))


def _calls(nat, lib, phys):
    """Every *_physics entry point with this SwarmPhysics (None = NULL) and otherwise empty arguments (never
    dereferenced: the physics check comes first)."""
    p, st, io = _params(nat), nat.SwarmState(), nat.SwarmStepIO()
    ph = ctypes.byref(phys) if phys is not None else None
    out = (ctypes.c_int32 * 8)()
    return [lib.swarm_reset_physics(ctypes.byref(p), ctypes.byref(st), ph, None, None, None),
            lib.swarm_step_physics(ctypes.byref(p), ctypes.byref(st), ctypes.byref(io), None, ph, None, None),
            lib.swarm_forces_physics(ctypes.byref(p), ph, None, None, None, None, None),
            lib.swarm_step_plan_physics(ctypes.byref(p), ctypes.byref(st), ctypes.byref(io), ph, out)]


def test_physics_argument_errors_without_gpu(pkg):
    nat = pkg._native
    lib = nat.load()
    R = nat.SWARM_PHYSICS_RESAMPLE
    lo, hi = list(DEFAULT_ROW), list(DEFAULT_ROW)
    cases = [(None, -1), (_phys(nat, table=0), -1),
             (_phys(nat, table=0x10008), -4),                    # not 16-byte aligned
             (_phys(nat, flags=2), -4), (_phys(nat, flags=R | 4), -4), (_phys(nat, reserved=1), -4)]
    for c, bad in ((3, np.inf), (3, np.nan), (0, -np.inf)):      # non-finite bound
        b = list(lo)
        b[c] = bad
        cases.append((_phys(nat, flags=R, lo=b, hi=hi), -2))
        cases.append((_phys(nat, flags=R, lo=lo, hi=b), -2))
    b_lo, b_hi = list(lo), list(hi)
    b_lo[3], b_hi[3] = 0.7, 0.3                                   # lo > hi
    cases.append((_phys(nat, flags=R, lo=b_lo, hi=b_hi), -2))
    b_lo, b_hi = list(lo), list(hi)
    b_lo[1], b_hi[1] = -1e308, 1e308                              # hi - lo overflows
    cases.append((_phys(nat, flags=R, lo=b_lo, hi=b_hi), -2))
    for l_lo in (0.0, -1.0):                                      # L must stay positive
        b_lo = list(lo)
        b_lo[4] = l_lo
        cases.append((_phys(nat, flags=R, lo=b_lo, hi=hi), -2))
    for phys, want in cases:
        assert _calls(nat, lib, phys) == [want] * 4, (phys and list(phys.lo), phys and list(phys.hi), want)
    # the ranges are only checked with RESAMPLE; the table's values never are.  A valid physics argument reaches the
    # checks of the other arguments (NULL state / io / buffers)
    b_lo = list(lo)
    b_lo[4] = -1.0
    assert _calls(nat, lib, _phys(nat, lo=b_lo)) == [-1, -1, -1, -1]
    assert _calls(nat, lib, _phys(nat, flags=R)) == [-1, -1, -1, -1]
    # sizes are validated before the physics argument, like every call
    p = _params(nat, n_envs=0)
    assert lib.swarm_forces_physics(ctypes.byref(p), None, None, None, None, None, None) == -2


def test_resampled_row_restatement():
    lo = np.array([0.0, -2.0, -2.0, 0.2, 2.0, 0.01])
    hi = np.array([1e-3, 0.5, 2.0, 0.9, 20.0, 0.1])
    rows = np.stack([resampled_row(11, g, ep, lo, hi) for g in range(64) for ep in range(4)])
    assert ((rows >= lo) & (rows <= hi)).all()
    assert len(np.unique(rows[:, 3])) == len(rows)                # a different draw per (env, episode)
    # only (seed, global id, episode) matter
    assert np.array_equal(resampled_row(11, 5, 2, lo, hi), rows[5 * 4 + 2])
    assert not np.array_equal(resampled_row(12, 5, 2, lo, hi), rows[5 * 4 + 2])
    # lo == hi gives lo exactly, also for values that are not representable sums
    fixed = np.array([1e-4, -1.0, 1.0, 0.5, 10.0, 0.05]) * (1.0 + 1e-15)
    for g in range(16):
        assert np.array_equal(resampled_row(3, g, g, fixed, fixed), fixed)
    # column c takes pair c // 2: .x for even, .y for odd -- the two halves of one pair differ
    u = resampled_row(7, 1, 0, np.zeros(6), np.ones(6))
    from oracle import philox
    assert np.array_equal(u, philox.uniform_pairs(7, 1, 0, 5, 3).reshape(6))


def test_explicit_constant_step_is_oracle_step_at_defaults():
    rs = np.random.RandomState(3)
    E, N, A = 3, 80, 10
    x = rs.rand(E, N, 2)
    xa = rs.rand(E, A, 2)
    act = rs.normal(size=(E, A, 2))
    na, nx = rs.normal(size=(E, A, 2)), rs.normal(size=(E, N, 2))
    x1, xa1, x2, xa2 = x.copy(), xa.copy(), x.copy(), xa.copy()
    r1, _ = so.step(x1, xa1, act, na, nx)
    r2, _ = step_with(x2, xa2, act, na, nx, DEFAULT_ROW)
    assert np.array_equal(x1, x2) and np.array_equal(xa1, xa2) and np.array_equal(r1, r2)
    # another row really changes the step
    row = DEFAULT_ROW.copy()
    row[3] = 0.7
    x3, xa3 = x.copy(), xa.copy()
    step_with(x3, xa3, act, na, nx, row)
    assert not np.array_equal(x3, x1) and np.array_equal(xa3, xa1)


def test_physics_torch_ops_and_script_flag(pkg):
    ops = pkg.load_torch_ops()
    for name in ("reset_physics", "step_physics", "forces_physics"):
        schema = str(getattr(ops, name).default._schema)
        for arg in ("physics", "physics_flags", "physics_lo", "physics_hi"):
            assert arg in schema, (name, arg)
    assert "final_positions" in str(ops.step_physics.default._schema)
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import train_paac_conv as tp
    args = tp.get_arg_parser().parse_args(["--physics", "F=0.3:0.7,L=5:15"])
    assert args.physics == {"F": (0.3, 0.7), "L": (5.0, 15.0)}
    assert tp.get_arg_parser().parse_args([]).physics is None
    with pytest.raises(SystemExit):
        tp.get_arg_parser().parse_args(["--physics", "F=0.3"])
