"""CPU: action repeat (swarm_step_repeat) -- the new prototypes match the header, every argument error is returned
before any CUDA call, the NumPy fold the GPU twin tests build their expectations with behaves as documented, and the
Python surface takes the repeat count."""
import ctypes
import os
import re
import sys
import types

import numpy as np
import pytest

from _action_repeat import fold_substeps, substep_elapsed
from _env_physics import DEFAULT_ROW

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NULL, SIZE, FLAGS = -1, -2, -4


def _c_params(header, name):
    src = open(header).read()
    m = re.search(r"\bint\s+%s\s*\(([^;]*)\)\s*;" % name, src)
    assert m, name
    return [" ".join(a.split()) for a in m.group(1).split(",")]


def test_prototypes_match_header(pkg):
    nat = pkg._native
    P = ctypes.POINTER
    kinds = {"const SwarmParams*": P(nat.SwarmParams), "const SwarmState*": P(nat.SwarmState),
             "const SwarmStepIO*": P(nat.SwarmStepIO), "const SwarmStepFinal*": P(nat.SwarmStepFinal),
             "const SwarmPhysics*": P(nat.SwarmPhysics), "const SwarmInjectedDraws*": P(nat.SwarmInjectedDraws),
             "int32_t": ctypes.c_int32, "swarm_stream_t": ctypes.c_void_p, "int32_t[8]": ctypes.c_void_p}
    for name, n in (("swarm_step_repeat", 8), ("swarm_step_plan_repeat", 6)):
        params = _c_params(nat.HEADER, name)
        assert len(params) == n, params
        want = []
        for prm in params:
            typ, arg = prm.rsplit(" ", 1)
            if "[" in arg:                                    # int32_t out[8]
                typ += arg[arg.index("["):]
            want.append(kinds[typ])
        res, args = nat.SYMBOLS[name]
        assert res is ctypes.c_int and args == want, name
        assert getattr(nat.load(), name).argtypes == want


def _params(nat, **kw):
    base = dict(n_envs=4, n_locusts=80, n_agents=10, grid_size=84, n_burn_in=10, max_episode_steps=128,
                math_mode=0, tuning=0, noise=1e-4, gravity=-1.0, wind=1.0, F=0.5, L=10.0, dt=0.05,
                box_width=3.0, box_height=3.0, seed=1, env_id_offset=0)
    base.update(kw)
    return nat.SwarmParams(**base)


def _phys(nat, table=0x10000, flags=0):
    return nat.SwarmPhysics(table, flags, 0, (ctypes.c_double * 6)(*DEFAULT_ROW), (ctypes.c_double * 6)(*DEFAULT_ROW))


def test_argument_errors_without_gpu(pkg):
    nat = pkg._native
    lib = nat.load()
    B = ctypes.byref
    p, st, io = _params(nat), nat.SwarmState(), nat.SwarmStepIO()
    out = (ctypes.c_int32 * 8)()

    def both(p_, st_, io_, fin, phys, k):
        return (lib.swarm_step_repeat(p_, st_, io_, fin, phys, k, None, None),
                lib.swarm_step_plan_repeat(p_, st_, io_, phys, k, out))

    # the repeat count: refused before anything else is looked at (state / io would be NULL here)
    for k in (0, -1, -(2 ** 31)):
        assert both(B(p), B(st), B(io), None, None, k) == (SIZE, SIZE), k
    # NULL params / state / io, at every repeat count
    for k in (1, 2, 4):
        assert both(None, B(st), B(io), None, None, k) == (NULL, NULL)
        assert both(B(p), None, B(io), None, None, k) == (NULL, NULL)
        assert both(B(p), B(st), None, None, None, k) == (NULL, NULL)
        assert both(B(p), B(st), B(io), None, None, k) == (NULL, NULL)        # the state's NULL pointers
    # sizes are validated first, like every call
    assert both(B(_params(nat, n_envs=0)), B(st), B(io), None, None, 2) == (SIZE, SIZE)
    assert both(B(_params(nat, grid_size=1)), B(st), B(io), None, None, 0) == (SIZE, SIZE)
    assert both(B(_params(nat, math_mode=2)), B(st), B(io), None, None, 2) == (FLAGS, FLAGS)
    # swarm_step_physics' checks of the physics argument (phys is nullable here: NULL is "no physics")
    for k in (1, 3):
        assert both(B(p), B(st), B(io), None, B(_phys(nat, table=0)), k) == (NULL, NULL)
        assert both(B(p), B(st), B(io), None, B(_phys(nat, table=0x10008)), k) == (FLAGS, FLAGS)
        assert both(B(p), B(st), B(io), None, B(_phys(nat, flags=2)), k) == (FLAGS, FLAGS)
        assert both(B(p), B(st), B(io), None, B(_phys(nat)), k) == (NULL, NULL)   # valid: the state is next
    # swarm_step_final's checks of the terminal outputs, before the state is looked at
    f = nat.SwarmStepFinal
    for k in (1, 2):
        for fin, want in ((f(grid=0x10000), FLAGS), (f(positions=0x10000), FLAGS),
                          (f(grid=0x10000, positions=0x20000), FLAGS),                        # no x / xa
                          (f(x=0x30000, xa=0x40000, grid=0x10004, positions=0x20000), FLAGS),  # misaligned grid
                          (f(x=0x30000, xa=0x40000, grid=0x10000, positions=0x20000), NULL),   # valid: the state
                          (f(), NULL)):
            assert lib.swarm_step_repeat(B(p), B(st), B(io), B(fin), None, k, None, None) == want, (k, want)
    # plan: NULL out
    assert lib.swarm_step_plan_repeat(B(p), B(st), B(io), None, 2, None) == NULL


def test_fold_substeps_reward_order_and_early_stop():
    f32 = np.float32
    # a sum whose FP32 value depends on the order: 1 + 2^-24 + 2^-24 is 1 in order, 1 + 2^-23 the other way round
    r = np.array([[1.0], [2.0 ** -24], [2.0 ** -24]], dtype=f32)
    reward, done, last = fold_substeps(r, np.zeros((3, 1), bool))
    assert reward.dtype == f32 and reward[0] == f32(1.0) and last[0] == 2 and not done[0]
    assert fold_substeps(r[::-1], np.zeros((3, 1), bool))[0][0] == f32(1.0) + f32(2.0 ** -23)
    # starts from the first substep's reward: -0.0 keeps its sign at K = 1 and through a sum of -0.0
    z = np.array([[-0.0]], dtype=f32)
    assert np.signbit(fold_substeps(z, np.zeros((1, 1), bool))[0][0])
    assert np.signbit(fold_substeps(np.array([[-0.0], [-0.0]], f32), np.zeros((2, 1), bool))[0][0])
    # early stop: env 0 ends at substep 1, env 1 at 0, env 2 never, env 3 at the last; later substeps do not count
    rw = np.array([[-1, -2, -3, -4], [-5, -6, -7, -8], [-9, -10, -11, -12]], dtype=f32)
    dn = np.array([[0, 1, 0, 0], [1, 1, 0, 0], [1, 1, 0, 1]], dtype=bool)
    reward, done, last = fold_substeps(rw, dn)
    assert last.tolist() == [1, 0, 2, 2]
    assert done.tolist() == [True, True, False, True]
    assert reward.tolist() == [-6.0, -2.0, -21.0, -24.0]


def test_substep_elapsed_with_timelimit_k_does_not_divide():
    # TimeLimit 128 with K = 3: 42 decisions of 3 substeps, then one of 2
    el0 = np.array([0])
    n, d = 0, 0
    while True:
        el, tr = substep_elapsed(el0, 3, 128)
        _, done, last = fold_substeps(np.full((3, 1), -1, np.float32), tr)
        d += 1
        if done[0]:
            assert last[0] == 1 and el[last[0], 0] == 128 and tr[last[0], 0]
            break
        assert last[0] == 2
        el0 = el[-1]
        n += 1
    assert (n, d) == (42, 43)
    # every substep index is the end of some staggered env: limit 7, K = 3
    el, tr = substep_elapsed(np.arange(7), 3, 7)
    _, done, last = fold_substeps(np.zeros((3, 7), np.float32) - 1, tr)
    assert done.tolist() == [False] * 4 + [True] * 3 and last[4:].tolist() == [2, 1, 0]
    assert el[:, 6].tolist() == [7, 8, 9]
    # no TimeLimit
    assert not substep_elapsed(np.array([10 ** 6]), 4, 0)[1].any()


def test_python_surface(pkg):
    ops = pkg.load_torch_ops()
    schema = str(ops.step_repeat.default._schema)
    for arg in ("int repeat", "physics", "final_positions", "reset_draws"):
        assert arg in schema, arg
    M = pkg.submodule("envs.multiagent")
    for k in (1, 2, 8):
        assert M.BatchedSwarmEnv._repeat(types.SimpleNamespace(action_repeat=k)) == k
    for k in (0, -3, 2.5, True, 2 ** 31):
        with pytest.raises(ValueError):
            M.BatchedSwarmEnv._repeat(types.SimpleNamespace(action_repeat=k))
    ec = pkg.submodule("agents.paac.environment_creator")
    assert ec.SwarmEnvironmentCreator(action_repeat=4).action_repeat == 4
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import train_paac_conv as tp
    assert tp.get_arg_parser().parse_args(["--action_repeat", "4"]).action_repeat == 4
    assert tp.get_arg_parser().parse_args([]).action_repeat == 1
