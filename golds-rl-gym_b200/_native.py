"""ctypes binding of libswarm_b200.so (the C ABI in include/swarm_b200.h).

This is the binding a reference maintainer would add (INTEGRATION.md): plain pointers and
sizes go across, torch only provides device memory and the current stream.  There is NO CPU
fallback: if the library is missing and cannot be built, importing the env classes raises.
"""
import ctypes
import hashlib
import os
import shutil
import subprocess

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_PKG_DIR, "csrc")
_REPO = os.path.dirname(_PKG_DIR)
LIB_PATH = os.path.join(_PKG_DIR, "libswarm_b200.so")
# experiments only (scripts/build_variants.py): load another build of the same ABI through the ctypes binding
_LIB_OVERRIDE = os.environ.get("SWARM_B200_LIB")
SOURCES = [os.path.join(_CSRC, f) for f in ("swarm_b200.cu", "swarm_kernels.cuh", "swarm_cluster.cuh", "swarm_philox.cuh")]
HEADER = os.path.join(_REPO, "include", "swarm_b200.h")

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared"]

c_void_p, c_int, c_int32, c_int64, c_uint32, c_uint64, c_double, c_float = (
    ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_uint64,
    ctypes.c_double, ctypes.c_float)

ABI_VERSION = 3
SWARM_STEP_AUTO_RESET = 1
SWARM_STEP_CLIP_ACTIONS = 2
SWARM_STEP_ACTIONS_F64 = 4
SWARM_STEP_NO_ACTION_WIND = 8
SWARM_STEP_INKERNEL_RASTER = 16
SWARM_STEP_FRESH_NOISE = 32
SWARM_PHYSICS_RESAMPLE = 1
# the columns of a SwarmPhysics table row (SwarmParams' order)
PHYSICS_COLUMNS = ("noise", "gravity", "wind", "F", "L", "dt")
# SwarmParams.tuning: bits 4-5 = rasteriser placement (0 automatic); bits 8-12 = the cluster layout (0 one CTA per env,
# 1..16 a thread-block cluster of K CTAs per env, 31 the library picks K; 512 < N <= 8192); every other bit must be 0
TUNE_RASTER_FOLLOW, TUNE_RASTER_WARPS, TUNE_RASTER_SELF = 1 << 4, 2 << 4, 3 << 4
TUNE_CLUSTER_SHIFT = 8
TUNE_CLUSTER_MASK = 31 << TUNE_CLUSTER_SHIFT
TUNE_CLUSTER_AUTO = 31 << TUNE_CLUSTER_SHIFT
CLUSTER_MAX_K = 16
CLUSTER_MIN_LOCUSTS, CLUSTER_MAX_LOCUSTS = 513, 8192
MAX_LOCUSTS_ONE_CTA = 2048


def tune_cluster(k):
    """The tuning bits of the cluster layout: k CTAs per env, or None for the library's choice."""
    return TUNE_CLUSTER_AUTO if k is None else (int(k) & 31) << TUNE_CLUSTER_SHIFT


class SwarmParams(ctypes.Structure):
    _fields_ = [("n_envs", c_int32), ("n_locusts", c_int32), ("n_agents", c_int32), ("grid_size", c_int32),
                ("n_burn_in", c_int32), ("max_episode_steps", c_int32), ("math_mode", c_int32),
                ("tuning", c_int32),
                ("noise", c_double), ("gravity", c_double), ("wind", c_double), ("F", c_double),
                ("L", c_double), ("dt", c_double), ("box_width", c_double), ("box_height", c_double),
                ("seed", c_uint64), ("env_id_offset", c_int64)]


class SwarmState(ctypes.Structure):
    _fields_ = [("x", c_void_p), ("xa", c_void_p), ("noise_x", c_void_p), ("noise_a", c_void_p),
                ("elapsed", c_void_p), ("episode", c_void_p), ("work", c_void_p), ("work_words", c_uint64)]


class SwarmInjectedDraws(ctypes.Structure):
    _fields_ = [("x0", c_void_p), ("xa0", c_void_p), ("burn_actions", c_void_p),
                ("agent_noise", c_void_p), ("particle_noise", c_void_p)]


class SwarmStepIO(ctypes.Structure):
    _fields_ = [("actions_f32", c_void_p), ("actions_f64", c_void_p), ("noise_a", c_void_p),
                ("noise_x", c_void_p), ("reward", c_void_p), ("done", c_void_p), ("grid", c_void_p),
                ("positions", c_void_p), ("v_out", c_void_p), ("flags", c_uint32), ("reserved", c_uint32)]


class SwarmStepFinal(ctypes.Structure):
    _fields_ = [("x", c_void_p), ("xa", c_void_p), ("terminated", c_void_p), ("truncated", c_void_p),
                ("grid", c_void_p), ("positions", c_void_p)]


class SwarmPhysics(ctypes.Structure):
    _fields_ = [("table", c_void_p), ("flags", c_uint32), ("reserved", c_uint32), ("lo", c_double * 6),
                ("hi", c_double * 6)]


# name -> (restype, argtypes); every symbol include/swarm_b200.h declares
_P = ctypes.POINTER
SYMBOLS = {
    "swarm_abi_version": (c_int, []),
    "swarm_strerror": (ctypes.c_char_p, [c_int]),
    "swarm_last_cuda_error": (ctypes.c_char_p, []),
    "swarm_validate": (c_int, [_P(SwarmParams)]),
    "swarm_reset": (c_int, [_P(SwarmParams), _P(SwarmState), c_void_p, _P(SwarmInjectedDraws), c_void_p]),
    "swarm_step": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmStepIO), _P(SwarmInjectedDraws), c_void_p]),
    "swarm_step_final": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmStepIO), _P(SwarmStepFinal),
                                 _P(SwarmInjectedDraws), c_void_p]),
    "swarm_step_plan": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmStepIO), c_void_p]),
    "swarm_reset_physics": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmPhysics), c_void_p, _P(SwarmInjectedDraws),
                                    c_void_p]),
    "swarm_step_physics": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmStepIO), _P(SwarmStepFinal),
                                   _P(SwarmPhysics), _P(SwarmInjectedDraws), c_void_p]),
    "swarm_forces_physics": (c_int, [_P(SwarmParams), _P(SwarmPhysics), c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p]),
    "swarm_step_plan_physics": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmStepIO), _P(SwarmPhysics), c_void_p]),
    "swarm_step_repeat": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmStepIO), _P(SwarmStepFinal), _P(SwarmPhysics),
                                  c_int32, _P(SwarmInjectedDraws), c_void_p]),
    "swarm_step_plan_repeat": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmStepIO), _P(SwarmPhysics), c_int32,
                                       c_void_p]),
    "swarm_step_host": (c_int, [_P(SwarmParams), _P(SwarmState), _P(SwarmStepIO), c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p]),
    "swarm_step_host_clear": (None, []),
    "swarm_debug_trace": (None, [c_void_p, c_int64]),
    "swarm_rasterize": (c_int, [_P(SwarmParams), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "swarm_expand_obs": (c_int, [_P(SwarmParams), c_void_p, c_void_p, c_void_p, c_void_p]),
    "swarm_forces": (c_int, [_P(SwarmParams), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "swarm_x_update": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_double, c_void_p]),
    "swarm_xv_cutoff": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "swarm_s_potential": (c_int, [c_void_p, c_void_p, c_int64, c_double, c_double, c_void_p]),
    "swarm_clip_actions": (c_int, [c_void_p, c_int64, c_float, c_void_p]),
    "swarm_philox_draws": (c_int, [_P(SwarmParams), _P(SwarmState), c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "swarm_philox_noise_rows": (c_int, [_P(SwarmParams), _P(SwarmState), c_int32, c_int32, c_void_p, c_void_p,
                                        c_void_p]),
    "swarm_philox_raw": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
}

TORCH_LIB_PATH = os.path.join(_PKG_DIR, "libswarm_b200_torch.so")
TORCH_SOURCE = os.path.join(_CSRC, "torch_binding.cpp")

_lib = None
_torch_ops = None


class SwarmNativeError(RuntimeError):
    pass


def _digest(paths):
    h = hashlib.sha256()
    for p in paths:
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _stamp_path(lib_path):
    return lib_path + ".srchash"


def _is_stale(lib_path, sources):
    """A library is current iff it sits next to a stamp holding the SHA-256 of the sources it was built from
    (content, not mtimes: the snapshot that carries the built .so to the GPU box does not preserve them)."""
    if not os.path.isfile(lib_path):
        return True
    try:
        with open(_stamp_path(lib_path)) as f:
            return f.read().strip() != _digest(sources)
    except OSError:
        return True


def needs_build():
    return _is_stale(LIB_PATH, SOURCES + [HEADER])


def build(force=False, verbose=False):
    """Compile csrc/swarm_b200.cu for sm_100a into the in-tree libswarm_b200.so (nvcc cross-compiles
    without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(nvcc):
        raise SwarmNativeError("nvcc not found; cannot build %s" % LIB_PATH)
    tmp = LIB_PATH + ".tmp.%d" % os.getpid()
    cmd = [nvcc] + NVCC_FLAGS + ["-o", tmp, SOURCES[0]]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
        print(" ".join(cmd))
    digest = _digest(SOURCES + [HEADER])
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise SwarmNativeError("nvcc failed:\n%s\n%s" % (res.stdout, res.stderr))
    if verbose:
        print(res.stderr)
    os.replace(tmp, LIB_PATH)
    with open(_stamp_path(LIB_PATH), "w") as f:
        f.write(digest + "\n")
    return LIB_PATH


def load():
    """Load the C-ABI library, building it first if it is missing or was built from other sources.  A library
    that is stale and cannot be rebuilt is an ERROR (running old kernels silently is worse than not running)."""
    global _lib
    if _lib is not None:
        return _lib
    if _LIB_OVERRIDE:
        lib = ctypes.CDLL(_LIB_OVERRIDE)
    else:
        if needs_build():
            build()                     # raises SwarmNativeError: no compiler, or the compile failed
        lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)           # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.swarm_abi_version() != ABI_VERSION:
        raise SwarmNativeError("ABI version mismatch: %d" % lib.swarm_abi_version())
    _lib = lib
    return lib


def check(status, what="swarm call"):
    if status != 0:
        lib = load()
        msg = lib.swarm_strerror(status).decode()
        if status == -3:
            msg += ": " + lib.swarm_last_cuda_error().decode()
        raise SwarmNativeError("%s failed (%d): %s" % (what, status, msg))


# ------------------------------------------------------------------------------------------------
# The same C ABI exposed as a PyTorch extension (csrc/torch_binding.cpp -> torch.ops.swarm_b200.*)
def torch_ext_needs_build():
    return _is_stale(TORCH_LIB_PATH, [TORCH_SOURCE, HEADER])


def build_torch_ext(force=False):
    """g++ csrc/torch_binding.cpp against the installed torch headers/libs and the in-tree libswarm_b200.so."""
    if not force and not torch_ext_needs_build():
        return TORCH_LIB_PATH
    import torch
    from torch.utils import cpp_extension as ce
    build()
    gxx = shutil.which("g++")
    if gxx is None:
        raise SwarmNativeError("g++ not found; cannot build %s" % TORCH_LIB_PATH)
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    tmp = TORCH_LIB_PATH + ".tmp.%d" % os.getpid()
    cmd = [gxx, "-O2", "-std=c++17", "-fPIC", "-shared",
           "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI)]
    cmd += ["-I" + p for p in ce.include_paths()] + ["-I" + cuda_inc, TORCH_SOURCE, "-o", tmp]
    for lp in ce.library_paths():
        cmd += ["-L" + lp, "-Wl,-rpath," + lp]
    cmd += ["-ltorch", "-ltorch_cpu", "-lc10", "-lc10_cuda", "-ltorch_cuda", "-L" + _PKG_DIR, "-l:libswarm_b200.so",
            "-Wl,-rpath,$ORIGIN"]
    digest = _digest([TORCH_SOURCE, HEADER])
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise SwarmNativeError("g++ failed:\n%s\n%s" % (res.stdout, res.stderr))
    os.replace(tmp, TORCH_LIB_PATH)
    with open(_stamp_path(TORCH_LIB_PATH), "w") as f:
        f.write(digest + "\n")
    return TORCH_LIB_PATH


def load_torch_ops():
    """-> torch.ops.swarm_b200 (building the extension first if its source is newer and g++ exists)."""
    global _torch_ops
    if _torch_ops is not None:
        return _torch_ops
    import torch
    load()                                  # libswarm_b200.so first: the extension links against it
    if torch_ext_needs_build():
        build_torch_ext()                   # raises when the stale extension cannot be rebuilt
    torch.ops.load_library(TORCH_LIB_PATH)
    if int(torch.ops.swarm_b200.abi_version()) != ABI_VERSION:
        raise SwarmNativeError("torch extension ABI version mismatch")
    _torch_ops = torch.ops.swarm_b200
    return _torch_ops


def params_blob(params):
    """The SwarmParams POD as the CPU uint8 tensor the torch ops take."""
    import torch
    return torch.frombuffer(bytearray(bytes(params)), dtype=torch.uint8)
