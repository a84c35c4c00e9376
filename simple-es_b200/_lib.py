"""ctypes binding of libses_b200.so (C ABI: include/ses_b200.h)."""
import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
# SES_B200_LIB: an alternative build of the same sources (A/B timing of compile-time choices; tools/ only)
LIB_PATH = os.environ.get("SES_B200_LIB") or os.path.join(_PKG, "libses_b200.so")
# the -DSES_BUILD_TESTS build (include/ses_b200_test.h): test hooks + the alternative kernels behind SES_K1_VARIANT,
# SES_GRU_VARIANT, SES_K2_FUSED, SES_SPREAD_SLOTS8.  Loaded by tests/ and tools/ only (RolloutEngine(test_build=True)).
TEST_LIB_PATH = os.path.join(_PKG, "libses_b200_tests.so")
SOURCES = [os.path.join(_PKG, "csrc", f) for f in (
    "ses_abi.cu", "ses_common.cuh", "rollout_slots.cuh", "rollout_cartpole_mlp.cuh", "rollout_cartpole_gru.cuh", "rollout_mpe.cuh",
    "rollout_classic.cuh", "rollout_gru_generic.cuh",
    "rank.cuh", "update.cuh", "novelty.cuh")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false",           # numerical contract: FMAs only where written (DESIGN.md section 4)
              "-Xcompiler", "-fPIC", "-shared"]


class ses_config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "env", "obs_dim", "act_dim", "gru", "pomdp", "n_agents", "max_step", "eval_ep_num", "population", "group",
        "n_head", "n_parents")] + [("seed", C.c_uint32)] + [(n, C.c_int32) for n in (
            "init_mode", "id_begin", "id_end", "device", "antithetic", "shard_block", "shard_rank", "shard_world", "continuous_action")] + [("reserved", C.c_int32 * 2)]


# every symbol include/ses_b200.h declares: name -> (restype, argtypes)
_vp, _i32, _i64, _u32, _f32, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_float, C.c_double
SYMBOLS = {
    "ses_abi_version": (C.c_int, []),
    "ses_last_error": (C.c_char_p, []),
    "ses_param_count": (C.c_int, [_i32, _i32, _i32]),
    "ses_create": (C.c_int, [C.POINTER(ses_config), C.POINTER(_vp)]),
    "ses_destroy": (C.c_int, [_vp]),
    "ses_rollout": (C.c_int, [_vp, _u32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "ses_evaluate": (C.c_int, [_vp, _u32, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "ses_record": (C.c_int, [_vp, _u32, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ses_rank_desc": (C.c_int, [_vp, _vp, _i32, _i32, _f64, _vp, _vp, _vp]),
    "ses_update_openai": (C.c_int, [_vp, _u32, _vp, _vp, _f64, _f64, _f64, _f64, _f64, _vp, _vp, _vp, _vp, _vp]),
    "ses_update_openai_sgd": (C.c_int, [_vp, _u32, _vp, _vp, _f64, _f64, _f64, _vp, _vp, _vp, _vp]),
    "ses_materialize": (C.c_int, [_vp, _u32, _f32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "ses_update_elite_mean": (C.c_int, [_vp, _u32, _f32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "ses_generation_openai_host": (C.c_int, [_vp, _u32, _f32, _f64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ses_generation_evolution_host": (C.c_int, [_vp, _u32, _f32, _i32, _vp, _vp, _vp, _vp]),
    "ses_generation_genetic_host": (C.c_int, [_vp, _u32, _f32, _vp, _vp, _vp, _vp]),
    "ses_peer_export": (C.c_int, [_vp, _vp]),
    "ses_peer_attach": (C.c_int, [_vp, _vp, _i32, _i32]),
    "ses_peer_fitness_ptr": (C.c_int, [_vp, _i32, C.POINTER(_vp)]),
    "ses_peer_barrier": (C.c_int, [_vp, _vp]),
    "ses_peer_check": (C.c_int, [_vp]),
    "ses_measure_fp32_peak": (C.c_int, [_i32, C.POINTER(C.c_double)]),
    "ses_measure_fp32x2_peak": (C.c_int, [_i32, C.POINTER(C.c_double)]),
    "ses_set_step_counter": (C.c_int, [_vp, _vp]),
    "ses_launch_count": (_i64, [_vp]),
    "ses_set_final_states": (C.c_int, [_vp, _vp]),
    "ses_behavior": (C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    "ses_novelty": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _i32, _vp, _vp]),
    "ses_blend_shaped": (C.c_int, [_vp, _vp, _vp, _i32, _f64, _vp, _vp]),
}
# include/ses_b200_test.h: only in the test build
TEST_SYMBOLS = {
    "ses_test_math": (C.c_int, [_i32, _vp, _vp, _i64, _vp]),
    "ses_test_normals": (C.c_int, [_vp, _u32, _i32, _vp, _vp]),
    "ses_test_k1_geometry": (C.c_int, [_vp, C.POINTER(C.c_int32)]),
    "ses_test_div_total_mass": (C.c_int, [C.c_uint64, C.POINTER(C.c_uint64)]),
    "ses_test_ddiv_fast": (C.c_int, [C.c_uint64, C.POINTER(C.c_uint64)]),
    "ses_test_tanh_fast_exhaustive": (C.c_int, [_f32, _f32, C.POINTER(C.c_uint64)]),
    "ses_test_tanh_x2_exhaustive": (C.c_int, [_i32, _f32, _f32, C.POINTER(C.c_uint64)]),
}


def _nvcc_cmd(out, tests, verbose=False):
    return (["nvcc"] + NVCC_FLAGS + (["-DSES_BUILD_TESTS"] if tests else []) + (["-Xptxas", "-v"] if verbose else []) +
            ["-o", out, SOURCES[0]])


def _stale(path):
    deps = SOURCES + [os.path.join(_ROOT, "include", "ses_b200.h"), os.path.join(_ROOT, "include", "ses_b200_test.h")]
    return not os.path.exists(path) or any(os.path.getmtime(path) < os.path.getmtime(d) for d in deps)


def build_library(force=False, verbose=False, tests=False):
    """Compile the CUDA library for sm_100a in-tree (nvcc cross-compiles without a GPU).  tests=True builds
    libses_b200_tests.so (-DSES_BUILD_TESTS) instead of the product library."""
    path = TEST_LIB_PATH if tests else LIB_PATH
    if force or _stale(path):
        subprocess.check_call(_nvcc_cmd(path, tests, verbose), cwd=_ROOT)
    return path


def build_all(force=False):
    """Product and test builds side by side (two nvcc processes)."""
    jobs = [(p, subprocess.Popen(_nvcc_cmd(p, t), cwd=_ROOT)) for p, t in ((LIB_PATH, False), (TEST_LIB_PATH, True)) if force or _stale(p)]
    for p, proc in jobs:
        if proc.wait() != 0:
            raise RuntimeError("nvcc failed for %s" % p)
    return LIB_PATH, TEST_LIB_PATH


_libs = {}


def load(tests=False):
    """Load libses_b200.so (tests=True: libses_b200_tests.so); no fallback -- a missing library is an error."""
    if tests in _libs:
        return _libs[tests]
    path = TEST_LIB_PATH if tests else LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(
            "simple-es_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). The engine has no CPU fallback." % path)
    lib = C.CDLL(path)
    syms = dict(SYMBOLS, **TEST_SYMBOLS) if tests else SYMBOLS
    for name, (res, args) in syms.items():
        fn = getattr(lib, name)          # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    if lib.ses_abi_version() != 1:
        raise RuntimeError("simple-es_b200: ABI version mismatch")
    _libs[tests] = lib
    return lib


def check(rc, lib=None):
    if rc != 0:
        raise RuntimeError("simple-es_b200: " + (lib or load()).ses_last_error().decode())
