"""ctypes binding of libcarenv_b200.so (C ABI: include/carenv_b200.h).

There is no CPU implementation behind this module: if the shared library has not been
built (``python -c "import __graft_entry__ as g; g.build()"`` or ``ppo_car_b200.build()``)
every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_PKG)
LIB_PATH = os.environ.get("CARENV_LIB") or os.path.join(_PKG, "libcarenv_b200.so")   # override: kernel experiments
SOURCES = [os.path.join(_PKG, "csrc", f)
           for f in ("carenv_kernels.cu", "carenv_core.cuh", "carenv_tables.h", "policy_core.cuh", "tc_mlp.cuh",
                     "ppo_update.cuh", "ppo_epoch.cuh", "policy_rollout.cuh", "policy_abi.cuh", "policy_eval.cuh",
                     "population.cuh")]
HEADER = os.path.join(ROOT, "include", "carenv_b200.h")

ACT_U8, ACT_I32, ACT_I64 = 0, 1, 2
FLAG_U8, FLAG_F32 = 0, 1

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "--shared",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off", "-std=c++17"]

_lib = None


class CarEnvError(RuntimeError):
    pass


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    deps = SOURCES + [HEADER]
    if (not force and os.path.exists(LIB_PATH)
            and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps)):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH, SOURCES[0]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise CarEnvError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


def lib():
    """Load the shared library (once).  Raises CarEnvError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CarEnvError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built and there is no CPU fallback. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'`.")
    L = C.CDLL(LIB_PATH)
    vp, i32, f64 = C.c_void_p, C.c_int, C.c_double
    L.carenv_abi_version.restype = i32
    L.carenv_last_error.restype = C.c_char_p
    L.carenv_create.argtypes = [vp, i32, vp, i32, f64, f64, f64, i32, C.POINTER(vp)]
    L.carenv_destroy.argtypes = [vp]
    L.carenv_reset_obs.argtypes = [vp, vp]
    L.carenv_reset.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    L.carenv_step.argtypes = [vp, i32, vp, vp, vp, vp, i32, f64, vp, vp, vp, vp, i32, vp, vp]
    L.carenv_rollout.argtypes = [vp, i32, i32, vp, vp, vp, vp, i32, f64, vp, vp, vp, vp, i32, vp, vp]
    L.carenv_step_host.argtypes = L.carenv_step.argtypes
    L.carenv_step_host_records.argtypes = [vp, i32, vp, vp, vp, vp, i32, f64, vp, vp, vp, vp]
    L.carenv_step_records.argtypes = [vp, i32, vp, vp, vp, vp, i32, f64, vp, vp, vp, vp]
    L.carenv_step_final.argtypes = [vp, i32, vp, vp, vp, vp, i32, f64, vp, vp, vp, vp, vp, i32, vp, vp]
    L.carenv_multi_create.argtypes = [vp, i32, C.POINTER(vp)]
    L.carenv_multi_destroy.argtypes = [vp]
    L.carenv_multi_reset.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp]
    L.carenv_multi_rollout.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, i32, f64, vp, vp, vp, vp, i32, vp, vp]
    L.carenv_render.argtypes = [vp, i32, i32, vp, vp, vp, vp, i32, i32, vp, vp]
    L.carenv_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    L.carenv_host_free.argtypes = [vp]
    L.carenv_rollout_poses.argtypes = L.carenv_rollout.argtypes
    L.carenv_observe.argtypes = [vp, C.c_longlong, vp, vp, vp, vp]
    L.carenv_stats.argtypes = [vp, vp, i32]
    L.carenv_set_option.argtypes = [vp, C.c_char_p, i32]
    L.gae_reverse_scan.argtypes = [vp] * 9 + [i32, i32, f64, f64, vp]
    L.carenv_bench_ffma.argtypes = [i32, i32, vp, vp]
    L.carenv_tc_gemm_test.argtypes = [vp, vp, vp, vp]
    L.carenv_tc_gemm_test.restype = i32
    L.carenv_ppo_num_params.restype = i32
    L.carenv_ppo_scratch_floats.argtypes = [i32]
    L.carenv_ppo_scratch_floats.restype = i32
    L.carenv_ppo_grad.argtypes = [vp] * 8 + [vp, i32, vp, vp, vp, vp, vp, i32, f64, f64, f64, vp, vp, vp]
    L.carenv_ppo_grad.restype = i32
    L.carenv_ppo_adam.argtypes = [vp] * 8 + [vp, f64, vp, vp, vp, vp, f64, f64, f64, f64, vp, i32, f64, f64, vp, vp]
    L.carenv_ppo_adam.restype = i32
    L.carenv_ppo_comm_create.argtypes = [i32, i32, C.POINTER(vp), vp]
    L.carenv_ppo_comm_create.restype = i32
    L.carenv_ppo_comm_connect.argtypes = [vp, vp]
    L.carenv_ppo_comm_connect.restype = i32
    L.carenv_ppo_comm_destroy.argtypes = [vp]
    L.carenv_ppo_comm_destroy.restype = i32
    L.carenv_ppo_epoch_workspace_floats.restype = i32
    L.carenv_ppo_epoch.argtypes = [vp] * 8 + [vp] * 6 + [i32, i32, f64, f64, f64, vp, vp, vp, vp, f64, f64, f64, f64,
                                                         vp, vp, vp, vp, i32, vp, vp]
    L.carenv_ppo_epoch.restype = i32
    L.carenv_ppo_epoch_kl.argtypes = L.carenv_ppo_epoch.argtypes + [f64, vp, vp]
    L.carenv_ppo_epoch_kl.restype = i32
    L.carenv_pack_policy.argtypes = [i32] + [vp] * 10
    L.carenv_pack_policy.restype = i32
    L.carenv_policy_weights_floats.restype = i32
    L.carenv_policy_rollout.argtypes = [vp, vp, i32, i32, i32, C.c_ulonglong, C.c_ulonglong, vp, vp, vp, vp, vp, vp,
                                        f64] + [vp] * 10
    L.carenv_policy_rollout_warp.argtypes = [vp] + [vp] * 8 + [i32, i32, i32, C.c_ulonglong, C.c_ulonglong, vp, vp, vp, vp, vp,
                                                            vp, f64] + [vp] * 10
    L.carenv_policy_rollout_warp.restype = i32
    L.carenv_policy_weights_floats_tc.restype = i32
    L.carenv_policy_rollout_tc.argtypes = L.carenv_policy_rollout.argtypes
    L.carenv_policy_eval.argtypes = [vp] * 5 + [C.c_longlong, C.c_ulonglong, i32, C.c_ulonglong, vp, i32, vp, vp, vp]
    L.carenv_policy_eval.restype = i32
    L.carenv_policy_rollout_tc_multi.argtypes = [vp, vp] + L.carenv_policy_rollout_tc.argtypes[1:]
    L.carenv_policy_rollout_tc_multi.restype = i32
    L.carenv_policy_eval_multi.argtypes = [vp, vp] + L.carenv_policy_eval.argtypes[1:]
    L.carenv_policy_eval_multi.restype = i32
    L.carenv_pack_policy_pop.argtypes = [i32, i32] + [vp] * 10
    L.carenv_policy_rollout_warp_pop.argtypes = [vp, i32] + [vp] * 8 + [i32, i32, vp, C.c_ulonglong] + [vp] * 6 + \
        [f64] + [vp] * 10
    L.carenv_policy_rollout_tc_pop.argtypes = [vp, i32, vp, i32, i32, vp, C.c_ulonglong] + [vp] * 6 + [f64] + [vp] * 10
    L.carenv_ppo_epoch_pop.argtypes = [i32] + [vp] * 8 + [vp] * 6 + [i32, i32] + [vp] * 5 + [f64, f64, f64] + [vp] * 5
    L.carenv_ppo_epoch_pop_kl.argtypes = L.carenv_ppo_epoch_pop.argtypes + [f64, vp, vp]
    L.carenv_ppo_epoch_pop_resident_clusters.argtypes = [vp]
    L.carenv_policy_eval_pop.argtypes = [vp, i32] + [vp] * 4 + [C.c_longlong, C.c_ulonglong, i32, vp, vp, i32, vp, vp,
                                                               vp]
    for name in ("carenv_pack_policy_pop", "carenv_policy_rollout_warp_pop", "carenv_policy_rollout_tc_pop",
                 "carenv_ppo_epoch_pop", "carenv_ppo_epoch_pop_kl", "carenv_ppo_epoch_pop_cluster_size", "carenv_ppo_epoch_pop_resident_clusters",
                 "carenv_policy_eval_pop"):
        getattr(L, name).restype = i32
    for name in ("carenv_create", "carenv_destroy", "carenv_reset_obs", "carenv_reset", "carenv_step",
                 "carenv_rollout", "carenv_rollout_poses", "carenv_observe", "carenv_step_host", "carenv_step_host_records", "carenv_step_records", "carenv_step_final", "carenv_multi_create", "carenv_multi_destroy", "carenv_multi_reset",
                 "carenv_multi_rollout", "carenv_render", "carenv_host_alloc", "carenv_host_free", "carenv_stats", "gae_reverse_scan", "carenv_bench_ffma", "carenv_set_option", "carenv_policy_rollout", "carenv_policy_rollout_tc"):
        getattr(L, name).restype = i32
    if L.carenv_abi_version() != 1:
        raise CarEnvError("libcarenv_b200.so ABI version mismatch; rebuild")
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().carenv_last_error()
        raise CarEnvError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
