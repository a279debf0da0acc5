"""ctypes binding of libpbn_b200.so (include/pbn_b200.h).

There is no CPU fallback: if the shared library is missing, or a call fails, this module
raises.  PyTorch only lends device memory (``tensor.data_ptr()``) and the current stream.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

__all__ = ["lib", "load_library", "PbnError", "NetDesc", "StepArgs", "HostIO", "Replay", "Per", "check", "LIB_PATH", "EXPORTS"]

LIB_PATH = Path(__file__).resolve().parent / "libpbn_b200.so"

PBN_OK = 0
PBN_ERR_INVALID = -1
PBN_ERR_UNSUPPORTED = -3
DP_MAX_GENES = 28  # PBN_DP_MAX_GENES
PERT_MODES = {"none": 0, "A": 1, "B": 2, "C": 3}
KERNEL_KINDS = {"auto": 0, "scalar": 1, "sliced": 2}
STEP_AUTORESET = 1
STEP_PDL = 2
STEP_NO_COUNT = 4
STEP_CHAIN = 8
UNPACK_U8, UNPACK_F32 = 0, 1
N_STATS = 8
STAT_NAMES = ("steps", "episodes", "terminated", "truncated", "ep_len_sum", "flips", "perturbed", "reserved")

# every symbol include/pbn_b200.h declares (tests check the built library exports them all)
EXPORTS = (
    "pbn_create", "pbn_destroy", "pbn_update_attractors", "pbn_step", "pbn_step_injected", "pbn_reset",
    "pbn_unpack", "pbn_pack", "pbn_attractor_id", "pbn_kernel_kind", "pbn_words_per_state",
    "pbn_launch_count", "pbn_last_error", "pbn_version", "pbn_jit_source", "pbn_jit_precompile",
    "pbn_advance_counter", "pbn_step_host", "pbn_replay_observe", "pbn_replay_commit", "pbn_replay_sample",
    "pbn_observe", "pbn_in_target", "pbn_rollout_track", "pbn_rollout_reduce",
    "pbn_visit_count", "pbn_successor_sets", "pbn_closure_expand", "pbn_closure_reach",
    "pbn_rollout", "pbn_rollout_record", "pbn_record_states",
    "pbn_resident_words", "pbn_resident_import", "pbn_resident_export", "pbn_reward_table", "pbn_attractor_hash_slots",
    "pbn_per_tree_floats", "pbn_per_init", "pbn_per_push", "pbn_per_update", "pbn_per_sample",
    "pbn_dp_workspace_bytes", "pbn_dp_expect", "pbn_dp_improve", "pbn_dp_push",
)


class PbnError(RuntimeError):
    def __init__(self, code: int, message: str = ""):
        super().__init__("pbn_b200 error %d: %s" % (code, message))
        self.code = code
        self.message = message

    def __reduce__(self):   # picklable (worker processes of build() report JIT failures)
        return (PbnError, (self.code, self.message))


class NetDesc(C.Structure):
    _fields_ = [
        ("n_genes", C.c_int32),
        ("n_funcs", C.c_int32),
        ("func_offset", C.c_void_p),
        ("func_arity", C.c_void_p),
        ("func_inputs", C.c_void_p),
        ("func_lut", C.c_void_p),
        ("func_cum", C.c_void_p),
        ("survival", C.c_void_p),
        ("bins", C.c_int32),
        ("horizon", C.c_int32),
        ("perturb_mode", C.c_int32),
        ("perturb_p", C.c_double),
        ("r_success", C.c_float),
        ("r_step", C.c_float),
        ("r_action", C.c_float),
        ("seed", C.c_uint64),
        ("device", C.c_int32),
        ("kernel", C.c_int32),
        ("n_wide", C.c_int32),
        ("reserved0", C.c_int32),
        ("wide_inputs", C.c_void_p),
        ("wide_lut_offset", C.c_void_p),
        ("wide_lut", C.c_void_p),
        ("r_wrong", C.c_float),
        ("reserved1", C.c_float),
    ]


class StepArgs(C.Structure):
    _fields_ = [
        ("state", C.c_void_p),
        ("actions", C.c_void_p),
        ("target_id", C.c_void_p),
        ("source_id", C.c_void_p),
        ("t", C.c_void_p),
        ("reward", C.c_void_p),
        ("terminated", C.c_void_p),
        ("truncated", C.c_void_p),
        ("final_state", C.c_void_p),
        ("pert_mask", C.c_void_p),
        ("sel", C.c_void_p),
        ("stats", C.c_void_p),
        ("step_ctr_dev", C.c_void_p),
        ("step_ctr", C.c_uint64),
        ("env_offset", C.c_int64),
        ("n_envs", C.c_int64),
        ("flags", C.c_uint32),
        ("reserved", C.c_uint32),
        ("resident", C.c_void_p),
    ]


class HostIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p),
        ("actions_dev", C.c_void_p),
        ("state", C.c_void_p),
        ("reward", C.c_void_p),
        ("terminated", C.c_void_p),
        ("truncated", C.c_void_p),
        ("n_chunks", C.c_int32),
        ("reserved", C.c_int32),
        ("state32", C.c_void_p),
        ("done", C.c_void_p),
        ("packed", C.c_void_p),
        ("actions16", C.c_void_p),
        ("actions16_dev", C.c_void_p),
    ]


class Replay(C.Structure):
    _fields_ = [
        ("state", C.c_void_p),
        ("next_state", C.c_void_p),
        ("target_id", C.c_void_p),
        ("actions", C.c_void_p),
        ("reward", C.c_void_p),
        ("done", C.c_void_p),
        ("capacity", C.c_int64),
    ]


class Per(C.Structure):
    _fields_ = [
        ("tree", C.c_void_p),
        ("max_p", C.c_void_p),
        ("capacity", C.c_int64),
        ("alpha", C.c_float),
        ("reserved", C.c_float),
    ]


_lib: Optional[C.CDLL] = None


def load_library(path: Optional[os.PathLike] = None) -> C.CDLL:
    """dlopen the C-ABI library and declare its prototypes.  Raises if it has not been built
    (``python -c 'import __graft_entry__ as g; g.build()'`` or ``make -C pbn_rl_b200/csrc``)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path is not None else LIB_PATH
    if not p.exists():
        raise FileNotFoundError(
            "%s not found: the CUDA extension is not built (run __graft_entry__.build()); "
            "pbn_rl_b200 has no CPU fallback" % p)
    lib = C.CDLL(str(p))
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    lib.pbn_create.argtypes = [C.POINTER(NetDesc), C.POINTER(vp)]
    lib.pbn_create.restype = C.c_int
    lib.pbn_destroy.argtypes = [vp]
    lib.pbn_destroy.restype = None
    lib.pbn_update_attractors.argtypes = [vp, vp, vp, vp, i32, vp, vp]
    lib.pbn_update_attractors.restype = C.c_int
    lib.pbn_step.argtypes = [vp, C.POINTER(StepArgs), vp]
    lib.pbn_step.restype = C.c_int
    lib.pbn_step_host.argtypes = [vp, C.POINTER(StepArgs), C.POINTER(HostIO), vp]
    lib.pbn_step_host.restype = C.c_int
    lib.pbn_replay_observe.argtypes = [vp, C.POINTER(Replay), i64, vp, vp, i64, vp]
    lib.pbn_replay_observe.restype = C.c_int
    lib.pbn_replay_commit.argtypes = [vp, C.POINTER(Replay), i64, vp, vp, vp, vp, vp, i64, vp]
    lib.pbn_replay_commit.restype = C.c_int
    lib.pbn_replay_sample.argtypes = [vp, C.POINTER(Replay), vp, i64, vp, vp, vp, vp, vp, vp]
    lib.pbn_replay_sample.restype = C.c_int
    lib.pbn_per_tree_floats.argtypes = [i64]
    lib.pbn_per_tree_floats.restype = i64
    lib.pbn_per_init.argtypes = [vp, C.POINTER(Per), vp]
    lib.pbn_per_init.restype = C.c_int
    lib.pbn_per_push.argtypes = [vp, C.POINTER(Per), i64, i64, vp]
    lib.pbn_per_push.restype = C.c_int
    lib.pbn_per_update.argtypes = [vp, C.POINTER(Per), vp, vp, i64, C.c_float, vp]
    lib.pbn_per_update.restype = C.c_int
    lib.pbn_per_sample.argtypes = [vp, C.POINTER(Per), vp, i64, C.c_float, vp, vp, vp]
    lib.pbn_per_sample.restype = C.c_int
    lib.pbn_dp_workspace_bytes.argtypes = [vp]
    lib.pbn_dp_workspace_bytes.restype = i64
    lib.pbn_dp_expect.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.pbn_dp_expect.restype = C.c_int
    lib.pbn_dp_improve.argtypes = [vp, vp, u64, i32, C.c_double, vp, vp, vp, vp]
    lib.pbn_dp_improve.restype = C.c_int
    lib.pbn_dp_push.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.pbn_dp_push.restype = C.c_int
    lib.pbn_observe.argtypes = [vp, vp, vp, vp, i64, vp]
    lib.pbn_observe.restype = C.c_int
    lib.pbn_in_target.argtypes = [vp, vp, vp, vp, i64, vp]
    lib.pbn_in_target.restype = C.c_int
    lib.pbn_rollout_track.argtypes = [vp, vp, vp, vp, i32, i64, vp, vp]
    lib.pbn_rollout_track.restype = C.c_int
    lib.pbn_rollout_reduce.argtypes = [vp, vp, vp, i64, i32, i32, vp, vp, vp]
    lib.pbn_rollout_reduce.restype = C.c_int
    lib.pbn_visit_count.argtypes = [vp, vp, vp, i64, vp, vp, vp, i64, vp, vp]
    lib.pbn_visit_count.restype = C.c_int
    lib.pbn_successor_sets.argtypes = [vp, vp, i64, vp, vp, vp]
    lib.pbn_successor_sets.restype = C.c_int
    lib.pbn_closure_expand.argtypes = [vp, vp, i64, i64, i64, vp, vp, vp, vp, i64, i32, vp, vp]
    lib.pbn_closure_expand.restype = C.c_int
    lib.pbn_closure_reach.argtypes = [vp, vp, i64, vp, vp, vp, vp, i64, vp, vp]
    lib.pbn_closure_reach.restype = C.c_int
    lib.pbn_attractor_hash_slots.argtypes = [vp]
    lib.pbn_attractor_hash_slots.restype = C.c_int
    lib.pbn_reward_table.argtypes = [vp, vp, i32]
    lib.pbn_reward_table.restype = C.c_int
    lib.pbn_resident_words.argtypes = [vp, i64]
    lib.pbn_resident_words.restype = i64
    lib.pbn_resident_import.argtypes = [vp, vp, vp, vp, vp, i64, vp]
    lib.pbn_resident_import.restype = C.c_int
    lib.pbn_resident_export.argtypes = [vp, vp, vp, vp, vp, i64, vp]
    lib.pbn_resident_export.restype = C.c_int
    lib.pbn_rollout.argtypes = [vp, vp, i64, u64, i64, i64, vp, vp]
    lib.pbn_rollout.restype = C.c_int
    lib.pbn_rollout_record.argtypes = [vp, vp, i64, u64, i64, i64, i32, vp, i32, vp, vp, vp, vp]
    lib.pbn_rollout_record.restype = C.c_int
    lib.pbn_record_states.argtypes = [vp, vp, i64, vp, i32, vp, vp, vp]
    lib.pbn_record_states.restype = C.c_int
    lib.pbn_step_injected.argtypes = [vp, C.POINTER(StepArgs), vp]
    lib.pbn_step_injected.restype = C.c_int
    lib.pbn_reset.argtypes = [vp, vp, vp, vp, vp, vp, u64, i64, i64, vp]
    lib.pbn_reset.restype = C.c_int
    lib.pbn_unpack.argtypes = [vp, vp, vp, i32, i64, vp]
    lib.pbn_unpack.restype = C.c_int
    lib.pbn_pack.argtypes = [vp, vp, vp, i64, vp]
    lib.pbn_pack.restype = C.c_int
    lib.pbn_attractor_id.argtypes = [vp, vp, vp, i64, vp]
    lib.pbn_attractor_id.restype = C.c_int
    lib.pbn_kernel_kind.argtypes = [vp]
    lib.pbn_kernel_kind.restype = C.c_int
    lib.pbn_words_per_state.argtypes = [vp]
    lib.pbn_words_per_state.restype = C.c_int
    lib.pbn_launch_count.argtypes = [vp, C.POINTER(u64)]
    lib.pbn_launch_count.restype = C.c_int
    lib.pbn_jit_source.argtypes = [C.POINTER(NetDesc), C.c_int, C.c_char_p, i64]
    lib.pbn_jit_source.restype = i64
    lib.pbn_jit_precompile.argtypes = [C.POINTER(NetDesc)]
    lib.pbn_jit_precompile.restype = C.c_int
    lib.pbn_advance_counter.argtypes = [vp, vp, u64, vp]
    lib.pbn_advance_counter.restype = C.c_int
    lib.pbn_last_error.argtypes = []
    lib.pbn_last_error.restype = C.c_char_p
    lib.pbn_version.argtypes = []
    lib.pbn_version.restype = C.c_char_p
    if path is None:
        _lib = lib
    return lib


def lib() -> C.CDLL:
    return load_library()


def check(code: int) -> None:
    if code != PBN_OK:
        msg = lib().pbn_last_error()
        raise PbnError(code, msg.decode("utf-8", "replace") if msg else "")
