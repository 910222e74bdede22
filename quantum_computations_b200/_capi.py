"""ctypes declarations for the C ABI in ``include/qsim_b200.h``.

``declare(lib)`` attaches argument/return types to a loaded library.  The
product binds ``csrc/libqsim_b200.so`` through ``engine.py``; the CPU tests bind
the host emulator (same ABI, host pointers) through a backend class of their own.
"""
from __future__ import annotations

import ctypes as C

c_int_p = C.POINTER(C.c_int)
c_double_p = C.POINTER(C.c_double)
c_void_pp = C.POINTER(C.c_void_p)


class PlanOptions(C.Structure):
    _fields_ = [
        ("tile_bits", C.c_int32),
        ("low_bits", C.c_int32),
        ("max_group", C.c_int32),
        ("max_dense_ops", C.c_int32),
        ("lookahead", C.c_int32),
        ("merge_1q", C.c_int32),
        ("defer_tail", C.c_int32),
        ("max_layers", C.c_int32),
        ("cta_log2", C.c_int32),
        ("reserved0", C.c_int32),
        ("apply_tail_mask", C.c_uint64),
    ]


class PlanStats(C.Structure):
    _fields_ = [
        ("n_input_ops", C.c_int64),
        ("n_merged_ops", C.c_int64),
        ("n_passes", C.c_int64),
        ("n_steps", C.c_int64),
        ("n_dense", C.c_int64),
        ("n_sign", C.c_int64),
        ("n_generic", C.c_int64),
        ("n_warp_syncs", C.c_int64),
        ("n_layers", C.c_int64),
    ]

    def as_dict(self) -> dict:
        return {name: int(getattr(self, name)) for name, _ in self._fields_}


# name -> (restype, argtypes); this table is also what tests/test_capi_symbols.py
# checks against include/qsim_b200.h
SIGNATURES = {
    "qsim_last_error": (C.c_char_p, []),
    "qsim_version": (C.c_int, []),
    "qsim_has_cuda": (C.c_int, []),
    "qsim_circuit_create": (C.c_int, [C.c_int, c_void_pp]),
    "qsim_circuit_add_matrix": (C.c_int, [C.c_void_p, C.c_int, c_int_p, c_double_p]),
    "qsim_circuit_add_many": (C.c_int, [C.c_void_p, C.c_int64, c_int_p, c_int_p, c_double_p]),
    "qsim_circuit_num_ops": (C.c_int, [C.c_void_p]),
    "qsim_circuit_destroy": (None, [C.c_void_p]),
    "qsim_plan_compile": (C.c_int, [C.c_void_p, C.POINTER(PlanOptions), c_void_pp]),
    "qsim_plan_stats": (C.c_int, [C.c_void_p, C.POINTER(PlanStats)]),
    "qsim_plan_execute": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "qsim_plan_residual": (C.c_int, [C.c_void_p, c_double_p]),
    "qsim_plan_destroy": (None, [C.c_void_p]),
    "qsim_apply_matrix": (C.c_int, [C.c_void_p, C.c_int, c_int_p, C.c_int, c_double_p, C.c_void_p, C.c_void_p]),
    "qsim_apply_diagonal": (C.c_int, [C.c_void_p, C.c_int, c_int_p, C.c_int, c_double_p, C.c_void_p]),
    "qsim_apply_permutation": (C.c_int, [C.c_void_p, C.c_int, c_int_p, C.c_int, c_int_p, C.c_void_p]),
    "qsim_apply_superop": (C.c_int, [C.c_void_p, C.c_int, c_int_p, C.c_int, c_double_p, C.c_void_p, C.c_void_p]),
    "qsim_init_product": (C.c_int, [C.c_void_p, C.c_int, c_double_p, C.c_void_p]),
    "qsim_measure_probs": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_double_p, c_double_p, c_double_p, C.c_void_p]),
    "qsim_collapse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, c_double_p, C.c_double, C.c_void_p]),
    "qsim_insert": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, c_double_p, C.c_void_p]),
    "qsim_reduce_norm2": (C.c_int, [C.c_void_p, C.c_uint64, c_double_p, C.c_void_p]),
    "qsim_reduce_inner": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, c_double_p, C.c_void_p]),
    "qsim_reduce_expect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, c_double_p, C.c_void_p]),
    "qsim_reduce_purity": (C.c_int, [C.c_void_p, C.c_int, c_double_p, C.c_void_p]),
    "qsim_reduce_trace": (C.c_int, [C.c_void_p, C.c_int, c_double_p, C.c_void_p]),
    "qsim_expect_pauli": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, c_double_p, C.c_void_p]),
    "qsim_expect_pauli_dm": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, c_double_p,
                                       C.c_void_p]),
    "qsim_marginal_probs": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_int_p, C.c_void_p, C.c_void_p]),
    "qsim_marginal_probs_dm": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_int_p, C.c_void_p, C.c_void_p]),
    "qsim_sample_workspace_bytes": (C.c_int, [C.c_int, C.c_int64, C.POINTER(C.c_uint64)]),
    "qsim_sample": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, c_double_p, C.c_void_p,
                              C.c_uint64, C.c_void_p]),
    "qsim_sample_dm": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, c_double_p, C.c_void_p,
                                 C.c_uint64, C.c_void_p]),
    "qsim_rb_batch": (C.c_int, [C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "qsim_traj_batch": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "qsim_swap_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                 C.c_uint64, C.c_uint64, C.c_void_p]),
    "qsim_swap_unpack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                   C.c_uint64, C.c_uint64, C.c_void_p]),
    "qsim_peer_alloc": (C.c_int, [C.c_int, C.c_uint64, c_void_pp]),
    "qsim_peer_free": (C.c_int, [C.c_void_p]),
    "qsim_ipc_export": (C.c_int, [C.c_void_p, C.c_char_p]),
    "qsim_ipc_import": (C.c_int, [C.c_int, C.c_char_p, c_void_pp]),
    "qsim_ipc_release": (C.c_int, [C.c_void_p]),
    "qsim_peer_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "qsim_ipc_export_ex": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_uint64)]),
    "qsim_exchange_p2p": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.POINTER(C.c_int),
                                    C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]),
    "qsim_launch_count": (C.c_int64, []),
}


def declare(lib) -> None:
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes


class QsimError(RuntimeError):
    """A C-ABI call returned a non-zero status."""


_ARG, _CUDA, _UNSUPPORTED, _NOMEM = -1, -2, -3, -4


def check(lib, status: int) -> None:
    if status == 0:
        return
    msg = lib.qsim_last_error()
    text = msg.decode("utf-8", "replace") if msg else "unknown error"
    if status == _ARG:
        raise ValueError(text)
    if status == _UNSUPPORTED:
        raise NotImplementedError(text)
    if status == _NOMEM:
        raise MemoryError(text)
    raise QsimError(text)
