"""ctypes binding of include/qubism_sv.h (the C ABI the Haskell shim binds with
``foreign import ccall``; INTEGRATION.md).  Thin and literal: one Python function per entry
point, status codes turned into exceptions.  No torch, no numpy compute -- numpy arrays are
only the host buffers handed across the boundary."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("QB_LIB") or os.path.join(_HERE, "libqubism_sv.so")

QB_OK = 0
QB_ERR_ARG, QB_ERR_OOM, QB_ERR_CUDA, QB_ERR_NCCL, QB_ERR_UNSUPPORTED, QB_ERR_STATE = -1, -2, -3, -4, -5, -6
QB_MAX_KQ = 5


class QbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"qubism_sv error {code}: {msg}")
        self.code = code


class QbC64(C.Structure):
    _fields_ = [("re", C.c_double), ("im", C.c_double)]


class QbOp(C.Structure):
    _fields_ = [("kind", C.c_int32), ("target", C.c_int32), ("nctrl", C.c_int32), ("ctrl", C.c_int32 * 4),
                ("_pad", C.c_int32), ("m", QbC64 * 4)]


class QbStats(C.Structure):
    _fields_ = [("ops_submitted", C.c_uint64), ("ops_folded", C.c_uint64), ("ops_executed", C.c_uint64),
                ("passes", C.c_uint64), ("rounds", C.c_uint64), ("simple_launches", C.c_uint64),
                ("reduce_launches", C.c_uint64), ("exchange_bytes", C.c_uint64), ("exchanges", C.c_uint64),
                ("plan_ms", C.c_double), ("fused_ms", C.c_double), ("fused_timed", C.c_uint64), ("tiles", C.c_uint64),
                ("jit_compiled", C.c_uint64), ("jit_launches", C.c_uint64), ("jit_compile_ms", C.c_double),
                ("clones", C.c_uint64), ("cow_fused", C.c_uint64), ("cow_copies", C.c_uint64),
                ("exchanges_fused", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# name -> (restype, argtypes); every symbol include/qubism_sv.h declares
_VP, _I, _U64, _I64, _D = C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_double
_PC64 = C.POINTER(QbC64)
SIGNATURES = {
    "qb_init": (_I, [_I, C.POINTER(_VP)]),
    "qb_dist_unique_id": (_I, [_VP]),
    "qb_init_dist": (_I, [_I, _I, _I, _VP, C.POINTER(_VP)]),
    "qb_init_group": (_I, [C.POINTER(_I), _I, C.POINTER(_VP)]),
    "qb_shutdown": (_I, [_VP]),
    "qb_ctx_rank": (_I, [_VP]),
    "qb_ctx_nranks": (_I, [_VP]),
    "qb_barrier": (_I, [_VP]),
    "qb_last_error": (C.c_char_p, []),
    "qb_version": (C.c_char_p, []),
    "qb_state_create": (_I, [_VP, _I, _I, C.POINTER(_VP)]),
    "qb_state_from_host": (_I, [_VP, _I, _VP, C.POINTER(_VP)]),
    "qb_state_clone": (_I, [_VP, C.POINTER(_VP)]),
    "qb_state_apply_pure": (_I, [_VP, C.POINTER(QbOp), _I64, C.POINTER(_VP)]),
    "qb_state_free": (None, [_VP]),
    "qb_state_nqubits": (_I, [_VP]),
    "qb_state_local_len": (_U64, [_VP]),
    "qb_state_read": (_I, [_VP, _U64, _U64, _VP]),
    "qb_state_read_local": (_I, [_VP, _U64, _U64, _VP]),
    "qb_state_write_local": (_I, [_VP, _U64, _U64, _VP]),
    "qb_apply_1q": (_I, [_VP, _I, _PC64]),
    "qb_apply_1q_range": (_I, [_VP, _I, _I, _PC64]),
    "qb_apply_ctrl_1q": (_I, [_VP, C.POINTER(_I), _I, _I, _PC64]),
    "qb_apply_cnot": (_I, [_VP, _I, _I]),
    "qb_apply_kq": (_I, [_VP, C.POINTER(_I), _I, _VP, C.POINTER(_I), _I]),
    "qb_submit": (_I, [_VP, C.POINTER(QbOp), _I64]),
    "qb_flush": (_I, [_VP]),
    "qb_sync": (_I, [_VP]),
    "qb_sumsq": (_I, [_VP, _I, C.POINTER(_D), C.POINTER(_D)]),
    "qb_collapse": (_I, [_VP, _I, _I]),
    "qb_measure_qubit": (_I, [_VP, _I, _D, C.POINTER(_I), C.POINTER(_D)]),
    "qb_measure_all": (_I, [_VP, C.POINTER(_D), C.POINTER(_I)]),
    "qb_scale": (_I, [_VP, QbC64]),
    "qb_axpy": (_I, [_VP, QbC64, _VP]),
    "qb_neg": (_I, [_VP]),
    "qb_scale_ri": (_I, [_VP, _D, _D]),
    "qb_axpy_ri": (_I, [_VP, _D, _D, _VP]),
    "qb_dotc": (_I, [_VP, _VP, _PC64]),
    "qb_norm2": (_I, [_VP, C.POINTER(_D)]),
    "qb_normalize": (_I, [_VP]),
    "qb_tensor": (_I, [_VP, _VP, C.POINTER(_VP)]),
    "qb_expect_pauli": (_I, [_VP, C.POINTER(_U64), C.POINTER(_U64), _I64, C.POINTER(_D)]),
    "qb_apply_pauli_rot": (_I, [_VP, C.POINTER(_U64), C.POINTER(_U64), C.POINTER(_D), _I64]),
    "qb_pauli_sum": (_I, [_VP, C.POINTER(_U64), C.POINTER(_U64), _VP, _I64, C.POINTER(_VP)]),
    "qb_pauli_rot_grad": (_I, [_VP, C.POINTER(_U64), C.POINTER(_U64), C.POINTER(_D), _I64, C.POINTER(_U64),
                               C.POINTER(_U64), C.POINTER(_D), _I64, C.POINTER(_D), C.POINTER(_D)]),
    "qb_pauli_evolve": (_I, [_VP, C.POINTER(_U64), C.POINTER(_U64), C.POINTER(_D), _I64, _D, C.POINTER(_I64)]),
    "qb_get_stats": (_I, [_VP, C.POINTER(QbStats)]),
    "qb_reset_stats": (_I, [_VP]),
    "qb_ctx_stream": (_VP, [_VP]),
    "qb_set_option": (_I, [_VP, C.c_char_p, _I64]),
    "qb_get_option": (_I64, [_VP, C.c_char_p]),
    "qb_plan_describe": (_I64, [_I, C.POINTER(QbOp), _I64, C.c_char_p, C.c_char_p, _I64]),
    "qb_jit_compile_check": (_I, [C.c_char_p, C.POINTER(_I64)]),
    "qb_jit_sync": (_I, [_VP]),
    "qb_jit_toolchain": (C.c_char_p, []),
}

_lib = None


def lib():
    """Load libqubism_sv.so.  Fails loudly if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -m qubism_b200.build` "
                              "(nvcc, sm_100a).  qubism_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != QB_OK:
        raise QbError(rc, lib().qb_last_error().decode())


def mat4(m) -> "C.Array":
    """2x2 complex (any array-like, row-major [[a,b],[c,d]]) -> qb_c64[4]."""
    a = np.asarray(m, dtype=np.complex128).reshape(4)
    out = (QbC64 * 4)()
    for i in range(4):
        out[i].re, out[i].im = a[i].real, a[i].imag
    return out


def pack_ops(ops):
    """Op stream [("U", q, m) | ("CX", c, t) | ("CU", ctrls, t, m)] -> qb_op array."""
    arr = (QbOp * len(ops))()
    for o, op in zip(arr, ops):
        if op[0] == "U":
            o.kind, o.target, o.nctrl = 0, op[1], 0
            m = np.asarray(op[2], dtype=np.complex128).reshape(4)
        elif op[0] == "CX":
            o.kind, o.target, o.nctrl = 1, op[2], 1
            o.ctrl[0] = op[1]
            continue
        elif op[0] == "CU":
            o.kind, o.target, o.nctrl = 0, op[2], len(op[1])
            for i, c in enumerate(op[1]):
                o.ctrl[i] = c
            m = np.asarray(op[3], dtype=np.complex128).reshape(4)
        else:
            raise ValueError(f"op {op[0]} cannot be packed")
        for i in range(4):
            o.m[i].re, o.m[i].im = m[i].real, m[i].imag
    return arr


def plan_describe(nlocal: int, ops, options: str = "") -> str:
    """Host-only planner dump (no GPU needed)."""
    arr = ops if isinstance(ops, C.Array) else pack_ops(ops)
    need = lib().qb_plan_describe(nlocal, arr, len(arr), options.encode(), None, 0)
    if need < 0:
        check(int(need))
    buf = C.create_string_buffer(int(need))
    lib().qb_plan_describe(nlocal, arr, len(arr), options.encode(), buf, need)
    return buf.value.decode()
