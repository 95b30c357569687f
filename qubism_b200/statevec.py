"""Host-side mirror of ``Qubism.StateVec`` (src/Qubism/StateVec.hs:14-25) over the C ABI.

Same names and argument meaning as the reference module; the state lives on the GPU and is
uniquely owned by the Python object (the role a ``ForeignPtr`` plays in the Haskell shim).
Functions that are pure in the reference (``normalize``, ``collapse``, ``tensor``, ``#>``)
return a NEW ``StateVec`` (clone + in-place op); the ``StateT``-style ones (``measureQubit``,
``measure``, ``gate``) mutate in place.  Bits are the ints 0 (Zero) / 1 (One), CReg.hs:14.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi


class Context:
    """One per process and GPU (qb_ctx).  ``Context.default()`` is device 0 / LOCAL_RANK."""

    _default = None

    def __init__(self, device: int = 0, rank: int = 0, nranks: int = 1, nccl_id: bytes | None = None):
        self.L = capi.lib()
        self.h = C.c_void_p()
        if nranks > 1:
            buf = C.create_string_buffer(nccl_id, 128)
            capi.check(self.L.qb_init_dist(device, rank, nranks, buf, C.byref(self.h)))
        else:
            capi.check(self.L.qb_init(device, C.byref(self.h)))
        self.device, self.rank, self.nranks = device, rank, nranks

    @classmethod
    def default(cls) -> "Context":
        if cls._default is None:
            cls._default = Context(0)
        return cls._default

    @classmethod
    def group(cls, devices) -> list:
        """Rank group inside this process (qb_init_group): one Context per entry of ``devices``; the
        same device repeated gives virtual ranks on one GPU.  Drive each rank from its own thread."""
        L = capi.lib()
        n = len(devices)
        arr = (C.c_int * n)(*devices)
        hs = (C.c_void_p * n)()
        capi.check(L.qb_init_group(arr, n, hs))
        out = []
        for r in range(n):
            c = cls.__new__(cls)
            c.L, c.h, c.device, c.rank, c.nranks = L, C.c_void_p(hs[r]), devices[r], r, n
            out.append(c)
        return out

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        capi.check(capi.lib().qb_dist_unique_id(buf))
        return buf.raw

    def set_option(self, name: str, value: int):
        capi.check(self.L.qb_set_option(self.h, name.encode(), int(value)))

    def get_option(self, name: str) -> int:
        return int(self.L.qb_get_option(self.h, name.encode()))

    def stats(self) -> dict:
        st = capi.QbStats()
        capi.check(self.L.qb_get_stats(self.h, C.byref(st)))
        return st.as_dict()

    def reset_stats(self):
        capi.check(self.L.qb_reset_stats(self.h))

    def sync(self):
        capi.check(self.L.qb_sync(self.h))

    def jit_wait(self):
        """Block until no specialised kernel is being compiled in the background."""
        capi.check(self.L.qb_jit_sync(self.h))

    def barrier(self):
        capi.check(self.L.qb_barrier(self.h))

    def stream(self) -> int:
        return int(self.L.qb_ctx_stream(self.h) or 0)

    def close(self):
        if self.h:
            self.L.qb_shutdown(self.h)
            self.h = C.c_void_p()


class StateVec:
    """``StateVec n`` (StateVec.hs:43-44): 2^n Complex Double amplitudes, device resident."""

    def __init__(self, handle, ctx: Context):
        self._h = handle
        self.ctx = ctx

    def __del__(self):
        try:
            if self._h:
                self.ctx.L.qb_state_free(self._h)
                self._h = None
        except Exception:
            pass

    # -- construction ------------------------------------------------------------------
    @staticmethod
    def create(n: int, basis: bool = True, ctx: Context | None = None) -> "StateVec":
        ctx = ctx or Context.default()
        h = C.c_void_p()
        capi.check(ctx.L.qb_state_create(ctx.h, n, 1 if basis else 0, C.byref(h)))
        return StateVec(h, ctx)

    @staticmethod
    def from_host(amps, n: int | None = None, ctx: Context | None = None) -> "StateVec":
        """``UnsafeMkStateVec (LA.fromList ...)``.  Distributed: pass this rank's shard and n."""
        ctx = ctx or Context.default()
        a = np.ascontiguousarray(amps, dtype=np.complex128)
        if n is None:
            n = int(a.size).bit_length() - 1
            if a.size != 1 << n:
                raise ValueError("length is not a power of two")
        h = C.c_void_p()
        capi.check(ctx.L.qb_state_from_host(ctx.h, n, a.ctypes.data_as(C.c_void_p), C.byref(h)))
        return StateVec(h, ctx)

    def clone(self) -> "StateVec":
        h = C.c_void_p()
        capi.check(self.ctx.L.qb_state_clone(self._h, C.byref(h)))
        return StateVec(h, self.ctx)

    def apply_pure(self, ops) -> "StateVec":
        """``g #> sv`` in one crossing (qb_state_apply_pure): a NEW state, ``self`` stays valid."""
        arr = ops if isinstance(ops, C.Array) else capi.pack_ops(ops)
        h = C.c_void_p()
        capi.check(self.ctx.L.qb_state_apply_pure(self._h, arr, len(arr), C.byref(h)))
        return StateVec(h, self.ctx)

    def free(self):
        """Release the handle now (what the ForeignPtr finalizer does at some later GC)."""
        if self._h:
            self.ctx.L.qb_state_free(self._h)
            self._h = None

    # -- observation -------------------------------------------------------------------
    @property
    def n(self) -> int:
        return int(self.ctx.L.qb_state_nqubits(self._h))

    def to_host(self, first: int = 0, count: int | None = None) -> np.ndarray:
        count = (1 << self.n) - first if count is None else count
        out = np.empty(count, dtype=np.complex128)
        capi.check(self.ctx.L.qb_state_read(self._h, first, count, out.ctypes.data_as(C.c_void_p)))
        return out

    def local_to_host(self, first: int = 0, count: int | None = None) -> np.ndarray:
        total = int(self.ctx.L.qb_state_local_len(self._h))
        count = total - first if count is None else count
        out = np.empty(count, dtype=np.complex128)
        capi.check(self.ctx.L.qb_state_read_local(self._h, first, count, out.ctypes.data_as(C.c_void_p)))
        return out

    def write_local(self, amps, first: int = 0):
        """Upload a host buffer into this rank's shard (qb_state_write_local).  ``amps`` may be a
        numpy complex128 array or a raw (pointer, count) pair, e.g. pinned memory."""
        if isinstance(amps, tuple):
            ptr, count = amps
        else:
            a = np.ascontiguousarray(amps, dtype=np.complex128)
            ptr, count = a.ctypes.data, a.size
        capi.check(self.ctx.L.qb_state_write_local(self._h, first, count, C.c_void_p(ptr)))
        return self

    def show(self) -> str:
        """``Show (StateVec n)`` (StateVec.hs:60-68)."""
        n, v = self.n, self.to_host()
        rows = []
        for i, z in enumerate(v):
            bits = "".join("0" if (i // (1 << (n - j - 1))) % 2 == 0 else "1" for j in range(n))
            rows.append("% 6.4f" % z.real + "  + " + "% 6.4f" % z.imag + "i" + "  " + "|" + bits + ">\n")
        return "".join(rows)

    __str__ = show

    # -- in-place primitives (the C ABI, one call each) -----------------------------------
    def apply_1q(self, q: int, m):
        capi.check(self.ctx.L.qb_apply_1q(self._h, q, capi.mat4(m)))
        return self

    def apply_1q_range(self, qlo: int, qhi: int, m):
        capi.check(self.ctx.L.qb_apply_1q_range(self._h, qlo, qhi, capi.mat4(m)))
        return self

    def apply_ctrl_1q(self, ctrls, t: int, m):
        arr = (C.c_int * max(1, len(ctrls)))(*ctrls)
        capi.check(self.ctx.L.qb_apply_ctrl_1q(self._h, arr, len(ctrls), t, capi.mat4(m)))
        return self

    def apply_cnot(self, c: int, t: int):
        capi.check(self.ctx.L.qb_apply_cnot(self._h, c, t))
        return self

    def apply_kq(self, qs, M, ctrls=()):
        k = len(qs)
        a = np.ascontiguousarray(M, dtype=np.complex128).reshape(1 << k, 1 << k)
        qa = (C.c_int * k)(*qs)
        ca = (C.c_int * max(1, len(ctrls)))(*ctrls)
        capi.check(self.ctx.L.qb_apply_kq(self._h, qa, k, a.ctypes.data_as(C.c_void_p), ca, len(ctrls)))
        return self

    def submit(self, ops):
        """Batch submission of an op stream (qb_submit): one boundary crossing."""
        arr = ops if isinstance(ops, C.Array) else capi.pack_ops(ops)
        capi.check(self.ctx.L.qb_submit(self._h, arr, len(arr)))
        return self

    def run_ops(self, ops):
        """Apply an op stream (("U", q, m) | ("CX", c, t) | ("CU", ctrls, t, m) | ("KQ", qs, M[, ctrls]) |
        ("COLLAPSE", q, b) | ("MEASURE", q, r)) one ABI call per op, the way
        the interpreter drives the boundary.  Returns the list of (q, bit, pOne) measured."""
        rec = []
        for op in ops:
            k = op[0]
            if k == "U":
                self.apply_1q(op[1], op[2])
            elif k == "CX":
                self.apply_cnot(op[1], op[2])
            elif k == "CU":
                self.apply_ctrl_1q(list(op[1]), op[2], op[3])
            elif k == "KQ":
                self.apply_kq(list(op[1]), op[2], list(op[3]) if len(op) > 3 else ())
            elif k == "COLLAPSE":
                self.collapse_(op[1], op[2])
            elif k == "MEASURE":
                bit, p = self.measure_qubit_(op[1], op[2])
                rec.append((op[1], bit, p))
            else:
                raise ValueError(k)
        return rec

    def flush(self):
        capi.check(self.ctx.L.qb_flush(self._h))
        return self

    def sumsq(self, q: int):
        s0, s1 = C.c_double(), C.c_double()
        capi.check(self.ctx.L.qb_sumsq(self._h, q, C.byref(s0), C.byref(s1)))
        return s0.value, s1.value

    def collapse_(self, q: int, bit: int):
        capi.check(self.ctx.L.qb_collapse(self._h, q, bit))
        return self

    def measure_qubit_(self, q: int, r: float):
        bit, p = C.c_int(), C.c_double()
        capi.check(self.ctx.L.qb_measure_qubit(self._h, q, r, C.byref(bit), C.byref(p)))
        return bit.value, p.value

    def measure_(self, rs):
        n = self.n
        ra = (C.c_double * n)(*rs)
        ba = (C.c_int * n)()
        capi.check(self.ctx.L.qb_measure_all(self._h, ra, ba))
        return list(ba)

    def scale_(self, z: complex):
        z = complex(z)
        capi.check(self.ctx.L.qb_scale(self._h, capi.QbC64(z.real, z.imag)))
        return self

    def axpy_(self, z: complex, x: "StateVec"):
        z = complex(z)
        capi.check(self.ctx.L.qb_axpy(self._h, capi.QbC64(z.real, z.imag), x._h))
        return self

    def norm2(self) -> float:
        out = C.c_double()
        capi.check(self.ctx.L.qb_norm2(self._h, C.byref(out)))
        return out.value

    # -- VectorSpace / HilbertSpace instances (StateVec.hs:51-58, Algebra.hs:17-36) --------
    def __rmul__(self, z):  # z .: v
        return self.clone().scale_(z)

    def __add__(self, other):  # a +: b
        return self.clone().axpy_(1.0, other)

    def __sub__(self, other):  # a -: b = a +: neg b
        return self.clone().axpy_(-1.0, other)

    def __neg__(self):  # neg
        out = self.clone()
        capi.check(self.ctx.L.qb_neg(out._h))
        return out

    def inner(self, other) -> complex:  # a <.> b (conjugates a)
        out = capi.QbC64()
        capi.check(self.ctx.L.qb_dotc(self._h, other._h, C.byref(out)))
        return complex(out.re, out.im)

    def expect_pauli(self, terms) -> np.ndarray:
        """``realPart (sv <.> (p #> sv))`` for each Pauli string ``p`` of ``terms`` (qb_expect_pauli), in one
        read-only sweep per distinct X mask; the state is not normalised first and keeps its value.
        A term is a string over ``IXYZ`` of length n (character q acts on qubit q) or an
        ``(xmask, zmask)`` pair (bit q = qubit q; X: x only, Z: z only, Y: both).  Returns float64[len(terms)]."""
        n = self.n
        xs, zs = pauli_masks(terms, n)
        out = np.zeros(len(xs), dtype=np.float64)
        P64 = C.POINTER(C.c_uint64)
        capi.check(self.ctx.L.qb_expect_pauli(self._h, xs.ctypes.data_as(P64), zs.ctypes.data_as(P64), len(xs),
                                              out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def pauli_rot_(self, terms, thetas):
        """Apply ``exp(-i theta/2 P)`` for each Pauli string ``P`` of ``terms`` with the angle of ``thetas``, in
        order, in place (qb_apply_pauli_rot).  Terms are spelled as for ``expect_pauli``.  Queued like a gate."""
        xs, zs = pauli_masks(terms, self.n)
        th = np.ascontiguousarray(thetas, dtype=np.float64).reshape(-1)
        if th.size != xs.size:
            raise ValueError(f"{xs.size} Pauli strings but {th.size} angles")
        P64 = C.POINTER(C.c_uint64)
        capi.check(self.ctx.L.qb_apply_pauli_rot(self._h, xs.ctypes.data_as(P64), zs.ctypes.data_as(P64),
                                                 th.ctypes.data_as(C.POINTER(C.c_double)), len(xs)))
        return self

    def norm(self) -> float:  # Algebra.hs:35-36: realPart (a <.> a), the SQUARED norm
        return self.inner(self).real

    def __eq__(self, other):  # StateVec.hs:47-49: norm_2 (a - b) < 1e-6
        if not isinstance(other, StateVec):
            return NotImplemented
        return (self - other).norm2() < 0.000001

    __hash__ = None


def pauli_masks(terms, n: int):
    """Pauli strings (``"XIZY"``, character q = qubit q) or ``(xmask, zmask)`` pairs -> two uint64 arrays."""
    xs, zs = [], []
    for term in terms:
        if isinstance(term, str):
            if len(term) != n or any(ch not in "IXYZ" for ch in term.upper()):
                raise ValueError(f"Pauli string {term!r}: want {n} characters of IXYZ")
            x = sum(1 << q for q, ch in enumerate(term.upper()) if ch in "XY")
            z = sum(1 << q for q, ch in enumerate(term.upper()) if ch in "ZY")
        else:
            x, z = (int(m) for m in term)
        xs.append(x)
        zs.append(z)
    return np.array(xs, dtype=np.uint64), np.array(zs, dtype=np.uint64)


# ---- module-level functions with the reference's names (StateVec.hs:14-25) -----------------
def mkStateVec(n: int, ctx: Context | None = None) -> StateVec:
    """StateVec.hs:78-85: |0...0>."""
    return StateVec.create(n, True, ctx)


def zero(n: int, ctx: Context | None = None) -> StateVec:
    """StateVec.hs:52."""
    return StateVec.create(n, False, ctx)


def mkQubit(ctx: Context | None = None) -> StateVec:
    """StateVec.hs:88-89."""
    return StateVec.create(1, True, ctx)


def dimension(sv: StateVec) -> int:
    """StateVec.hs:74-75."""
    return sv.n


def normalize(sv: StateVec) -> StateVec:
    """StateVec.hs:91-92 (pure)."""
    out = sv.clone()
    capi.check(out.ctx.L.qb_normalize(out._h))
    return out


def tensor(a: StateVec, b: StateVec) -> StateVec:
    """StateVec.hs:98-100."""
    h = C.c_void_p()
    capi.check(a.ctx.L.qb_tensor(a._h, b._h, C.byref(h)))
    return StateVec(h, a.ctx)


def collapse(i: int, b: int, sv: StateVec) -> StateVec:
    """StateVec.hs:104-114 (pure)."""
    return sv.clone().collapse_(i, b)


def measureQubit(i: int, sv: StateVec, r: float) -> int:
    """StateVec.hs:118-129 in its StateT form: mutates ``sv``; ``r`` is the uniform draw the
    Haskell side takes from MonadRandom."""
    return sv.measure_qubit_(i, r)[0]


def measure(sv: StateVec, rs) -> list:
    """StateVec.hs:133-137."""
    return sv.measure_(rs)


def expectPauli(terms, sv: StateVec) -> np.ndarray:
    """``[realPart (sv <.> (p #> sv)) | p <- terms]`` without building any ``p #> sv`` (see StateVec.expect_pauli)."""
    return sv.expect_pauli(terms)


def pauliRotate(terms, thetas, sv: StateVec) -> StateVec:
    """``exp(-i theta_k/2 P_k) ... exp(-i theta_0/2 P_0) #> sv`` as a new value; ``sv`` keeps its own
    (a lazy clone rotated in place, see StateVec.pauli_rot_)."""
    return sv.clone().pauli_rot_(terms, thetas)
