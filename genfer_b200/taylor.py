"""Host-side mirror of the reference's ``TaylorPoly<F64>`` / ``TaylorExpansion<F64>`` operator surface
over the C ABI of ``libgenfer_taylor.so``.

Names, argument meaning and error behaviour follow /root/reference/src/multivariate_taylor.rs and
src/univariate_taylor.rs (where the reference panics, :class:`TaylorPanic` is raised), so parity tests
read like the reference's own unit tests.  All arithmetic happens on the GPU; this module only moves
handles around.  There is no CPU fallback: creating a :class:`Context` without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import UNBOUNDED


class TaylorError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"{_lib.STATUS.get(status, status)}: {msg}")
        self.status = status


class TaylorPanic(TaylorError):
    """GTP_ERR_INDEX: the reference's assert!/panic (bad variable, order or index)."""


def _u64(xs) -> C.Array:
    xs = [int(x) for x in xs]
    return (C.c_uint64 * max(len(xs), 1))(*xs)


class Context:
    """One CUDA device + one stream (gtp_ctx).  ``stream`` may be a raw cudaStream_t (int)."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.gtp_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != 0:
            raise TaylorError(rc, "gtp_ctx_create failed (no CUDA device? there is no CPU fallback)")
        self.h = h
        self.device = device

    @classmethod
    def create_group(cls, device: int, rank: int, world: int, unique_id: bytes, stream: Optional[int] = None) -> "Context":
        """Group context (gtp_ctx_create_group): one NCCL communicator on the context's stream.  `unique_id` are the 128
        bytes of :func:`nccl_unique_id` from rank 0, shipped to every rank by the caller (bench.py: torch.distributed)."""
        self = cls.__new__(cls)
        self.lib = _lib.load()
        assert len(unique_id) == 128
        h = C.c_void_p()
        buf = C.create_string_buffer(bytes(unique_id), 128)
        rc = self.lib.gtp_ctx_create_group(device, C.c_void_p(stream) if stream else None, rank, world, buf, C.byref(h))
        if rc != 0:
            raise TaylorError(rc, "gtp_ctx_create_group failed (no CUDA device / NCCL?)")
        self.h = h
        self.device = device
        return self

    def group_info(self):
        """(rank, world, partitioned products so far, replications so far)"""
        r, w = C.c_int(), C.c_int()
        pp, g = C.c_uint64(), C.c_uint64()
        self.check(self.lib.gtp_ctx_group_info(self.h, C.byref(r), C.byref(w), C.byref(pp), C.byref(g)))
        return r.value, w.value, int(pp.value), int(g.value)

    def set_partition_threshold(self, coefficients: int):
        self.check(self.lib.gtp_ctx_set_partition_threshold(self.h, int(coefficients)))

    def close(self):
        if getattr(self, "h", None):
            self.lib.gtp_ctx_destroy(self.h)
            self.h = None

    def check(self, rc: int):
        if rc != 0:
            msg = self.lib.gtp_last_error(self.h).decode()
            raise (TaylorPanic if rc == 1 else TaylorError)(rc, msg)

    def synchronize(self):
        self.check(self.lib.gtp_ctx_synchronize(self.h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.gtp_ctx_launch_count(self.h))

    @property
    def stream(self) -> int:
        return int(self.lib.gtp_ctx_stream(self.h) or 0)

    def set_fast_mul(self, enabled):
        """0/False: reference-order kernel only; 1/True: fastest applicable; 2: prefer the generic blocked kernel."""
        self.check(self.lib.gtp_ctx_set_fast_mul(self.h, int(enabled)))

    def fp64_peak_probe(self, kind: int, iters: int = 4096):
        fl, ms = C.c_double(), C.c_double()
        self.check(self.lib.gtp_fp64_peak_probe(self.h, kind, iters, C.byref(fl), C.byref(ms)))
        return fl.value, ms.value

    # -- raw product (bench / sharding) -------------------------------------------------
    def mul_rows_raw(self, xshape, x_ptr: int, yshape, y_ptr: int, rshape, row_begin: int, row_step: int,
                     row_count: int, out_ptr: int):
        self.check(self.lib.gtp_mul_rows_raw(self.h, len(rshape), _u64(xshape), C.c_void_p(x_ptr), _u64(yshape),
                                             C.c_void_p(y_ptr), _u64(rshape), row_begin, row_step, row_count,
                                             C.c_void_p(out_ptr)))

    def mul_rowlist_raw(self, xshape, x_ptr: int, yshape, y_ptr: int, rshape, rows: Sequence[int], out_ptr: int):
        self.check(self.lib.gtp_mul_rowlist_raw(self.h, len(rshape), _u64(xshape), C.c_void_p(x_ptr), _u64(yshape),
                                                C.c_void_p(y_ptr), _u64(rshape), _u64(rows), len(rows),
                                                C.c_void_p(out_ptr)))

    def mul_kernel_kind(self, xshape, yshape, rshape) -> int:
        return int(self.lib.gtp_mul_kernel_kind(self.h, len(rshape), _u64(xshape), _u64(yshape), _u64(rshape)))


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    rc = _lib.load().gtp_nccl_unique_id(buf)
    if rc != 0:
        raise TaylorError(rc, "gtp_nccl_unique_id failed (NCCL not loadable?)")
    return buf.raw


def partition_rows(n_rows: int, world: int, rank: int):
    """Folded-cyclic leading-axis rows of `rank` (gtp_partition_rows; integer work, no device needed)."""
    out = (C.c_uint64 * max(n_rows, 1))()
    n = int(_lib.load().gtp_partition_rows(n_rows, world, rank, out))
    return [int(out[i]) for i in range(n)]


def partition_block(n_slices: int, world: int, rank: int):
    lo, hi, b = C.c_uint64(), C.c_uint64(), C.c_uint64()
    _lib.load().gtp_partition_block(n_slices, world, rank, C.byref(lo), C.byref(hi), C.byref(b))
    return int(lo.value), int(hi.value), int(b.value)


def mul_macs(xshape, yshape, rshape) -> float:
    return float(_lib.load().gtp_mul_macs(len(rshape), _u64(xshape), _u64(yshape), _u64(rshape)))


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


def set_default_context(ctx: Optional[Context]):
    global _default_ctx
    _default_ctx = ctx


class TaylorPoly:
    """Device-resident TaylorPoly<F64> (multivariate_taylor.rs:13-19)."""

    __slots__ = ("ctx", "_h")

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self._h = handle

    def __del__(self):
        try:
            if self._h and self.ctx.h:
                self.ctx.lib.gtp_free(self.ctx.h, self._h)
        except Exception:
            pass

    # -- plumbing -------------------------------------------------------------------------
    @classmethod
    def _make(cls, ctx: Context, fn: str, *args) -> "TaylorPoly":
        h = C.c_void_p()
        ctx.check(getattr(ctx.lib, fn)(ctx.h, *args, C.byref(h)))
        return cls(ctx, h)

    def _op(self, fn: str, *args) -> "TaylorPoly":
        return self._make(self.ctx, fn, self._h, *args)

    # -- constructors (:33-46, :208-259, :626-656) -----------------------------------------
    @classmethod
    def new(cls, coeffs, degrees_p1: Sequence[int], ctx: Optional[Context] = None) -> "TaylorPoly":
        ctx = ctx or default_context()
        a = np.array(coeffs, dtype=np.float64, order="C")
        assert a.ndim == len(degrees_p1), "coeffs.ndim() != degrees_p1.len()"
        return cls._make(ctx, "gtp_from_host", a.ndim, _u64(a.shape), _u64(degrees_p1),
                         a.ctypes.data_as(_lib.f64p))

    @classmethod
    def from_host_ptr(cls, ptr: int, shape: Sequence[int], degrees_p1: Sequence[int],
                      ctx: Optional[Context] = None) -> "TaylorPoly":
        """Upload prod(shape) doubles from a host address (e.g. a pinned staging buffer) without a numpy copy."""
        ctx = ctx or default_context()
        return cls._make(ctx, "gtp_from_host", len(shape), _u64(shape), _u64(degrees_p1),
                         C.cast(C.c_void_p(ptr), _lib.f64p))

    @classmethod
    def from_host_block_ptr(cls, ptr: int, shape: Sequence[int], degrees_p1: Sequence[int], ctx: Context) -> "TaylorPoly":
        """Block-sharded upload (gtp_from_host_block): `ptr` holds this rank's leading-axis slices of the FULL `shape`."""
        return cls._make(ctx, "gtp_from_host_block", len(shape), _u64(shape), _u64(degrees_p1), C.c_void_p(ptr))

    @classmethod
    def from_device_block(cls, ptr: int, shape: Sequence[int], degrees_p1: Sequence[int], ctx: Context) -> "TaylorPoly":
        return cls._make(ctx, "gtp_from_device_block", len(shape), _u64(shape), _u64(degrees_p1), C.c_void_p(ptr))

    def is_distributed(self) -> bool:
        return bool(self.ctx.lib.gtp_is_distributed(self._h))

    def replicate(self) -> "TaylorPoly":
        self.ctx.check(self.ctx.lib.gtp_replicate(self.ctx.h, self._h))
        return self

    def local_rows(self):
        n0 = self.array_shape()[0] if self.num_vars() else 1
        out = (C.c_uint64 * max(n0, 1))()
        n = int(self.ctx.lib.gtp_local_rows(self._h, out))
        return [int(out[i]) for i in range(n)]

    def to_host_local_ptr(self, ptr: int) -> None:
        """D2H of this rank's rows of a row-sharded result (no collective; synchronises)."""
        self.ctx.check(self.ctx.lib.gtp_to_host_local(self.ctx.h, self._h, C.c_void_p(ptr)))

    def to_host_ptr(self, ptr: int) -> None:
        """Copy the stored coefficients to a host address (synchronises)."""
        self.ctx.check(self.ctx.lib.gtp_to_host(self.ctx.h, self._h, C.c_void_p(ptr)))

    @classmethod
    def from_coeffs(cls, coeffs, ctx: Optional[Context] = None) -> "TaylorPoly":
        a = np.asarray(coeffs, dtype=np.float64)
        return cls.new(a, a.shape, ctx)

    @classmethod
    def from_device(cls, ptr: int, shape: Sequence[int], degrees_p1: Sequence[int],
                    ctx: Optional[Context] = None) -> "TaylorPoly":
        """Wrap an existing device buffer (e.g. a torch tensor's data_ptr) without copying."""
        ctx = ctx or default_context()
        return cls._make(ctx, "gtp_from_device", len(shape), _u64(shape), _u64(degrees_p1), C.c_void_p(ptr))

    @classmethod
    def from_scalar(cls, x: float, ctx: Optional[Context] = None) -> "TaylorPoly":
        return cls._make(ctx or default_context(), "gtp_from_scalar", float(x))

    @classmethod
    def zero(cls, ctx=None): return cls.from_scalar(0.0, ctx)
    @classmethod
    def one(cls, ctx=None): return cls.from_scalar(1.0, ctx)
    @classmethod
    def from_u32(cls, c: int, ctx=None): return cls.from_scalar(float(c), ctx)

    @classmethod
    def zero_with(cls, degrees_p1: Sequence[int], ctx=None) -> "TaylorPoly":
        return cls._make(ctx or default_context(), "gtp_zero_with", len(degrees_p1), _u64(degrees_p1))

    @classmethod
    def var(cls, v: int, x: float, length: int, ctx=None) -> "TaylorPoly":
        return cls._make(ctx or default_context(), "gtp_var", v, float(x), length)

    @classmethod
    def var_at_zero(cls, v: int, length: int, ctx=None) -> "TaylorPoly":
        return cls._make(ctx or default_context(), "gtp_var_at_zero", v, length)

    @classmethod
    def var_with_degrees_p1(cls, v: int, x: float, degrees_p1: Sequence[int], ctx=None) -> "TaylorPoly":
        return cls._make(ctx or default_context(), "gtp_var_with_degrees_p1", v, float(x), len(degrees_p1),
                         _u64(degrees_p1))

    # -- accessors ---------------------------------------------------------------------------
    def num_vars(self) -> int:
        return int(self.ctx.lib.gtp_ndim(self._h))

    def array_shape(self) -> tuple:
        n = self.num_vars()
        out = (C.c_uint64 * max(n, 1))()
        self.ctx.lib.gtp_shape(self._h, out)
        return tuple(int(out[i]) for i in range(n))

    def shape(self) -> tuple:
        """`shape()` of the reference returns degrees_p1 (:53-56)."""
        n = self.num_vars()
        out = (C.c_uint64 * max(n, 1))()
        self.ctx.lib.gtp_degrees_p1(self._h, out)
        return tuple(int(out[i]) for i in range(n))

    degrees_p1 = property(lambda self: self.shape())

    def len_of(self, v: int) -> int:
        d = self.shape()
        return d[v] if v < len(d) else UNBOUNDED

    def array(self) -> np.ndarray:
        a = np.empty(self.array_shape(), dtype=np.float64)
        self.ctx.check(self.ctx.lib.gtp_to_host(self.ctx.h, self._h, a.ctypes.data_as(C.c_void_p)))
        return a

    def device_ptr(self) -> int:
        p = C.c_void_p()
        self.ctx.check(self.ctx.lib.gtp_device_ptr(self.ctx.h, self._h, C.byref(p)))
        return int(p.value or 0)

    def clone(self) -> "TaylorPoly":
        return self._op("gtp_clone")

    def is_constant(self) -> bool:
        return int(self.ctx.lib.gtp_len(self._h)) == 1

    def _flag(self, fn: str) -> bool:
        out = C.c_int()
        self.ctx.check(getattr(self.ctx.lib, fn)(self.ctx.h, self._h, C.byref(out)))
        return bool(out.value)

    def is_zero(self) -> bool: return self._flag("gtp_is_zero")
    def is_one(self) -> bool: return self._flag("gtp_is_one")

    def _scalar(self, fn: str, *args) -> float:
        out = C.c_double()
        self.ctx.check(getattr(self.ctx.lib, fn)(self.ctx.h, self._h, *args, C.byref(out)))
        return out.value

    def constant_term(self) -> float: return self._scalar("gtp_constant_term")
    def evaluate_all_one(self) -> float: return self._scalar("gtp_evaluate_all_one")

    def coefficient(self, index: Sequence[int]) -> float:
        return self._scalar("gtp_coefficient", _u64(index), len(index))

    def gather_axis(self, v: int, count: int) -> np.ndarray:
        """coefficient([0,..,i (axis v),..,0]) for i < count as one gather + one D2H copy."""
        out = np.empty(count, dtype=np.float64)
        self.ctx.check(self.ctx.lib.gtp_gather_axis(self.ctx.h, self._h, v, count, out.ctypes.data_as(_lib.f64p)))
        return out

    def extract_constant(self) -> Optional[float]:
        flag, val = C.c_int(), C.c_double()
        self.ctx.check(self.ctx.lib.gtp_extract_constant(self.ctx.h, self._h, C.byref(flag), C.byref(val)))
        return val.value if flag.value else None

    def extract_linear(self) -> Optional[tuple]:
        flag, c, m, v = C.c_int(), C.c_double(), C.c_double(), C.c_uint64()
        self.ctx.check(self.ctx.lib.gtp_extract_linear(self.ctx.h, self._h, C.byref(flag), C.byref(c), C.byref(m),
                                                       C.byref(v)))
        return (c.value, m.value, int(v.value)) if flag.value else None

    # -- operators (impl Add/Sub/Mul/Div/Neg) -----------------------------------------------
    def _coerce(self, o) -> "TaylorPoly":
        return o if isinstance(o, TaylorPoly) else TaylorPoly.from_scalar(float(o), self.ctx)

    def _binop(self, fn: str, o) -> "TaylorPoly":
        other = self._coerce(o)          # keep a coerced scalar alive across the call (its __del__ frees the handle)
        return self._op(fn, other._h)

    def __add__(self, o): return self._binop("gtp_add", o)
    def __sub__(self, o): return self._binop("gtp_sub", o)
    def __mul__(self, o): return self._binop("gtp_mul", o)
    def __truediv__(self, o): return self._binop("gtp_div", o)
    def __neg__(self): return self._op("gtp_neg")

    def __eq__(self, other) -> bool:  # derive(PartialEq) (:10)
        out = C.c_int()
        self.ctx.check(self.ctx.lib.gtp_eq(self.ctx.h, self._h, other._h, C.byref(out)))
        return bool(out.value)

    def __ne__(self, other) -> bool:
        return not self.__eq__(other)

    __hash__ = None

    def exp(self): return self._op("gtp_exp")
    def log(self): return self._op("gtp_log")
    def pow(self, e: int): return self._op("gtp_pow", e)
    def derivative(self, v: int, n: int): return self._op("gtp_derivative", v, n)
    def taylor_expansion_of_coeff(self, v: int, n: int): return self._op("gtp_taylor_expansion_of_coeff", v, n)
    def shift_down(self, v: int, n: int): return self._op("gtp_shift_down", v, n)
    def coefficients_of_term(self, v: int, order: int): return self._op("gtp_coefficients_of_term", v, order)
    def taylor_polynomial(self, v: int, order: int): return self._op("gtp_taylor_polynomial", v, order)
    def taylor_polynomial_terms(self, v: int, orders: Sequence[int]):
        return self._op("gtp_taylor_polynomial_terms", v, _u64(orders), len(orders))
    def subst_var(self, v: int, subst: "TaylorPoly"): return self._op("gtp_subst_var", v, subst._h)
    def truncate_to_degree_p1(self, d: int): return self._op("gtp_truncate_to_degree_p1", d)
    def remove_last_variable(self): return self._op("gtp_remove_last_variable")
    def extend_to_dim(self, ndim: int, d: int): return self._op("gtp_extend_to_dim", ndim, d)
    def extend(self, new_size: Sequence[int]): return self._op("gtp_extend", len(new_size), _u64(new_size))

    def __repr__(self) -> str:
        if not self._h or not self.ctx.h:     # context closed: do not call into the library from a traceback formatter
            return "TaylorPoly(<released>)"
        return f"TaylorPoly({list(self.shape())}, {self.array().tolist()})"


def taylor(coeffs, degrees_p1: Optional[Sequence[int]] = None, ctx: Optional[Context] = None) -> TaylorPoly:
    """The reference's `taylor!` test macro (:659-692)."""
    if degrees_p1 is None:
        return TaylorPoly.from_coeffs(coeffs, ctx)
    return TaylorPoly.new(coeffs, degrees_p1, ctx)


class TaylorExpansion:
    """Device-resident univariate TaylorExpansion<F64> (univariate_taylor.rs:9-13)."""

    __slots__ = ("ctx", "_h")

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self._h = handle

    def __del__(self):
        try:
            if self._h and self.ctx.h:
                self.ctx.lib.gtu_free(self.ctx.h, self._h)
        except Exception:
            pass

    @classmethod
    def _make(cls, ctx, fn, *args):
        h = C.c_void_p()
        ctx.check(getattr(ctx.lib, fn)(ctx.h, *args, C.byref(h)))
        return cls(ctx, h)

    def _op(self, fn, *args): return self._make(self.ctx, fn, self._h, *args)

    @classmethod
    def constant(cls, x: float, ctx=None): return cls._make(ctx or default_context(), "gtu_constant", float(x))
    @classmethod
    def zero(cls, ctx=None): return cls.constant(0.0, ctx)
    @classmethod
    def one(cls, ctx=None): return cls.constant(1.0, ctx)
    @classmethod
    def from_coefficients(cls, xs, ctx=None):
        a = np.ascontiguousarray(xs, dtype=np.float64)
        return cls._make(ctx or default_context(), "gtu_from_coefficients", a.ctypes.data_as(_lib.f64p), a.shape[0])
    @classmethod
    def var(cls, x: float, order: int, ctx=None): return cls._make(ctx or default_context(), "gtu_var", float(x), order)

    def is_const(self) -> bool: return bool(self.ctx.lib.gtu_is_constant(self._h))
    def order(self) -> int: return int(self.ctx.lib.gtu_order(self._h))

    def coeffs(self) -> np.ndarray:
        n = 1 if self.is_const() else self.order()
        a = np.empty(n, dtype=np.float64)
        self.ctx.check(self.ctx.lib.gtu_to_host(self.ctx.h, self._h, a.ctypes.data_as(_lib.f64p)))
        return a

    def coeff(self, order: int) -> float:
        out = C.c_double()
        self.ctx.check(self.ctx.lib.gtu_coeff(self.ctx.h, self._h, order, C.byref(out)))
        return out.value

    def derivative(self, order: int) -> float:
        out = C.c_double()
        self.ctx.check(self.ctx.lib.gtu_derivative(self.ctx.h, self._h, order, C.byref(out)))
        return out.value

    def __add__(self, o): return self._op("gtu_add", o._h)
    def __sub__(self, o): return self._op("gtu_sub", o._h)
    def __mul__(self, o): return self._op("gtu_mul", o._h)
    def __truediv__(self, o): return self._op("gtu_div", o._h)
    def __neg__(self): return self._op("gtu_neg")
    def exp(self): return self._op("gtu_exp")
    def log(self): return self._op("gtu_log")
    def pow(self, e: int): return self._op("gtu_pow", e)
    def subst(self, s): return self._op("gtu_subst", s._h)
    def taylor_expansion_of_coeff(self, n: int): return self._op("gtu_taylor_expansion_of_coeff", n)

    def __eq__(self, o) -> bool:
        out = C.c_int()
        self.ctx.check(self.ctx.lib.gtu_eq(self.ctx.h, self._h, o._h, C.byref(out)))
        return bool(out.value)

    def __ne__(self, o): return not self.__eq__(o)
    __hash__ = None

    def __repr__(self):
        if not self._h or not self.ctx.h:
            return "TaylorExpansion(<released>)"
        return f"TaylorExpansion({'Constant' if self.is_const() else 'Polynomial'}, {self.coeffs().tolist()})"


GTU_ADD, GTU_SUB, GTU_MUL, GTU_DIV, GTU_NEG, GTU_EXP, GTU_LOG, GTU_POW, GTU_MAX = range(9)


class UniProgram:
    """A DAG of univariate TaylorExpansion<F64> ops recorded on the host and run by one kernel launch (gtu_program_*).

    Each op means exactly the TaylorExpansion operator of the same name, with the same bits; its errors are raised when it
    is recorded.  ``run(*slots)`` runs every recorded op and returns the slots' coefficients as numpy arrays (one element
    for a Constant)."""

    def __init__(self, ctx: Optional[Context] = None):
        self.ctx = ctx or default_context()
        self._h = C.c_void_p()
        self.ctx.check(self.ctx.lib.gtu_program_create(self.ctx.h, C.byref(self._h)))

    def __del__(self):
        try:
            if self._h and self.ctx.h:
                self.ctx.lib.gtu_program_free(self.ctx.h, self._h)
        except Exception:
            pass

    def _slot(self, fn: str, *args) -> "UniSlot":
        s = C.c_uint32()
        self.ctx.check(getattr(self.ctx.lib, fn)(self.ctx.h, self._h, *args, C.byref(s)))
        return UniSlot(self, s.value)

    def constant(self, x: float) -> "UniSlot": return self._slot("gtu_program_constant", float(x))
    def var(self, x: float, order: int) -> "UniSlot": return self._slot("gtu_program_var", float(x), order)

    def from_coefficients(self, xs) -> "UniSlot":
        a = np.ascontiguousarray(xs, dtype=np.float64)
        return self._slot("gtu_program_from_coefficients", a.ctypes.data_as(_lib.f64p), a.shape[0])

    def op(self, op: int, a: "UniSlot", b: Optional["UniSlot"] = None, exp: int = 0) -> "UniSlot":
        for s in (a, b):
            if s is not None and s.program is not self:
                raise ValueError("slot of another program")
        return self._slot("gtu_program_op", op, a.index, b.index if b is not None else 0, exp)

    def run(self, *slots: "UniSlot"):
        for s in slots:
            if s.program is not self:
                raise ValueError("slot of another program")
        lens = [1 if s.is_const() else s.order() for s in slots]
        out = np.empty(max(sum(lens), 1), dtype=np.float64)
        idx = (C.c_uint32 * max(len(slots), 1))(*[s.index for s in slots])
        self.ctx.check(self.ctx.lib.gtu_program_run(self.ctx.h, self._h, idx, len(slots), out.ctypes.data_as(_lib.f64p)))
        return np.split(out[:sum(lens)], np.cumsum(lens)[:-1]) if slots else []


class UniSlot:
    """A value of a :class:`UniProgram`: supports ``+ - * /``, unary ``-``, ``exp``, ``log``, ``pow`` and ``max``."""

    __slots__ = ("program", "index")

    def __init__(self, program: UniProgram, index: int):
        self.program = program
        self.index = index

    def _info(self):
        c, n = C.c_int(), C.c_uint64()
        self.program.ctx.check(self.program.ctx.lib.gtu_program_slot(self.program._h, self.index, C.byref(c), C.byref(n)))
        return bool(c.value), int(n.value)

    def is_const(self) -> bool: return self._info()[0]
    def order(self) -> int: return self._info()[1]

    def __add__(self, o): return self.program.op(GTU_ADD, self, o)
    def __sub__(self, o): return self.program.op(GTU_SUB, self, o)
    def __mul__(self, o): return self.program.op(GTU_MUL, self, o)
    def __truediv__(self, o): return self.program.op(GTU_DIV, self, o)
    def __neg__(self): return self.program.op(GTU_NEG, self)
    def exp(self): return self.program.op(GTU_EXP, self)
    def log(self): return self.program.op(GTU_LOG, self)
    def pow(self, e: int): return self.program.op(GTU_POW, self, exp=e)
    def max(self, o): return self.program.op(GTU_MAX, self, o)
