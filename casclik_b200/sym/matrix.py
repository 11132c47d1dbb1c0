"""Dense matrices of scalar DAG nodes with the slice of the CasADi Python surface that CASCLIK and
its notebooks use (list in SURVEY.md §8b "Expression language the user hands in").

`MX`, `SX` and `DM` are thin subclasses of one dense container: MX/SX hold arbitrary nodes, DM holds
constants only.  The names exist so user code written against `import casadi as cs` keeps working
with `from casclik_b200 import cs`; the semantics mirrored are the documented CasADi ones
(SURVEY.md Appendix B), the implementation is independent.
"""
from __future__ import annotations

import numbers
from typing import List, Sequence

import numpy as np

from . import dag
from .dag import Node

inf = float("inf")
pi = float(np.pi)


def _is_scalar_number(x):
    return isinstance(x, (numbers.Real, np.floating, np.integer, np.bool_))


class GenericMatrixCommon(object):
    """Base class of MX / SX / DM (name kept for `isinstance(w, cs.GenericMatrixCommon)`,
    reference casclik/controllers/reactive_qp.py:69)."""

    __array_priority__ = 1.0e6
    __array_ufunc__ = None
    __hash__ = object.__hash__
    _rank = 0  # DM=0 < SX=1 < MX=2 : result class of mixed arithmetic

    # ---- construction ------------------------------------------------------------------------
    def __init__(self, *args):
        if len(args) == 0:
            self._a = np.empty((0, 0), dtype=object)
        elif len(args) == 1:
            self._a = _to_nodes(args[0])
        elif len(args) == 2 and all(isinstance(k, (int, np.integer)) for k in args):
            self._a = _filled(int(args[0]), int(args[1]), dag.ZERO)
        else:
            raise TypeError("unsupported constructor arguments for %s" % type(self).__name__)
        if type(self) is DM and not self.is_constant():
            raise TypeError("DM can only hold numeric values")

    @classmethod
    def _wrap(cls, a: np.ndarray):
        obj = cls.__new__(cls)
        obj._a = a
        return obj

    @classmethod
    def sym(cls, name, n=1, m=1):
        if cls is DM:
            raise TypeError("DM has no symbols")
        if isinstance(n, (tuple, list)):
            n, m = n
        a = np.empty((n, m), dtype=object)
        scalar = (n == 1 and m == 1)
        for j in range(m):
            for i in range(n):
                a[i, j] = dag.symbol(name if scalar else "%s_%d" % (name, i + j * n))
        return cls._wrap(a)

    @classmethod
    def _shape_args(cls, n, m):
        if isinstance(n, (tuple, list)):
            n, m = n
        return int(n), int(m)

    @classmethod
    def zeros(cls, n=1, m=1):
        n, m = cls._shape_args(n, m)
        return cls._wrap(_filled(n, m, dag.ZERO))

    @classmethod
    def ones(cls, n=1, m=1):
        n, m = cls._shape_args(n, m)
        return cls._wrap(_filled(n, m, dag.ONE))

    @classmethod
    def eye(cls, n):
        a = _filled(n, n, dag.ZERO)
        for i in range(n):
            a[i, i] = dag.ONE
        return cls._wrap(a)

    @classmethod
    def inf(cls, n=1, m=1):
        n, m = cls._shape_args(n, m)
        return cls._wrap(_filled(n, m, dag.const(inf)))

    # ---- shape -------------------------------------------------------------------------------
    def size(self, axis=None):
        if axis is None:
            return (self._a.shape[0], self._a.shape[1])
        return self._a.shape[axis - 1]

    def size1(self):
        return self._a.shape[0]

    def size2(self):
        return self._a.shape[1]

    @property
    def shape(self):
        return (self._a.shape[0], self._a.shape[1])

    def numel(self):
        return self._a.size

    def rows(self):
        return self._a.shape[0]

    def columns(self):
        return self._a.shape[1]

    def __len__(self):
        return self._a.shape[0]

    def nnz(self):
        """Structural non-zeros: entries that are not the literal constant 0."""
        return sum(1 for n in self._a.flat if n is not dag.ZERO)

    def sparsity(self):
        return Sparsity(self._a.shape, [[n is not dag.ZERO for n in row] for row in self._a])

    def is_scalar(self):
        return self._a.shape == (1, 1)

    def is_vector(self):
        return 1 in self._a.shape

    def is_column(self):
        return self._a.shape[1] == 1

    def is_empty(self):
        return self._a.size == 0

    def is_constant(self):
        return all(n.is_const for n in self._a.flat)

    def is_symbolic(self):
        """True iff every entry is a pure symbol (CasADi: `is_symbolic`)."""
        return self._a.size > 0 and all(n.is_sym for n in self._a.flat)

    def is_valid_input(self):
        return self.is_symbolic()

    def is_zero(self):
        return all(n is dag.ZERO for n in self._a.flat)

    def name(self):
        if self._a.shape == (1, 1) and self._a[0, 0].is_sym:
            return self._a[0, 0].name
        if self.is_symbolic():
            return self._a.flat[0].name.rsplit("_", 1)[0]
        raise RuntimeError("name(): not a symbol")

    def nodes(self) -> List[Node]:
        """Entries in column-major order (CasADi's storage order)."""
        return list(self._a.flatten(order="F"))

    # ---- numeric views -----------------------------------------------------------------------
    def toarray(self, simplify=False):
        if not self.is_constant():
            raise RuntimeError("toarray(): expression is not constant")
        out = np.array([[n.val for n in row] for row in self._a], dtype=np.float64)
        out = out.reshape(self._a.shape)
        if simplify:
            if out.shape == (1, 1):
                return float(out[0, 0])
            if 1 in out.shape:
                return out.reshape(-1)
        return out

    def full(self):
        return self.toarray()

    def __array__(self, dtype=None, copy=None):
        if self.is_constant():
            out = self.toarray()
            if out.shape == (1, 1):
                # a numeric scalar acts as a 0-d array, so that NumPy accepts it as an element:
                # `y_sim[i, :] = [fcos(t), fsine(t), 0]` with DM-valued Function results
                # (ur5_input_experiment.ipynb cell 16).  toarray() / full() stay 2-D.
                out = out.reshape(())
            return out if dtype is None else out.astype(dtype)
        return self._a

    def __float__(self):
        if self._a.shape != (1, 1) or not self._a[0, 0].is_const:
            raise TypeError("only a constant 1x1 matrix converts to float")
        return float(self._a[0, 0].val)

    def __int__(self):
        return int(float(self))

    def __bool__(self):
        if self._a.shape == (1, 1) and self._a[0, 0].is_const:
            return self._a[0, 0].val != 0.0
        raise TypeError("truth value of a symbolic / non-scalar matrix is undefined")

    __nonzero__ = __bool__

    def __repr__(self):
        r, c = self._a.shape
        if r * c <= 12:
            body = "[" + ", ".join("[" + ", ".join(repr(n) for n in row) + "]" for row in self._a) + "]"
            if len(body) > 400:
                body = body[:400] + "..."
        else:
            body = "..."
        return "%s(%dx%d %s)" % (type(self).__name__, r, c, body)

    def __str__(self):
        """Constant matrices print like CasADi's DM ("1.0192", "[1, 2, 3]", "[[1, 0], \n [0, 1]]")."""
        if not self.is_constant() or self._a.size == 0:
            return repr(self)
        fmt = lambda n: "%g" % n.val  # noqa: E731
        r, c = self._a.shape
        if (r, c) == (1, 1):
            return fmt(self._a[0, 0])
        if c == 1:
            return "[" + ", ".join(fmt(n) for n in self._a[:, 0]) + "]"
        return "[" + ", \n ".join("[" + ", ".join(fmt(n) for n in row) + "]" for row in self._a) + "]"

    # ---- indexing ----------------------------------------------------------------------------
    def _norm_index(self, key):
        r, c = self._a.shape
        if isinstance(key, tuple):
            if len(key) != 2:
                raise IndexError("matrices are two-dimensional")
            return _axis_index(key[0], r), _axis_index(key[1], c), False
        return _axis_index(key, r * c), None, True

    def __getitem__(self, key):
        if isinstance(key, GenericMatrixCommon):
            key = [int(v) for v in np.asarray(key.toarray()).reshape(-1)]
        i, j, linear = self._norm_index(key)
        if linear:
            flat = self._a.flatten(order="F")
            sub = flat[i].reshape(-1, 1)
        else:
            sub = self._a[np.ix_(i, j)]
        return type(self)._wrap(np.array(sub, dtype=object, copy=True))

    def __setitem__(self, key, value):
        val = _to_nodes(value)
        if type(self) is DM and not all(n.is_const for n in val.flat):
            raise TypeError("cannot assign a symbolic value into a DM")
        i, j, linear = self._norm_index(key)
        if linear:
            r = self._a.shape[0]
            tgt = [(k % r, k // r) for k in i]
            src = _broadcast_to(val, (len(i), 1)).reshape(-1)
            for (a, b), s in zip(tgt, src):
                self._a[a, b] = s
        else:
            src = _broadcast_to(val, (len(i), len(j)))
            for p, a in enumerate(i):
                for q, b in enumerate(j):
                    self._a[a, b] = src[p, q]

    def __iter__(self):
        raise TypeError("%s is not iterable (use indexing)" % type(self).__name__)

    # ---- arithmetic --------------------------------------------------------------------------
    @property
    def T(self):
        return type(self)._wrap(np.array(self._a.T, dtype=object, copy=True))

    def __neg__(self):
        return _map1(dag.neg, self)

    def __pos__(self):
        return self

    def __abs__(self):
        return _map1(dag.fabs, self)

    def __add__(self, o): return _map2(dag.add, self, o)
    def __radd__(self, o): return _map2(dag.add, o, self)
    def __sub__(self, o): return _map2(dag.sub, self, o)
    def __rsub__(self, o): return _map2(dag.sub, o, self)
    def __mul__(self, o): return _map2(dag.mul, self, o)
    def __rmul__(self, o): return _map2(dag.mul, o, self)
    def __truediv__(self, o): return _map2(dag.div, self, o)
    def __rtruediv__(self, o): return _map2(dag.div, o, self)
    __div__ = __truediv__
    __rdiv__ = __rtruediv__
    def __pow__(self, o): return _map2(dag.pow_, self, o)
    def __rpow__(self, o): return _map2(dag.pow_, o, self)
    def __matmul__(self, o): return mtimes(self, o)
    def __rmatmul__(self, o): return mtimes(o, self)
    def __lt__(self, o): return _map2(dag.lt, self, o)
    def __le__(self, o): return _map2(dag.le, self, o)
    def __gt__(self, o): return _map2(dag.lt, o, self)
    def __ge__(self, o): return _map2(dag.le, o, self)
    def __eq__(self, o): return _map2(dag.eq, self, o)
    def __ne__(self, o): return _map2(dag.ne, self, o)


class MX(GenericMatrixCommon):
    _rank = 2


class SX(GenericMatrixCommon):
    _rank = 1


class DM(GenericMatrixCommon):
    _rank = 0


class Sparsity(object):
    """Pattern object returned by `.sparsity()` (only what `cs.conic` call sites need)."""

    def __init__(self, shape, mask):
        self.shape = tuple(shape)
        self.mask = np.array(mask, dtype=bool).reshape(self.shape)

    def size(self):
        return self.shape

    def size1(self):
        return self.shape[0]

    def size2(self):
        return self.shape[1]

    def nnz(self):
        return int(self.mask.sum())

    def __repr__(self):
        return "Sparsity(%dx%d, %d nnz)" % (self.shape[0], self.shape[1], self.nnz())


# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------

def _filled(n, m, node):
    a = np.empty((n, m), dtype=object)
    a.fill(node)
    return a


def _axis_index(key, n) -> List[int]:
    if isinstance(key, slice):
        return list(range(*key.indices(n)))
    if isinstance(key, (list, tuple, np.ndarray)):
        return [_one_index(k, n) for k in key]
    return [_one_index(key, n)]


def _one_index(k, n):
    k = int(k)
    if k < 0:
        k += n
    if not 0 <= k < n:
        raise IndexError("index %d out of range for dimension of size %d" % (k, n))
    return k


def _to_nodes(x) -> np.ndarray:
    """Anything matrix-like -> 2-D object array of nodes (1-D input becomes a column)."""
    if isinstance(x, GenericMatrixCommon):
        return x._a
    if isinstance(x, Node):
        return _filled(1, 1, x)
    if _is_scalar_number(x):
        return _filled(1, 1, dag.const(x))
    if isinstance(x, (list, tuple)) and any(isinstance(e, (GenericMatrixCommon, Node)) for e in x):
        return vertcat(*x)._a
    arr = np.asarray(x)
    if arr.dtype == object:
        arr2 = np.empty(arr.shape, dtype=object)
        for idx, e in np.ndenumerate(arr):
            if isinstance(e, GenericMatrixCommon):
                if e.shape != (1, 1):
                    raise ValueError("nested non-scalar matrix in array")
                e = e._a[0, 0]
            arr2[idx] = dag.as_node(e)
        arr = arr2
    else:
        arr = arr.astype(np.float64)
        arr2 = np.empty(arr.shape, dtype=object)
        for idx, e in np.ndenumerate(arr):
            arr2[idx] = dag.const(e)
        arr = arr2
    if arr.ndim == 0:
        return arr.reshape(1, 1)
    if arr.ndim == 1:
        return arr.reshape(-1, 1)
    if arr.ndim == 2:
        return arr
    raise ValueError("cannot convert a %d-D array to a matrix" % arr.ndim)


def _rank_of(x):
    return x._rank if isinstance(x, GenericMatrixCommon) else 0


_CLS = {0: DM, 1: SX, 2: MX}


def _cls_for(*xs):
    return _CLS[max([_rank_of(x) for x in xs] + [0])]


def _broadcast_to(a: np.ndarray, shape):
    if a.shape == tuple(shape):
        return a
    if a.shape == (1, 1):
        return _filled(shape[0], shape[1], a[0, 0])
    if a.size == shape[0] * shape[1] and 1 in a.shape and 1 in shape:
        return a.reshape(shape)
    raise ValueError("dimension mismatch: %s vs %s" % (a.shape, tuple(shape)))


def _map1(f, x):
    cls = _cls_for(x)
    a = _to_nodes(x)
    out = np.empty(a.shape, dtype=object)
    for idx, e in np.ndenumerate(a):
        out[idx] = f(e)
    return cls._wrap(out)


def _map2(f, x, y):
    cls = _cls_for(x, y)
    a, b = _to_nodes(x), _to_nodes(y)
    if a.shape != b.shape:
        if a.shape == (1, 1):
            a = _filled(b.shape[0], b.shape[1], a[0, 0])
        elif b.shape == (1, 1):
            b = _filled(a.shape[0], a.shape[1], b[0, 0])
        else:
            raise ValueError("dimension mismatch in element-wise operation: %s vs %s"
                             % (a.shape, b.shape))
    out = np.empty(a.shape, dtype=object)
    for idx in np.ndindex(*a.shape):
        out[idx] = f(a[idx], b[idx])
    return cls._wrap(out)


def _mat(x, like=None):
    """Wrap anything as a matrix object."""
    if isinstance(x, GenericMatrixCommon):
        return x
    return _cls_for(like)._wrap(_to_nodes(x)) if like is not None else DM._wrap(_to_nodes(x))


# ----------------------------------------------------------------------------------------------
# free functions (the `cs.` namespace)
# ----------------------------------------------------------------------------------------------

def _flatten_args(args):
    if len(args) == 1 and isinstance(args[0], (list, tuple)):
        return list(args[0])
    return list(args)


def vertcat(*args):
    args = _flatten_args(args)
    if len(args) == 0:
        return DM._wrap(np.empty((0, 1), dtype=object))
    cls = _cls_for(*args)
    parts = [_to_nodes(a) for a in args]
    parts = [p for p in parts if p.shape[0] > 0] or parts[:1]
    ncol = parts[0].shape[1]
    for p in parts:
        if p.shape[1] != ncol:
            raise ValueError("vertcat: column counts differ")
    return cls._wrap(np.concatenate(parts, axis=0))


def horzcat(*args):
    args = _flatten_args(args)
    if len(args) == 0:
        return DM._wrap(np.empty((1, 0), dtype=object))
    cls = _cls_for(*args)
    parts = [_to_nodes(a) for a in args]
    parts = [p for p in parts if p.shape[1] > 0] or parts[:1]
    nrow = parts[0].shape[0]
    for p in parts:
        if p.shape[0] != nrow:
            raise ValueError("horzcat: row counts differ")
    return cls._wrap(np.concatenate(parts, axis=1))


def _mtimes2(x, y):
    cls = _cls_for(x, y)
    a, b = _to_nodes(x), _to_nodes(y)
    if a.shape == (1, 1) or b.shape == (1, 1):
        return _map2(dag.mul, cls._wrap(a), cls._wrap(b))
    if a.shape[1] != b.shape[0]:
        raise ValueError("mtimes: inner dimensions differ: %s x %s" % (a.shape, b.shape))
    out = np.empty((a.shape[0], b.shape[1]), dtype=object)
    for i in range(a.shape[0]):
        for j in range(b.shape[1]):
            acc = dag.ZERO
            for k in range(a.shape[1]):
                acc = dag.add(acc, dag.mul(a[i, k], b[k, j]))
            out[i, j] = acc
    return cls._wrap(out)


def mtimes(*args):
    args = _flatten_args(args)
    if len(args) < 2:
        raise TypeError("mtimes needs at least two factors")
    res = args[0]
    for nxt in args[1:]:
        res = _mtimes2(res, nxt)
    return res


def transpose(x):
    return _mat(x).T


def dot(x, y):
    a, b = _to_nodes(x), _to_nodes(y)
    if a.size != b.size:
        raise ValueError("dot: sizes differ")
    acc = dag.ZERO
    for p, q in zip(a.flatten(order="F"), b.flatten(order="F")):
        acc = dag.add(acc, dag.mul(p, q))
    return _cls_for(x, y)._wrap(_filled(1, 1, acc))


def sumsqr(x):
    return dot(x, x)


def norm_2(x):
    a = _to_nodes(x)
    if 1 not in a.shape and a.size > 1:
        raise NotImplementedError("norm_2 of a matrix (spectral norm) is not supported")
    return _map1(dag.sqrt, sumsqr(x))


def norm_fro(x):
    return _map1(dag.sqrt, sumsqr(x))


def norm_1(x):
    a = _to_nodes(x)
    acc = dag.ZERO
    for e in a.flat:
        acc = dag.add(acc, dag.fabs(e))
    return _cls_for(x)._wrap(_filled(1, 1, acc))


def norm_inf(x):
    a = _to_nodes(x)
    acc = dag.ZERO
    for e in a.flat:
        acc = dag.fmax(acc, dag.fabs(e))
    return _cls_for(x)._wrap(_filled(1, 1, acc))


def sum1(x):
    a = _to_nodes(x)
    out = np.empty((1, a.shape[1]), dtype=object)
    for j in range(a.shape[1]):
        acc = dag.ZERO
        for i in range(a.shape[0]):
            acc = dag.add(acc, a[i, j])
        out[0, j] = acc
    return _cls_for(x)._wrap(out)


def sum2(x):
    return sum1(_mat(x).T).T


def trace(x):
    a = _to_nodes(x)
    acc = dag.ZERO
    for i in range(min(a.shape)):
        acc = dag.add(acc, a[i, i])
    return _cls_for(x)._wrap(_filled(1, 1, acc))


def diag(x):
    a = _to_nodes(x)
    cls = _cls_for(x)
    if 1 in a.shape:
        v = a.reshape(-1)
        out = _filled(len(v), len(v), dag.ZERO)
        for i, e in enumerate(v):
            out[i, i] = e
        return cls._wrap(out)
    n = min(a.shape)
    out = np.empty((n, 1), dtype=object)
    for i in range(n):
        out[i, 0] = a[i, i]
    return cls._wrap(out)


def reshape(x, *shape):
    if len(shape) == 1:
        shape = tuple(shape[0])
    a = _to_nodes(x)
    return _cls_for(x)._wrap(a.flatten(order="F").reshape(shape, order="F"))


def vec(x):
    a = _to_nodes(x)
    return _cls_for(x)._wrap(a.flatten(order="F").reshape(-1, 1))


def cross(x, y):
    a = _to_nodes(x).reshape(-1)
    b = _to_nodes(y).reshape(-1)
    if len(a) != 3 or len(b) != 3:
        raise ValueError("cross: 3-vectors expected")
    out = np.empty((3, 1), dtype=object)
    out[0, 0] = dag.sub(dag.mul(a[1], b[2]), dag.mul(a[2], b[1]))
    out[1, 0] = dag.sub(dag.mul(a[2], b[0]), dag.mul(a[0], b[2]))
    out[2, 0] = dag.sub(dag.mul(a[0], b[1]), dag.mul(a[1], b[0]))
    res = _cls_for(x, y)._wrap(out)
    return res if _to_nodes(x).shape[1] == 1 else res.T


def _elementwise(f):
    def g(x):
        if _is_scalar_number(x):
            return float(dag.as_node(f(dag.const(x))).val)
        return _map1(f, x)
    g.__name__ = f.__name__
    return g


sin = _elementwise(dag.sin)
cos = _elementwise(dag.cos)
tan = _elementwise(dag.tan)
asin = _elementwise(dag.asin)
acos = _elementwise(dag.acos)
atan = _elementwise(dag.atan)
exp = _elementwise(dag.exp)
log = _elementwise(dag.log)
sqrt = _elementwise(dag.sqrt)
fabs = _elementwise(dag.fabs)
sign = _elementwise(dag.sign)
floor = _elementwise(dag.floor)
ceil = _elementwise(dag.ceil)
logic_not = _elementwise(dag.logic_not)


def atan2(x, y): return _map2(dag.atan2, x, y)
def fmin(x, y): return _map2(dag.fmin, x, y)
def fmax(x, y): return _map2(dag.fmax, x, y)
def logic_and(x, y): return _map2(dag.logic_and, x, y)
def logic_or(x, y): return _map2(dag.logic_or, x, y)
def power(x, y): return _map2(dag.pow_, x, y)


def if_else(c, a, b, short_circuit=False):
    """Element-wise select; `short_circuit` is accepted for signature parity (the generated code
    evaluates both branches and selects, which is value-identical for finite operands)."""
    cls = _cls_for(c, a, b)
    cn, an, bn = _to_nodes(c), _to_nodes(a), _to_nodes(b)
    shape = max((an.shape, bn.shape, cn.shape), key=lambda s: s[0] * s[1])
    cn, an, bn = (_broadcast_to(z, shape) for z in (cn, an, bn))
    out = np.empty(shape, dtype=object)
    for idx in np.ndindex(*shape):
        out[idx] = dag.if_else(cn[idx], an[idx], bn[idx])
    return cls._wrap(out)


# ---- calculus -----------------------------------------------------------------------------------

def _sym_list(v) -> List[Node]:
    nodes = _mat(v).nodes()
    for n in nodes:
        if not n.is_sym:
            raise ValueError("differentiation variable must be purely symbolic")
    return nodes


def jacobian(expr, var):
    e = _mat(expr)
    outs = e.nodes()
    wrt = _sym_list(var)
    rows = dag.jacobian(outs, wrt)
    out = np.empty((len(outs), len(wrt)), dtype=object)
    for i, r in enumerate(rows):
        for j, n in enumerate(r):
            out[i, j] = n
    return _cls_for(expr, var)._wrap(out)


def jtimes(expr, var, direction, transposed=False):
    """J(expr, var) @ direction, without forming J (one forward sweep)."""
    if transposed:
        return mtimes(jacobian(expr, var).T, direction)
    e = _mat(expr)
    outs = e.nodes()
    wrt = _sym_list(var)
    dmat = _to_nodes(direction)
    if dmat.shape[0] != len(wrt):
        raise ValueError("jtimes: direction has %d rows, variable has %d" % (dmat.shape[0], len(wrt)))
    cols = []
    for j in range(dmat.shape[1]):
        seeds = {s.id: dmat[i, j] for i, s in enumerate(wrt)}
        cols.append(dag.forward(outs, seeds))
    out = np.empty((len(outs), dmat.shape[1]), dtype=object)
    for j, c in enumerate(cols):
        for i, n in enumerate(c):
            out[i, j] = n
    return _cls_for(expr, var, direction)._wrap(out)


def gradient(expr, var):
    return jacobian(expr, var).T


def hessian(expr, var):
    """-> (H, g): the Hessian of the scalar `expr` with respect to `var` and its gradient, as
    casadi.hessian returns them (H = jacobian(gradient(expr, var), var))."""
    g = gradient(expr, var)
    return jacobian(g, var), g


def substitute(expr, var, val):
    e = _mat(expr)
    syms = _sym_list(var)
    vals = _to_nodes(val).flatten(order="F")
    if len(vals) != len(syms):
        raise ValueError("substitute: size mismatch")
    new = dag.substitute(e.nodes(), {s.id: v for s, v in zip(syms, vals)})
    out = np.array(new, dtype=object).reshape(e._a.shape, order="F")
    return _cls_for(expr, val)._wrap(out)


def depends_on(expr, var):
    return dag.depends_on(_mat(expr).nodes(), _sym_list(var))


def symvar(expr):
    return [MX._wrap(_filled(1, 1, s)) for s in dag.symbols_of(_mat(expr).nodes())]


# ---- small dense linear algebra on expressions -----------------------------------------------------

def _solve_nodes(A: np.ndarray, B: np.ndarray) -> np.ndarray:
    """Gaussian elimination on node matrices.  Constant systems go through NumPy; symbolic ones
    are eliminated without pivoting except for structurally-zero pivots."""
    n = A.shape[0]
    if A.shape[0] != A.shape[1] or B.shape[0] != n:
        raise ValueError("solve: dimension mismatch")
    if all(e.is_const for e in A.flat) and all(e.is_const for e in B.flat):
        a = np.array([[e.val for e in r] for r in A], dtype=np.float64).reshape(A.shape)
        b = np.array([[e.val for e in r] for r in B], dtype=np.float64).reshape(B.shape)
        x = np.linalg.solve(a, b)
        return _to_nodes(x.reshape(B.shape))
    A = A.copy()
    B = B.copy()
    for k in range(n):
        if A[k, k] is dag.ZERO:
            for r in range(k + 1, n):
                if A[r, k] is not dag.ZERO:
                    A[[k, r]] = A[[r, k]]
                    B[[k, r]] = B[[r, k]]
                    break
            else:
                raise ZeroDivisionError("solve: structurally singular matrix")
        for r in range(k + 1, n):
            if A[r, k] is dag.ZERO:
                continue
            f = dag.div(A[r, k], A[k, k])
            for c in range(k + 1, n):
                A[r, c] = dag.sub(A[r, c], dag.mul(f, A[k, c]))
            for c in range(B.shape[1]):
                B[r, c] = dag.sub(B[r, c], dag.mul(f, B[k, c]))
            A[r, k] = dag.ZERO
    X = np.empty(B.shape, dtype=object)
    for c in range(B.shape[1]):
        for r in range(n - 1, -1, -1):
            acc = B[r, c]
            for k in range(r + 1, n):
                acc = dag.sub(acc, dag.mul(A[r, k], X[k, c]))
            X[r, c] = dag.div(acc, A[r, r])
    return X


def solve(A, B, *unused_solver_args):
    return _cls_for(A, B)._wrap(_solve_nodes(_to_nodes(A), _to_nodes(B)))


def inv(A):
    a = _to_nodes(A)
    return _cls_for(A)._wrap(_solve_nodes(a, DM.eye(a.shape[0])._a))


def det(A):
    a = _to_nodes(A)
    n = a.shape[0]
    if a.shape[0] != a.shape[1]:
        raise ValueError("det: square matrix expected")
    if n == 0:
        return DM(1.0)

    def minor(m, i, j):
        return np.delete(np.delete(m, i, axis=0), j, axis=1)

    def _det(m):
        if m.shape[0] == 1:
            return m[0, 0]
        acc = dag.ZERO
        for j in range(m.shape[0]):
            if m[0, j] is dag.ZERO:
                continue
            term = dag.mul(m[0, j], _det(minor(m, 0, j)))
            acc = dag.add(acc, term) if j % 2 == 0 else dag.sub(acc, term)
        return acc

    return _cls_for(A)._wrap(_filled(1, 1, _det(a)))


def pinv(A):
    """Moore-Penrose pseudo-inverse for full-rank matrices: A'(AA')^-1 (wide) or (A'A)^-1 A' (tall)."""
    a = _mat(A)
    if a.size2() >= a.size1():
        return solve(mtimes(a, a.T), a).T
    return solve(mtimes(a.T, a), a.T)


# ----------------------------------------------------------------------------------------------
# Function
# ----------------------------------------------------------------------------------------------

class Function(object):
    """`cs.Function(name, inputs, outputs[, in_names, out_names][, opts])`.

    Calling it with numbers evaluates numerically and returns DM; calling it with symbolic
    arguments returns the substituted expressions (this is how the notebooks use `T_fk(q)`).
    `opts` (jit flags etc., reference pseudo_inverse.py:59-65) is accepted and ignored here: the
    controllers compile whole skills to CUDA, not individual Functions.
    """

    def __init__(self, name, ins, outs, *rest):
        self._name = name
        in_names = out_names = None
        opts = {}
        rest = list(rest)
        if rest and isinstance(rest[-1], dict):
            opts = rest.pop()
        if len(rest) >= 2:
            in_names, out_names = rest[0], rest[1]
        self.opts = opts
        self._ins = [_mat(i) for i in ins]
        for k, i in enumerate(self._ins):
            if not i.is_symbolic() and i.numel() > 0:
                raise ValueError("Function %s: input %d is not purely symbolic" % (name, k))
        self._outs = [_mat(o) for o in outs]
        self._in_names = list(in_names) if in_names else ["i%d" % k for k in range(len(self._ins))]
        self._out_names = list(out_names) if out_names else ["o%d" % k for k in range(len(self._outs))]
        known = {n.id for i in self._ins for n in i.nodes()}
        out_nodes = [n for o in self._outs for n in o.nodes()]
        free = [s.name for s in dag.symbols_of(out_nodes) if s.id not in known]
        if free:
            raise RuntimeError("Function %s: free variables %s in outputs" % (name, sorted(set(free))))

    def name(self): return self._name
    def n_in(self): return len(self._ins)
    def n_out(self): return len(self._outs)
    def name_in(self, i=None): return self._in_names if i is None else self._in_names[i]
    def name_out(self, i=None): return self._out_names if i is None else self._out_names[i]
    def size_in(self, i): return self._ins[i].shape
    def size_out(self, i): return self._outs[i].shape
    def mx_in(self, i=None): return self._ins if i is None else self._ins[i]
    def mx_out(self, i=None): return self._outs if i is None else self._outs[i]

    def __repr__(self):
        sig = ",".join("%s[%dx%d]" % (n, *i.shape) for n, i in zip(self._in_names, self._ins))
        osig = ",".join("%s[%dx%d]" % (n, *o.shape) for n, o in zip(self._out_names, self._outs))
        return "Function(%s:(%s)->(%s))" % (self._name, sig, osig)

    def _bind(self, args):
        if len(args) != len(self._ins):
            raise TypeError("Function %s expects %d arguments, got %d"
                            % (self._name, len(self._ins), len(args)))
        mapping = {}
        cls_rank = 0
        for k, (formal, actual) in enumerate(zip(self._ins, args)):
            cls_rank = max(cls_rank, _rank_of(actual))
            a = _to_nodes(actual)
            if a.shape != formal._a.shape:
                if a.size == formal.numel() and (1 in a.shape or a.size == 1):
                    a = a.reshape(formal._a.shape, order="F")
                elif a.shape == (1, 1):
                    a = _filled(formal._a.shape[0], formal._a.shape[1], a[0, 0])
                else:
                    raise ValueError("Function %s: argument %d (%s) has shape %s, expected %s"
                                     % (self._name, k, self._in_names[k], a.shape, formal._a.shape))
            for s, v in zip(formal.nodes(), a.flatten(order="F")):
                mapping[s.id] = v
        return mapping, cls_rank

    def call(self, args):
        mapping, rank = self._bind(list(args))
        numeric = all(v.is_const for v in mapping.values())
        results = []
        if numeric:
            values = {k: v.val for k, v in mapping.items()}
            flat = [n for o in self._outs for n in o.nodes()]
            vals = dag.evaluate(flat, values) if flat else []
            pos = 0
            for o in self._outs:
                k = o.numel()
                arr = np.array([float(x) for x in vals[pos:pos + k]], dtype=np.float64)
                pos += k
                results.append(DM._wrap(_to_nodes(arr.reshape(o.shape, order="F"))))
        else:
            cls = _CLS[max(rank, 1)]
            for o in self._outs:
                new = dag.substitute(o.nodes(), mapping)
                results.append(cls._wrap(np.array(new, dtype=object).reshape(o.shape, order="F")))
        return results

    def __call__(self, *args, **kwargs):
        if kwargs:
            if args:
                raise TypeError("mixing positional and keyword arguments is not supported")
            ordered = []
            for nm, formal in zip(self._in_names, self._ins):
                ordered.append(kwargs.get(nm, DM.zeros(*formal.shape)))
            res = self.call(ordered)
            return dict(zip(self._out_names, res))
        res = self.call(args)
        if len(res) == 1:
            return res[0]
        return tuple(res)
