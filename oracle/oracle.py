"""oracle.py — numpy/ctypes front end of the CPU oracle (oracle/gnn_oracle.c).

TEST INFRASTRUCTURE, NOT PRODUCT: only tests/, __graft_entry__.smoke() and bench.py's CPU legs import this.
See the header of gnn_oracle.c for what is restated (reference file:line) and for the pinning statement
(known-answer vectors of the reference's own tests; max/min through propagate is "parity unpinned").

Array convention: numpy arrays are C-order "rows" — x has shape (N, D) which is the same memory as the
reference's column-major (D, N).  Indices are 1-based int64 like the reference's.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")

SUM, MEAN, MAX, MIN = 0, 1, 2, 3
DIR_OUT, DIR_IN, DIR_BOTH = 0, 1, 2
_AGGR = {"+": SUM, "sum": SUM, "mean": MEAN, "max": MAX, "min": MIN, SUM: SUM, MEAN: MEAN, MAX: MAX, MIN: MIN}


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("gnn_oracle.c", "gnn_oracle_impl.h", "Makefile")]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.orc_num_threads.restype = C.c_int
    return _lib


def _sfx(dtype):
    return "_f32" if np.dtype(dtype) == np.float32 else "_f64"


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _idx(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.int64))


def _f(a, dtype):
    return None if a is None else np.ascontiguousarray(np.asarray(a, dtype=dtype))


def num_threads() -> int:
    return int(lib().orc_num_threads())


def gather(x, idx):
    x = np.ascontiguousarray(x)
    idx = _idx(idx)
    D = int(np.prod(x.shape[1:])) if x.ndim > 1 else 1
    out = np.empty((len(idx),) + x.shape[1:], dtype=x.dtype)
    getattr(lib(), "orc_gather" + _sfx(x.dtype))(_p(x), _p(idx), C.c_int64(len(idx)), C.c_int64(D), _p(out))
    return out


def scatter(aggr, m, idx, n):
    m = np.ascontiguousarray(m)
    idx = _idx(idx)
    D = int(np.prod(m.shape[1:])) if m.ndim > 1 else 1
    out = np.empty((n,) + m.shape[1:], dtype=m.dtype)
    getattr(lib(), "orc_scatter" + _sfx(m.dtype))(C.c_int(_AGGR[aggr]), _p(m), _p(idx), C.c_int64(len(idx)),
                                                  C.c_int64(D), C.c_int64(n), _p(out))
    return out


def propagate_unfused(aggr, s, t, n, x, w=None):
    """gather -> (w .*) -> scatter, the path every GPU call and every mean/max call of the reference takes."""
    x = np.ascontiguousarray(x)
    s, t = _idx(s), _idx(t)
    w = _f(w, x.dtype)
    D = int(np.prod(x.shape[1:]))
    out = np.empty((n,) + x.shape[1:], dtype=x.dtype)
    rc = getattr(lib(), "orc_propagate_unfused" + _sfx(x.dtype))(
        C.c_int(_AGGR[aggr]), _p(s), _p(t), C.c_int64(len(s)), C.c_int64(n), _p(x), _p(w), C.c_int64(D), _p(out))
    assert rc == 0
    return out


def propagate_fused(s, t, n, x, w=None):
    """xj * adjacency_matrix(g): COO -> CSC rebuilt per call + serial dense x CSC (msgpass.jl:215-238)."""
    x = np.ascontiguousarray(x)
    s, t = _idx(s), _idx(t)
    w = _f(w, x.dtype)
    D = int(np.prod(x.shape[1:]))
    out = np.empty((n,) + x.shape[1:], dtype=x.dtype)
    rc = getattr(lib(), "orc_propagate_fused" + _sfx(x.dtype))(
        _p(s), _p(t), C.c_int64(len(s)), C.c_int64(n), _p(x), _p(w), C.c_int64(D), _p(out))
    assert rc == 0
    return out


def degree(s, t, n, dir="in", w=None, dtype=np.float32):
    s, t = _idx(s), _idx(t)
    w = _f(w, dtype)
    out = np.empty(n, dtype=dtype)
    d = {"out": DIR_OUT, "in": DIR_IN, "both": DIR_BOTH}[dir]
    getattr(lib(), "orc_degree" + _sfx(dtype))(_p(s), _p(t), C.c_int64(len(s)), C.c_int64(n), C.c_int(d), _p(w),
                                               _p(out))
    return out


def softmax_edge_neighbors(t, n, e):
    e = np.ascontiguousarray(e)
    t = _idx(t)
    K = int(np.prod(e.shape[1:])) if e.ndim > 1 else 1
    out = np.empty_like(e)
    getattr(lib(), "orc_softmax_edge_neighbors" + _sfx(e.dtype))(_p(t), C.c_int64(len(t)), C.c_int64(n), _p(e),
                                                                 C.c_int64(K), _p(out))
    return out


def gcn_propagate(s, t, n, x, w=None, fused=True):
    """c .* propagate(copy_xj|e_mul_xj, +, xj = x .* c'), c = 1/sqrt(in-degree) (conv.jl:52-67). Returns (out, c)."""
    x = np.ascontiguousarray(x)
    s, t = _idx(s), _idx(t)
    w = _f(w, x.dtype)
    D = int(np.prod(x.shape[1:]))
    out = np.empty_like(x)
    c = np.empty(n, dtype=x.dtype)
    rc = getattr(lib(), "orc_gcn_propagate" + _sfx(x.dtype))(
        _p(s), _p(t), C.c_int64(len(s)), C.c_int64(n), _p(x), _p(w), C.c_int64(D), C.c_int(1 if fused else 0),
        _p(out), _p(c))
    assert rc == 0
    return out, c


def gat_aggregate(s, t, n, Wx, a, slope=0.2):
    """Wx (N, H, C) rows, a (H, 2C) rows [= Julia (2C, H)].  Returns (out (N,H,C), alpha (E,H))."""
    Wx = np.ascontiguousarray(Wx)
    a = _f(a, Wx.dtype)
    s, t = _idx(s), _idx(t)
    N, H, Cc = Wx.shape
    assert a.shape == (H, 2 * Cc)
    out = np.empty_like(Wx)
    alpha = np.empty((len(s), H), dtype=Wx.dtype)
    ct = C.c_float if Wx.dtype == np.float32 else C.c_double
    rc = getattr(lib(), "orc_gat_aggregate" + _sfx(Wx.dtype))(
        _p(s), _p(t), C.c_int64(len(s)), C.c_int64(n), _p(Wx), _p(a), C.c_int64(Cc), C.c_int64(H), ct(slope),
        _p(out), _p(alpha))
    assert rc == 0
    return out, alpha


def gat_logit_halves(Wx, a):
    """el (N, H), er (N, H): the target and source halves of sum(a .* vcat(Wxi, Wxj), dims=1), in Wx's dtype.
    Wx (N, H, C) rows, a (H, 2C) rows."""
    Cc = Wx.shape[2]
    a = np.asarray(a, dtype=Wx.dtype)
    return (np.einsum("nhc,hc->nh", Wx, a[:, :Cc]), np.einsum("nhc,hc->nh", Wx, a[:, Cc:]))


def gat_aggregate_bwd(s, t, n, Wx, dout, slope=0.2, *, a=None, el=None, er=None):
    """Pullback of gat_aggregate for the upstream dout (N, H, C).  The logits come from el, er (N, H) or, given a (H, 2C),
    from gat_logit_halves(Wx, a).  Returns (dWx (N,H,C): the edge part only, del (N,H), der (N,H), alpha (E,H)); the
    logit chain into Wx and a is dWx += del a[:, :C] + der a[:, C:],  da = [Σ_n del Wx, Σ_n der Wx]."""
    Wx = np.ascontiguousarray(Wx)
    if a is not None:
        el, er = gat_logit_halves(Wx, a)
    el, er, dout = _f(el, Wx.dtype), _f(er, Wx.dtype), _f(dout, Wx.dtype)
    s, t = _idx(s), _idx(t)
    N, H, Cc = Wx.shape
    assert dout.shape == Wx.shape and el.shape == er.shape == (N, H)
    dWx = np.empty_like(Wx)
    del_, der = np.empty((n, H), dtype=Wx.dtype), np.empty((n, H), dtype=Wx.dtype)
    alpha = np.empty((len(s), H), dtype=Wx.dtype)
    ct = C.c_float if Wx.dtype == np.float32 else C.c_double
    rc = getattr(lib(), "orc_gat_aggregate_bwd" + _sfx(Wx.dtype))(
        _p(s), _p(t), C.c_int64(len(s)), C.c_int64(n), _p(Wx), _p(el), _p(er), C.c_int64(Cc), C.c_int64(H), ct(slope),
        _p(dout), _p(dWx), _p(del_), _p(der), _p(alpha))
    assert rc == 0
    return dWx, del_, der, alpha


def add_self_loops(s, t, n):
    s, t = _idx(s), _idx(t)
    s2 = np.empty(len(s) + n, dtype=np.int64)
    t2 = np.empty(len(s) + n, dtype=np.int64)
    lib().orc_add_self_loops(_p(s), _p(t), C.c_int64(len(s)), C.c_int64(n), _p(s2), _p(t2))
    return s2, t2


def csr(key, other, n):
    """stable CSR by key: (rowptr[n+1], col[E], perm[E]) all 0-based int32."""
    key, other = _idx(key), _idx(other)
    E = len(key)
    rowptr = np.empty(n + 1, dtype=np.int32)
    col = np.empty(E, dtype=np.int32)
    perm = np.empty(E, dtype=np.int32)
    lib().orc_csr(_p(key), _p(other), C.c_int64(E), C.c_int64(n), _p(rowptr), _p(col), _p(perm))
    return rowptr, col, perm


def rmat(n, E, seed=17):
    s = np.empty(E, dtype=np.int64)
    t = np.empty(E, dtype=np.int64)
    lib().orc_rmat(C.c_int64(n), C.c_int64(E), C.c_uint64(seed), _p(s), _p(t))
    return s, t


def spmm_csr_omp(rowptr, col, n, x, w=None, cs=None, ct=None):
    x = _f(x, np.float32)
    out = np.empty((n,) + x.shape[1:], dtype=np.float32)
    D = int(np.prod(x.shape[1:]))
    lib().orc_spmm_csr_omp(_p(np.ascontiguousarray(rowptr, dtype=np.int32)),
                           _p(np.ascontiguousarray(col, dtype=np.int32)), C.c_int64(n), _p(x),
                           _p(_f(w, np.float32)), _p(_f(cs, np.float32)), _p(_f(ct, np.float32)), C.c_int64(D),
                           _p(out))
    return out


# ---- pure-numpy cross-checks (independent of the C code; used to pin the oracle itself) ----------------
def dense_adjacency(s, t, n, w=None, dtype=np.float64):
    """A[i,j] = number (or summed weight) of edges i -> j (GNNGraphs/src/query.jl:220-231, duplicates summed)."""
    A = np.zeros((n, n), dtype=dtype)
    np.add.at(A, (np.asarray(s) - 1, np.asarray(t) - 1), 1.0 if w is None else np.asarray(w, dtype=dtype))
    return A


def csc_build(s, t, n, w=None, dtype=np.float32):
    """A = sparse(s, t, w, n, n): returns (colptr[n+1], rowval[nnz], nzval[nnz]) 0-based, duplicates summed."""
    s, t = _idx(s), _idx(t)
    w = _f(w, dtype)
    E = len(s)
    colptr = np.empty(n + 1, dtype=np.int64)
    rowval = np.empty(max(E, 1), dtype=np.int64)
    nzval = np.empty(max(E, 1), dtype=dtype)
    nnz = getattr(lib(), "orc_csc_build" + _sfx(dtype))
    nnz.restype = C.c_int64
    k = nnz(_p(s), _p(t), C.c_int64(E), C.c_int64(n), _p(w), _p(colptr), _p(rowval), _p(nzval))
    assert k >= 0
    return colptr, rowval[:k], nzval[:k]


def dense_times_csc(x, csc, transposed=False):
    """xj * A (forward) or Δ * A' (pullback) with the CSC from csc_build."""
    colptr, rowval, nzval = csc
    x = _f(x, nzval.dtype)
    n = len(colptr) - 1
    D = int(np.prod(x.shape[1:]))
    out = np.empty_like(x)
    name = ("orc_dense_times_csc_t" if transposed else "orc_dense_times_csc") + _sfx(x.dtype)
    getattr(lib(), name)(_p(x), C.c_int64(n), C.c_int64(D), _p(colptr), _p(np.ascontiguousarray(rowval)),
                         _p(np.ascontiguousarray(nzval)), _p(out))
    return out
