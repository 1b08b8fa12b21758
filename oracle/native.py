"""TEST INFRASTRUCTURE ONLY -- ctypes access to the CPU oracles. Not part of the product path.

Two back-ends, both CPU:

* ``port``  -- ``oracle/liboracle.so``: our C restatement (``oracle/d3f_oracle.c``).
* ``ref``   -- ``oracle/_ref/libref_tf.so`` / ``libref_wrap.so``: the reference's own C++ cores compiled
  from ``/root/reference`` by ``oracle/Makefile`` (prebuilt files travel to the GPU box).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may import this module.
"""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PORT = os.path.join(_HERE, "liboracle.so")
_REF_TF = os.path.join(_HERE, "_ref", "libref_tf.so")
_REF_WRAP = os.path.join(_HERE, "_ref", "libref_wrap.so")

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")


def build(ref=True):
    """Compile the oracle (and the reference cores when /root/reference is present)."""
    subprocess.check_call(["make", "-s", "-C", _HERE, "oracle"])
    if ref and os.path.isdir("/root/reference/tf_custom_ops"):
        subprocess.check_call(["make", "-s", "-C", _HERE, "ref"])


_port = None


def port():
    global _port
    if _port is None:
        if not os.path.exists(_PORT):
            build(ref=False)
        lib = C.CDLL(_PORT)
        lib.orc_grid_subsample.restype = C.c_int
        lib.orc_grid_subsample.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                           C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.orc_batch_grid_subsample.restype = C.c_int
        lib.orc_batch_grid_subsample.argtypes = [_f32p, C.c_int, _i32p, C.c_int, C.c_float, _f32p, _i32p]
        lib.orc_batch_neighbors_count.restype = C.c_int
        lib.orc_batch_neighbors_count.argtypes = [_f32p, C.c_int, _f32p, C.c_int, _i32p, _i32p, C.c_int,
                                                  C.c_float, _i32p]
        lib.orc_batch_neighbors_fill.restype = None
        lib.orc_batch_neighbors_fill.argtypes = [_f32p, C.c_int, _f32p, C.c_int, _i32p, _i32p, C.c_int,
                                                 C.c_float, C.c_int, C.c_int, _i32p]
        _port = lib
    return _port


def have_ref():
    return os.path.exists(_REF_TF) and os.path.exists(_REF_WRAP)


_ref_tf = None
_ref_wrap = None


def ref_tf():
    global _ref_tf
    if _ref_tf is None:
        lib = C.CDLL(_REF_TF)
        lib.ref_free.argtypes = [C.c_void_p]
        lib.ref_batch_neighbors.restype = C.POINTER(C.c_int)
        lib.ref_batch_neighbors.argtypes = [_f32p, C.c_int, _f32p, C.c_int, _i32p, _i32p, C.c_int, C.c_float,
                                            C.POINTER(C.c_int)]
        lib.ref_ordered_neighbors.restype = C.POINTER(C.c_int)
        lib.ref_ordered_neighbors.argtypes = [_f32p, C.c_int, _f32p, C.c_int, C.c_float, C.POINTER(C.c_int)]
        lib.ref_batch_subsampling.restype = C.POINTER(C.c_float)
        lib.ref_batch_subsampling.argtypes = [_f32p, C.c_int, _i32p, C.c_int, C.c_float, _i32p,
                                              C.POINTER(C.c_int)]
        lib.ref_grid_subsampling.restype = C.POINTER(C.c_float)
        lib.ref_grid_subsampling.argtypes = [_f32p, C.c_int, C.c_float, C.POINTER(C.c_int)]
        _ref_tf = lib
    return _ref_tf


def ref_wrap():
    global _ref_wrap
    if _ref_wrap is None:
        lib = C.CDLL(_REF_WRAP)
        lib.refw_free.argtypes = [C.c_void_p]
        lib.refw_grid_subsampling.restype = C.c_int
        lib.refw_grid_subsampling.argtypes = [_f32p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                              C.c_float, C.c_int, C.POINTER(C.POINTER(C.c_float)),
                                              C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.POINTER(C.c_int)),
                                              C.POINTER(C.c_int)]
        _ref_wrap = lib
    return _ref_wrap


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


# ----------------------------------------------------------------------------------------------------
#  port (C restatement)
# ----------------------------------------------------------------------------------------------------

def port_grid_subsample(points, features=None, classes=None, sampleDl=0.1, return_keys=False):
    """Canonical-order (ascending cell key) restatement of cpp_subsampling.compute."""
    pts = _f32(points)
    N = pts.shape[0]
    fdim = ldim = 0
    f = c = None
    if features is not None:
        f = _f32(features)
        fdim = f.shape[1]
    if classes is not None:
        c = _i32(classes).reshape(N, -1)
        ldim = c.shape[1]
    op = np.empty((max(N, 1), 3), np.float32)
    of = np.empty((max(N, 1), max(fdim, 1)), np.float32)
    oc = np.empty((max(N, 1), max(ldim, 1)), np.int32)
    ok = np.empty((max(N, 1),), np.uint64)
    M = port().orc_grid_subsample(pts.ctypes.data, N, f.ctypes.data if f is not None else None, fdim,
                                  c.ctypes.data if c is not None else None, ldim, float(sampleDl),
                                  op.ctypes.data, of.ctypes.data, oc.ctypes.data, ok.ctypes.data)
    out = [op[:M].copy()]
    if f is not None:
        out.append(of[:M, :fdim].copy())
    if c is not None:
        out.append(oc[:M, :ldim].copy())
    if return_keys:
        out.append(ok[:M].copy())
    return out[0] if len(out) == 1 else tuple(out)


def port_batch_subsampling(points, batches, sampleDl):
    pts, b = _f32(points), _i32(batches)
    op = np.empty((max(pts.shape[0], 1), 3), np.float32)
    ob = np.empty((b.shape[0],), np.int32)
    M = port().orc_batch_grid_subsample(pts, pts.shape[0], b, b.shape[0], float(sampleDl), op, ob)
    return op[:M].copy(), ob


def port_batch_neighbors(queries, supports, q_batches, s_batches, radius, pad_value=None, max_cols=None,
                         return_counts=False):
    """Canonical-order ((d2, index) ascending) restatement of batch_nanoflann_neighbors."""
    q, s, qb, sb = _f32(queries), _f32(supports), _i32(q_batches), _i32(s_batches)
    Nq, Ns, B = q.shape[0], s.shape[0], qb.shape[0]
    counts = np.zeros((max(Nq, 1),), np.int32)
    maxc = port().orc_batch_neighbors_count(q, Nq, s, Ns, qb, sb, B, float(radius), counts)
    cols = maxc if max_cols is None else min(maxc, int(max_cols))
    out = np.empty((Nq, cols), np.int32)
    if Nq * cols > 0:
        port().orc_batch_neighbors_fill(q, Nq, s, Ns, qb, sb, B, float(radius), cols,
                                        Ns if pad_value is None else int(pad_value), out)
    return (out, counts[:Nq]) if return_counts else out


def port_ordered_neighbors(queries, supports, radius):
    q, s = _f32(queries), _f32(supports)
    return port_batch_neighbors(q, s, [q.shape[0]], [s.shape[0]], radius, pad_value=-1)


# ----------------------------------------------------------------------------------------------------
#  ref (the reference's compiled C++ cores)
# ----------------------------------------------------------------------------------------------------

def ref_batch_neighbors(queries, supports, q_batches, s_batches, radius):
    q, s, qb, sb = _f32(queries), _f32(supports), _i32(q_batches), _i32(s_batches)
    cols = C.c_int(0)
    lib = ref_tf()
    p = lib.ref_batch_neighbors(q, q.shape[0], s, s.shape[0], qb, sb, qb.shape[0], float(radius), C.byref(cols))
    out = np.ctypeslib.as_array(p, shape=(q.shape[0] * cols.value + 1,))[:q.shape[0] * cols.value].copy()
    lib.ref_free(p)
    return out.reshape(q.shape[0], cols.value).astype(np.int32)


def ref_ordered_neighbors(queries, supports, radius):
    q, s = _f32(queries), _f32(supports)
    cols = C.c_int(0)
    lib = ref_tf()
    p = lib.ref_ordered_neighbors(q, q.shape[0], s, s.shape[0], float(radius), C.byref(cols))
    out = np.ctypeslib.as_array(p, shape=(q.shape[0] * cols.value + 1,))[:q.shape[0] * cols.value].copy()
    lib.ref_free(p)
    return out.reshape(q.shape[0], cols.value).astype(np.int32)


def ref_batch_subsampling(points, batches, sampleDl):
    pts, b = _f32(points), _i32(batches)
    ob = np.empty((b.shape[0],), np.int32)
    M = C.c_int(0)
    lib = ref_tf()
    p = lib.ref_batch_subsampling(pts, pts.shape[0], b, b.shape[0], float(sampleDl), ob, C.byref(M))
    out = np.ctypeslib.as_array(p, shape=(3 * M.value + 1,))[:3 * M.value].copy()
    lib.ref_free(p)
    return out.reshape(M.value, 3), ob


def ref_grid_subsampling_tf(points, sampleDl):
    pts = _f32(points)
    M = C.c_int(0)
    lib = ref_tf()
    p = lib.ref_grid_subsampling(pts, pts.shape[0], float(sampleDl), C.byref(M))
    out = np.ctypeslib.as_array(p, shape=(3 * M.value + 1,))[:3 * M.value].copy()
    lib.ref_free(p)
    return out.reshape(M.value, 3)


def ref_grid_subsample(points, features=None, classes=None, sampleDl=0.1, verbose=0):
    """The cpp_wrappers core (what cpp_subsampling.compute runs), reference order."""
    pts = _f32(points)
    N = pts.shape[0]
    f = c = None
    fdim = ldim = 0
    if features is not None:
        f = _f32(features)
        fdim = f.shape[1]
    if classes is not None:
        c = _i32(classes).reshape(N, -1)
        ldim = c.shape[1]
    lib = ref_wrap()
    pp, pf, pc = C.POINTER(C.c_float)(), C.POINTER(C.c_float)(), C.POINTER(C.c_int)()
    M = C.c_int(0)
    lib.refw_grid_subsampling(pts, N, f.ctypes.data if f is not None else None, fdim,
                              c.ctypes.data if c is not None else None, ldim, float(sampleDl), int(verbose),
                              C.byref(pp), C.byref(pf), C.byref(pc), C.byref(M))
    m = M.value
    out = [np.ctypeslib.as_array(pp, shape=(3 * m + 1,))[:3 * m].copy().reshape(m, 3)]
    lib.refw_free(pp)
    if f is not None:
        out.append(np.ctypeslib.as_array(pf, shape=(m * fdim + 1,))[:m * fdim].copy().reshape(m, fdim))
        lib.refw_free(pf)
    if c is not None:
        out.append(np.ctypeslib.as_array(pc, shape=(m * ldim + 1,))[:m * ldim].copy().reshape(m, ldim))
        lib.refw_free(pc)
    return out[0] if len(out) == 1 else tuple(out)


# ----------------------------------------------------------------------------------------------------
#  canonicalisation helpers (shared by the tests)
# ----------------------------------------------------------------------------------------------------

def sqdist_f32(q, s):
    """fp32 d2 with separately rounded ops: ((dx*dx) + dy*dy) + dz*dz  (nanoflann.hpp:432-440)."""
    d = (q.astype(np.float32) - s.astype(np.float32)).astype(np.float32)
    r = (d[..., 0] * d[..., 0]).astype(np.float32)
    r = (r + (d[..., 1] * d[..., 1]).astype(np.float32)).astype(np.float32)
    r = (r + (d[..., 2] * d[..., 2]).astype(np.float32)).astype(np.float32)
    return r


def canonicalize_neighbors(neigh, queries, supports, pad_value):
    """Re-order every row by (d2, index); padding stays at the end. Returns (canonical, n_rows_changed)."""
    neigh = np.asarray(neigh)
    if neigh.size == 0:
        return neigh.copy(), 0
    q, s = _f32(queries), _f32(supports)
    valid = neigh != pad_value
    safe = np.where(valid, neigh, 0)
    d2 = sqdist_f32(q[:, None, :], s[safe])
    d2 = np.where(valid, d2, np.float32(np.inf))
    key_idx = np.where(valid, neigh, np.iinfo(np.int32).max)
    order = np.lexsort((key_idx, d2), axis=1)
    canon = np.take_along_axis(neigh, order, axis=1)
    changed = int(np.any(canon != neigh, axis=1).sum())
    return canon, changed


def sort_rows(a):
    """Lexicographic row sort (canonical order for order-free comparison of point sets)."""
    a = np.asarray(a)
    if a.shape[0] == 0:
        return a, np.zeros((0,), np.int64)
    order = np.lexsort(tuple(a[:, k] for k in range(a.shape[1] - 1, -1, -1)))
    return a[order], order


def digest(a):
    """[shape, sha256 of the C-ordered bytes]: the stored form of a reference output too large to keep as an array
    (tests/golden/reference_digests.json)."""
    a = np.ascontiguousarray(a)
    return [list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()]


def pyramid_digests(pyr):
    """Digests of an input pyramid (kpconv_np.descriptor_input_pyramid form): per level the barycenter bits, the
    stack lengths and the int32 neighbour / pool / upsample matrices."""
    out = []
    for l in range(len(pyr["points"])):
        d = dict(points=digest(_f32(pyr["points"][l]).view(np.uint32)), lengths=_i32(pyr["lengths"][l]).tolist())
        for key in ("neighbors", "pools", "upsamples"):
            d[key] = digest(_i32(pyr[key][l]))
        out.append(d)
    return out
