"""oracle/canonical.py -- TEST INFRASTRUCTURE ONLY: ctypes front-end of the canonical C oracle
(tier "T1", oracle/gg_oracle.c; contract in oracle/gg_oracle.h).

The walk follows src/GraphGAN/graph_gan.py:182-270 with the arithmetic pinned down so the
CUDA kernels can be compared bit-for-bit.  Never imported by graphgan_b200/.
"""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

NOTRUN, DONE, VOID, SKIPPED = 0, 1, 2, 3
RNG_PHILOX, RNG_STREAM = 0, 1


def _source_hash():
    h = hashlib.sha256()
    for f in ("gg_oracle.c", "gg_oracle.h", "Makefile"):
        h.update(f.encode())
        with open(os.path.join(HERE, f), "rb") as src:
            h.update(src.read())
    return h.hexdigest()


def build(force=False):
    """Rebuild libgg_oracle.so when it is missing or was built from other sources.  The sources' content hash is
    kept in a sidecar file, not their mtimes: a copied tree has new mtimes, and may be read-only."""
    so = os.path.join(HERE, "libgg_oracle.so")
    stamp = so + ".hash"
    want = _source_hash()
    if not force and os.path.exists(so) and os.path.exists(stamp):
        with open(stamp) as f:
            if f.read().strip() == want:
                return so
    subprocess.check_call(["make", "-C", HERE, "-s", "-B", "libgg_oracle.so"])
    with open(stamp, "w") as f:
        f.write(want + "\n")
    return so


class _Args(C.Structure):
    _fields_ = [
        ("n_node", C.c_int64), ("ld", C.c_int32),
        ("emb", C.c_void_p), ("bias", C.c_void_p), ("indptr", C.c_void_p), ("adj", C.c_void_p),
        ("n_roots", C.c_int64), ("roots", C.c_void_p), ("parent", C.c_void_p), ("walk_ptr", C.c_void_p),
        ("for_d", C.c_int32), ("d1_bits", C.c_void_p), ("rng_mode", C.c_int32), ("seed", C.c_uint64),
        ("pass_tag", C.c_uint32), ("stream", C.c_void_p), ("n_stream", C.c_int64), ("update_ratio", C.c_double),
        ("max_path", C.c_int32),
        ("samples", C.c_void_p), ("status", C.c_void_p), ("first_edge", C.c_void_p), ("wsteps", C.c_void_p),
        ("wsuml", C.c_void_p), ("paths", C.c_void_p), ("path_len", C.c_void_p), ("root_ok", C.c_void_p),
        ("counters", C.c_void_p),
    ]


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.ggo_exp.restype = C.c_float
        _LIB.ggo_exp.argtypes = [C.c_float]
        _LIB.ggo_dot.restype = C.c_float
        _LIB.ggo_dot.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        _LIB.ggo_u53.restype = C.c_double
        _LIB.ggo_u53.argtypes = [C.c_uint32, C.c_uint32]
        _LIB.ggo_choose.restype = C.c_int
        _LIB.ggo_choose.argtypes = [C.c_void_p, C.c_int, C.c_double]
        _LIB.ggo_bfs_parent.restype = C.c_int64
        _LIB.ggo_bfs_parent.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        _LIB.ggo_walk_pass.restype = C.c_int
        _LIB.ggo_walk_pass.argtypes = [C.POINTER(_Args)]
        _LIB.ggo_philox4x32_10.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


# ----------------------------------------------------------------------------- small helpers
def round_up(x, m):
    return (x + m - 1) // m * m


def pad_rows(emb, ld=None):
    """[N, d] (any float) -> contiguous fp32 [N, ld], ld = round_up(d, 32), zero padded."""
    e = np.asarray(emb, np.float64).astype(np.float32)
    n, d = e.shape
    ld = round_up(d, 32) if ld is None else ld
    out = np.zeros((n, ld), np.float32)
    out[:, :d] = e
    return out


def unique_csr(graph):
    """graph: sequence node -> list of neighbours (raw, file order, with duplicates/self-loops
    as utils.py:27-37 produces).  Returns the walking CSR: first occurrences only, self-loops
    dropped -- exactly the entries the BFS of graph_gan.py:93-107 can ever turn into children."""
    indptr = np.zeros(len(graph) + 1, np.int64)
    flat = []
    for i, nb in enumerate(graph):
        seen = {i}
        for v in nb:
            v = int(v)
            if v not in seen:
                seen.add(v)
                flat.append(v)
        indptr[i + 1] = len(flat)
    return indptr, np.asarray(flat, np.int32)


def raw_csr(graph):
    indptr = np.zeros(len(graph) + 1, np.int64)
    flat = []
    for i, nb in enumerate(graph):
        flat.extend(int(v) for v in nb)
        indptr[i + 1] = len(flat)
    return indptr, np.asarray(flat, np.int32)


def philox(ctr, key):
    c = np.asarray(ctr, np.uint32)
    k = np.asarray(key, np.uint32)
    o = np.zeros(4, np.uint32)
    lib().ggo_philox4x32_10(_p(c), _p(k), _p(o))
    return o


def exp_c(x):
    return np.asarray([lib().ggo_exp(float(np.float32(v))) for v in np.ravel(x)], np.float32).reshape(np.shape(x))


def dot_c(a, b):
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    return np.float32(lib().ggo_dot(_p(a), _p(b), a.shape[0]))


def choose(scores, u):
    s = np.array(scores, np.float32, copy=True)
    return int(lib().ggo_choose(_p(s), s.shape[0], float(u)))


def bfs_parents(indptr, adj, roots):
    n = indptr.shape[0] - 1
    roots = np.asarray(roots, np.int32)
    out = np.empty((roots.shape[0], n), np.int32)
    q = np.empty(n, np.int32)
    for k, r in enumerate(roots):
        lib().ggo_bfs_parent(n, _p(indptr), _p(adj), int(r), _p(out[k]), _p(q))
    return out


class WalkResult(dict):
    __getattr__ = dict.__getitem__


def walk_pass(emb_padded, bias, indptr, adj, roots, parent, sample_num, for_d, d1_bits, *, rng_mode=RNG_PHILOX,
              seed=0, pass_tag=0, stream=None, update_ratio=1.0, max_path=0):
    """One sampling pass over ``roots`` in order.  d1_bits (uint32, one bit per CSR entry) is
    updated in place in D mode and read in G mode."""
    emb_padded = np.ascontiguousarray(emb_padded, np.float32)
    bias = np.ascontiguousarray(bias, np.float32)
    roots = np.ascontiguousarray(roots, np.int32)
    parent = np.ascontiguousarray(parent, np.int32)
    n = indptr.shape[0] - 1
    assert parent.shape == (roots.shape[0], n)
    walk_ptr = np.zeros(roots.shape[0] + 1, np.int64)
    walk_ptr[1:] = np.cumsum(np.asarray(sample_num, np.int64))
    W = int(walk_ptr[-1])
    res = WalkResult(
        samples=np.full(W, -1, np.int32), status=np.zeros(W, np.int32), first_edge=np.full(W, -1, np.int32),
        wsteps=np.zeros(W, np.int32), wsuml=np.zeros(W, np.int32),
        paths=np.full((W, max(max_path, 1)), -1, np.int32), path_len=np.zeros(W, np.int32),
        root_ok=np.zeros(roots.shape[0], np.int32), counters=np.zeros(8, np.int64), walk_ptr=walk_ptr)
    st = None if stream is None else np.ascontiguousarray(stream, np.float64)
    a = _Args(n_node=n, ld=emb_padded.shape[1], emb=_p(emb_padded), bias=_p(bias), indptr=_p(indptr), adj=_p(adj),
              n_roots=roots.shape[0], roots=_p(roots), parent=_p(parent), walk_ptr=_p(walk_ptr), for_d=int(for_d),
              d1_bits=_p(d1_bits), rng_mode=rng_mode, seed=seed, pass_tag=pass_tag, stream=_p(st),
              n_stream=0 if st is None else st.shape[0], update_ratio=float(update_ratio), max_path=max_path,
              samples=_p(res.samples), status=_p(res.status), first_edge=_p(res.first_edge), wsteps=_p(res.wsteps),
              wsuml=_p(res.wsuml), paths=_p(res.paths), path_len=_p(res.path_len), root_ok=_p(res.root_ok),
              counters=_p(res.counters))
    rc = lib().ggo_walk_pass(C.byref(a))
    if rc != 0:
        raise RuntimeError("ggo_walk_pass failed rc=%d" % rc)
    res["steps"], res["sum_l"], res["consumed"] = (int(x) for x in res.counters[:3])
    res["path_overflow"], res["max_l"] = int(res.counters[3]), int(res.counters[4])
    return res


def d_rows(res, roots, pos_indptr, pos_flat):
    """Assemble prepare_data_for_d's three lists (graph_gan.py:192-201) from a D-mode WalkResult."""
    center, neighbor, labels = [], [], []
    for k, r in enumerate(np.asarray(roots)):
        if res.root_ok[k]:
            pos = pos_flat[pos_indptr[r]:pos_indptr[r + 1]]
            neg = res.samples[res.walk_ptr[k]:res.walk_ptr[k + 1]]
            center.extend([int(r)] * len(pos)); neighbor.extend(pos.tolist()); labels.extend([1] * len(pos))
            center.extend([int(r)] * len(pos)); neighbor.extend(neg.tolist()); labels.extend([0] * len(neg))
    return np.asarray(center, np.int32), np.asarray(neighbor, np.int32), np.asarray(labels, np.int32)


def paths_list(res):
    out = []
    for w in range(res.samples.shape[0]):
        if res.status[w] == DONE:
            out.append(res.paths[w, :res.path_len[w]].tolist())
    return out
