"""Load the golden fixtures written by make_golden.py (test infrastructure).

Embeddings/biases are regenerated rather than stored: synthetic cases draw them from the
frozen legacy ``RandomState(seed + 1000)`` stream exactly as make_golden.run_case did;
``cagrqc`` rebuilds the shipped 6-decimal pretrain values from integers and fills the rows
absent from the file like the reference's reader does (utils.py:63, ``np.random.rand`` after
``np.random.seed(123)``).  The sha256 stored in the fixture proves the regeneration is exact.
"""
import hashlib
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


class Case(dict):
    __getattr__ = dict.__getitem__


def _sha(*arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.digest()


def load(name):
    z = np.load(os.path.join(HERE, name + ".npz"))
    c = Case({k: z[k] for k in z.files})
    n, d, seed = int(c["n_node"]), int(c["d"]), int(c["seed"])
    rs = np.random.RandomState(seed + 1000)
    if "pretrain_q1e6_bytes" in c:
        b = c["pretrain_q1e6_bytes"].astype(np.int64)          # byte planes of pretrain_q1e6 + 2**23
        q = (b[0] | b[1] << 8 | b[2] << 16) - (1 << 23)
        fill = np.random.RandomState(int(c["pretrain_fill_seed"])).rand(n, d)
        fill[c["pretrain_ids"]] = q.astype(np.float64) / 1e6
        emb_g, emb_d = fill, fill.copy()
    else:
        emb_g = rs.normal(0, 0.5, size=(n, d))
        emb_d = rs.normal(0, 0.5, size=(n, d))
    bias_g = rs.normal(0, 0.3, size=n).astype(np.float32)
    bias_d = rs.normal(0, 0.3, size=n).astype(np.float32)
    assert _sha(emb_g, emb_d, bias_g, bias_d) == c["emb_sha"].tobytes(), "fixture regeneration drifted"
    c.update(emb_g=emb_g, emb_d=emb_d, bias_g=bias_g, bias_d=bias_d, n=n, dim=d, name=name)
    # graph as python lists, exactly as the reference's read_edges produced it
    ptr, flat = c["graph_ptr"], c["graph_flat"]
    c["graph"] = [flat[ptr[i]:ptr[i + 1]].tolist() for i in range(n)]
    return c


def stream(case, n=None):
    """The MT19937 doubles the reference consumed (np.random.seed(seed) in make_golden)."""
    n = int(case["total_draws"]) + 16 if n is None else n
    return np.random.RandomState(int(case["seed"])).random_sample(n)
