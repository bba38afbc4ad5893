#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/ by running the UNMODIFIED reference.

Needs a checkout of the reference (hwwang55/GraphGAN); the tests only read the fixtures:

    python tests/golden/make_golden.py <reference checkout>

What runs: the reference's own host half -- ``GraphGAN.construct_trees``, ``sample``,
``prepare_data_for_d``, ``prepare_data_for_g``, ``get_node_pairs_from_path``
(src/GraphGAN/graph_gan.py:84-108, 182-291) and ``utils.read_edges`` /
``utils.softmax`` (src/utils.py:12-47, 131-133) -- imported from the
reference checkout, never copied.  TensorFlow 1.8 is not installed, so a stub
``tensorflow`` module satisfies the import and a stub session answers the two fetches the
sampling code makes (``generator.all_score`` = fp32 E.E^T + b, generator.py:21;
``discriminator.reward`` = log(1+exp(clip(score,-10,10))), discriminator.py:21-24,33-34)
with numpy.  Consequently the *control flow, RNG consumption, candidate order and tree
mutation* in these fixtures are the reference's; the dense arithmetic is numpy's.

``np.random.choice`` / ``np.random.rand`` are wrapped (not replaced) to record a per-step
trace: (candidate list, chosen node) plus the index of the uniform double consumed.
"""
import hashlib
import os
import sys
import tempfile
import types

import numpy as np

REF = None  # the reference checkout, set by main() from the command line
OUT = os.path.dirname(os.path.abspath(__file__))


# ----------------------------------------------------------------------------- reference import
def import_reference():
    tf = types.ModuleType("tensorflow")  # import-time stub only; no TF op is ever executed
    sys.modules["tensorflow"] = tf
    for p in (REF, os.path.join(REF, "src", "GraphGAN")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import graph_gan  # noqa: E402  (the reference module, unmodified)
    from src import utils as ref_utils  # noqa: E402
    return graph_gan, ref_utils


class Handle:
    def __init__(self, name):
        self.name = name


class StubModel:
    """Stand-in for generator.Generator / discriminator.Discriminator attribute handles."""

    def __init__(self, emb64):
        self.E = np.asarray(emb64, dtype=np.float64).astype(np.float32)  # tf fp32 variable
        self.b = np.zeros(self.E.shape[0], dtype=np.float32)
        self.all_score = Handle("all_score")
        self.reward = Handle("reward")
        self.node_id = Handle("node_id")
        self.node_neighbor_id = Handle("node_neighbor_id")
        self._all = None


class StubSession:
    def __init__(self, gen, dis):
        self.gen, self.dis = gen, dis
        self.reward_calls = []

    def run(self, fetch, feed_dict=None):
        if fetch is self.gen.all_score:  # generator.py:21
            if self.gen._all is None:
                self.gen._all = (self.gen.E @ self.gen.E.T + self.gen.b).astype(np.float32)
            return self.gen._all
        if fetch is self.dis.reward:  # discriminator.py:21-24, 33-34
            i = np.asarray(feed_dict[self.dis.node_id], dtype=np.int64)
            j = np.asarray(feed_dict[self.dis.node_neighbor_id], dtype=np.int64)
            if i.size == 0:
                return np.zeros(0, np.float32)
            s = np.sum(self.dis.E[i] * self.dis.E[j], axis=1, dtype=np.float32) + self.dis.b[j]
            s = np.clip(s, -10, 10).astype(np.float32)
            r = np.log(np.float32(1) + np.exp(s)).astype(np.float32)
            self.reward_calls.append((i.copy(), j.copy(), r.copy()))
            return r
        raise KeyError(fetch)


class Recorder:
    """Wraps np.random.choice / rand so every consumed uniform is indexed."""

    def __init__(self):
        self.draws = 0
        self.step_draw = []   # draw index used by each choice call
        self.cand_flat = []
        self.cand_ptr = [0]
        self.chosen = []
        self.root_draw = []   # draw index of each per-root rand()
        self._choice = np.random.choice
        self._rand = np.random.rand

    def install(self):
        rec = self

        def choice(a, size=None, replace=True, p=None):
            out = rec._choice(a, size=size, replace=replace, p=p)
            rec.step_draw.append(rec.draws)
            rec.draws += 1
            rec.cand_flat.extend(int(x) for x in a)
            rec.cand_ptr.append(len(rec.cand_flat))
            rec.chosen.append(int(out[0]))
            return out

        def rand(*shape):
            assert shape == ()
            rec.root_draw.append(rec.draws)
            rec.draws += 1
            return rec._rand()

        np.random.choice = choice
        np.random.rand = rand

    def uninstall(self):
        np.random.choice = self._choice
        np.random.rand = self._rand

    def arrays(self, prefix, steps=None):
        """The trace; ``steps`` keeps only the first steps (the per-root draws stay complete)."""
        k = len(self.chosen) if steps is None else min(steps, len(self.chosen))
        return {
            prefix + "step_draw": np.asarray(self.step_draw[:k], np.int64),
            prefix + "cand_flat": np.asarray(self.cand_flat[:self.cand_ptr[k]], np.int32),
            prefix + "cand_ptr": np.asarray(self.cand_ptr[:k + 1], np.int64),
            prefix + "chosen": np.asarray(self.chosen[:k], np.int32),
            prefix + "root_draw": np.asarray(self.root_draw, np.int64),
        }


def write_edges(path, edges):
    with open(path, "w") as f:
        for a, b in edges:
            f.write("%d\t%d\n" % (a, b))


def trees_to_parent(trees, n):
    """reference dict trees -> parent[R, N] (root slot and unreachable = -1)."""
    par = np.full((len(trees), n), -1, np.int32)
    for r in range(len(trees)):
        for node, lst in trees[r].items():
            if node != r:
                par[r, node] = lst[0]
    return par


def graph_to_lists(graph, n):
    ptr = [0]
    flat = []
    for i in range(n):
        flat.extend(graph.get(i, []))
        ptr.append(len(flat))
    return np.asarray(ptr, np.int64), np.asarray(flat, np.int32)


def flatten_paths(paths):
    ptr = [0]
    flat = []
    for p in paths:
        flat.extend(int(x) for x in p)
        ptr.append(len(flat))
    return np.asarray(flat, np.int32), np.asarray(ptr, np.int64)


def sha(*arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def run_case(gg_mod, ref_utils, name, train_edges, test_edges, d, seed, emb=None, trace_g=True,
             keep_parent=True, n_sample_gen=None, extra=None, d_trace_steps=None):
    import config as ref_config  # the reference's config module
    tmp = tempfile.mkdtemp()
    trf, tef = os.path.join(tmp, "train.txt"), os.path.join(tmp, "test.txt")
    write_edges(trf, train_edges)
    write_edges(tef, test_edges)
    n_node, graph = ref_utils.read_edges(trf, tef)  # utils.py:12-47

    rs = np.random.RandomState(seed + 1000)
    if emb is None:
        emb_g = rs.normal(0, 0.5, size=(n_node, d))
        emb_d = rs.normal(0, 0.5, size=(n_node, d))
    else:
        emb_g, emb_d = emb
    bias_g = (rs.normal(0, 0.3, size=n_node)).astype(np.float32)  # exercise the "+ b_j" column broadcast
    bias_d = (rs.normal(0, 0.3, size=n_node)).astype(np.float32)

    obj = gg_mod.GraphGAN.__new__(gg_mod.GraphGAN)
    obj.n_node, obj.graph = n_node, graph
    obj.root_nodes = [i for i in range(n_node)]
    for i in range(n_node):  # read_edges only creates keys for nodes that appear; all ids < n_node do here
        assert i in graph, "fixture graphs must use contiguous ids"
    obj.trees = obj.construct_trees(obj.root_nodes)  # graph_gan.py:84-108
    parent0 = trees_to_parent(obj.trees, n_node)
    gen, dis = StubModel(emb_g), StubModel(emb_d)
    gen.b[:] = bias_g
    dis.b[:] = bias_d
    obj.generator, obj.discriminator = gen, dis
    obj.sess = StubSession(gen, dis)
    if n_sample_gen is not None:
        ref_config.n_sample_gen = n_sample_gen

    stream = np.random.RandomState(seed).random_sample(4_000_000)
    np.random.seed(seed)
    # ---- D pass (graph_gan.py:182-202), then G pass (204-223) on the mutated trees
    rec_d = Recorder(); rec_d.install()
    center, neighbor, labels = obj.prepare_data_for_d()
    rec_d.uninstall()
    # which depth-1 lists lost their father entry (graph_gan.py:258-259 side effect)
    mutated = [(r, c) for r in range(n_node) for c in obj.trees[r][r][1:]
               if obj.trees[r][c][0] != r]
    rec_g = Recorder(); rec_g.install()
    rec_g.draws = rec_d.draws
    # capture paths: prepare_data_for_g discards them, so wrap sample
    all_paths = []
    orig_sample = obj.sample

    def sample_spy(root, tree, sample_num, for_d):
        s, p = orig_sample(root, tree, sample_num, for_d)
        if p is not None:
            all_paths.extend([list(map(int, q)) for q in p])
        return s, p

    obj.sample = sample_spy
    node_1, node_2, reward = obj.prepare_data_for_g()
    rec_g.uninstall()
    obj.sample = orig_sample
    total_draws = rec_g.draws
    # sanity: exactly one MT19937 double per rand()/choice call
    assert np.random.random_sample() == stream[total_draws], "RNG accounting broken"

    pos_ptr, pos_flat = graph_to_lists(graph, n_node)
    pflat, pptr = flatten_paths(all_paths)
    out = {
        "n_node": np.int64(n_node), "d": np.int64(d), "seed": np.int64(seed),
        "train_edges": np.asarray(train_edges, np.int32).reshape(-1, 2),
        "test_edges": np.asarray(test_edges, np.int32).reshape(-1, 2),
        "graph_ptr": pos_ptr, "graph_flat": pos_flat,
        # embeddings/biases are NOT stored: tests/golden/loader.py regenerates them from
        # RandomState(seed + 1000) (synthetic cases) or from pretrain_q1e6 (cagrqc)
        "emb_sha": np.frombuffer(bytes.fromhex(sha(np.asarray(emb_g, np.float64), np.asarray(emb_d, np.float64),
                                                   bias_g, bias_d)), np.uint8),
        "d_center": np.asarray(center, np.int32), "d_neighbor": np.asarray(neighbor, np.int32),
        "d_labels": np.asarray(labels, np.int32),
        "d_draws": np.int64(rec_d.draws), "total_draws": np.int64(total_draws),
        "d_steps": np.int64(len(rec_d.chosen)), "d_sum_l": np.int64(rec_d.cand_ptr[-1]),
        "mutated": np.asarray(mutated, np.int32).reshape(-1, 2),
        "g_n_pairs": np.int64(len(node_1)),
        "g_pairs_sha": np.frombuffer(bytes.fromhex(sha(np.asarray(node_1, np.int32), np.asarray(node_2, np.int32))),
                                     np.uint8),
        "g_n_paths": np.int64(len(all_paths)),
        "g_paths_sha": np.frombuffer(bytes.fromhex(sha(pflat, pptr)), np.uint8),
        "n_sample_gen": np.int64(ref_config.n_sample_gen),
        "window_size": np.int64(ref_config.window_size),
    }
    if keep_parent:
        out["parent"] = parent0
    out.update(rec_d.arrays("dtr_", d_trace_steps))
    if trace_g:
        out.update(rec_g.arrays("gtr_"))
        out["g_paths_flat"], out["g_paths_ptr"] = pflat, pptr
        out["g_node_1"], out["g_node_2"] = np.asarray(node_1, np.int32), np.asarray(node_2, np.int32)
        out["g_reward"] = np.asarray(reward, np.float32)
    else:
        keep = min(len(all_paths), 2000)
        out["g_paths_flat"], out["g_paths_ptr"] = flatten_paths(all_paths[:keep])
        out["g_node_1"], out["g_node_2"] = np.asarray(node_1[:4096], np.int32), np.asarray(node_2[:4096], np.int32)
        out["g_reward"] = np.asarray(reward[:4096], np.float32)
    if extra:
        out.update(extra)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print("%-14s N=%d d=%d  D rows=%d (steps %d)  G paths=%d pairs=%d  mutated=%d  draws=%d" % (
        name, n_node, d, len(center), len(rec_d.chosen), len(all_paths), len(node_1), len(mutated), total_draws))


def tiny_graph():
    # hand-checkable: hub 0; depth-1 leaf (node 5: voids root 0 if visited); self-loop on 3;
    # a duplicated edge (1,2)/(2,1); node 9 isolated (appears only in the test file);
    # node 10 has only a self-loop; a path tail 6-7-8 for depth.
    train = [(0, 1), (0, 2), (1, 3), (1, 2), (3, 3), (2, 4), (0, 5), (4, 6), (6, 7), (7, 8),
             (2, 1), (10, 10), (3, 4), (11, 8), (11, 7)]
    test = [(9, 0), (4, 8)]
    return train, test


def random_graph(n, m, seed):
    rs = np.random.RandomState(seed)
    e = rs.randint(0, n, size=(m, 2))
    # keep self-loops and duplicates: the reference's reader keeps them too (utils.py:36-37)
    edges = [(int(a), int(b)) for a, b in e]
    present = set(x for ab in edges for x in ab)
    test = [(i, (i + 1) % n) for i in range(n) if i not in present]  # test-only => isolated in train
    if not test:
        test = [(0, 1)]
    return edges, test


def main():
    global REF
    if len(sys.argv) != 2:
        sys.exit("usage: make_golden.py <reference checkout>")
    REF = os.path.abspath(sys.argv[1])
    gg_mod, ref_utils = import_reference()
    # (1) the only golden vector in the reference: graph_gan.py:276-277
    import config as ref_config
    assert ref_config.window_size == 2
    pairs = gg_mod.GraphGAN.get_node_pairs_from_path([1, 0, 2, 4, 2])
    assert pairs == [[1, 0], [1, 2], [0, 1], [0, 2], [0, 4], [2, 1], [2, 0], [2, 4], [4, 0], [4, 2]]
    rs = np.random.RandomState(7)
    win_paths = [[int(x) for x in rs.randint(0, 50, size=rs.randint(2, 14))] for _ in range(64)]
    win_out = [gg_mod.GraphGAN.get_node_pairs_from_path(p) for p in win_paths]
    wflat, wptr = flatten_paths(win_paths)
    oflat, optr = flatten_paths([[x for pr in o for x in pr] for o in win_out])
    extra = {"win_paths_flat": wflat, "win_paths_ptr": wptr, "win_pairs_flat": oflat, "win_pairs_ptr": optr}

    tr, te = tiny_graph()
    run_case(gg_mod, ref_utils, "tiny", tr, te, d=8, seed=11, n_sample_gen=6, extra=extra)
    ref_config.n_sample_gen = 20
    tr, te = random_graph(300, 620, seed=3)
    run_case(gg_mod, ref_utils, "rand300", tr, te, d=16, seed=5, n_sample_gen=8)
    ref_config.n_sample_gen = 20
    tr, te = random_graph(1200, 4200, seed=4)
    run_case(gg_mod, ref_utils, "rand1200", tr, te, d=50, seed=6, trace_g=False, keep_parent=False, n_sample_gen=5)
    ref_config.n_sample_gen = 20

    # (3) config C1: the shipped CA-GrQc graph + shipped pretrain embeddings
    ddir = os.path.join(REF, "data", "link_prediction")
    train = ref_utils.read_edges_from_file(os.path.join(ddir, "CA-GrQc_train.txt"))
    test = ref_utils.read_edges_from_file(os.path.join(ddir, "CA-GrQc_test.txt"))
    test_neg = ref_utils.read_edges_from_file(os.path.join(ddir, "CA-GrQc_test_neg.txt"))
    n_node = len(set(x for e in train + test for x in e))
    np.random.seed(123)  # read_embeddings fills missing rows from the global RNG (utils.py:63)
    pre = ref_utils.read_embeddings(os.path.join(REF, "pre_train", "link_prediction", "CA-GrQc_pre_train.emb"),
                                    n_node=n_node, n_embed=50)
    # store the file's 6-decimal values exactly as integers; rows absent from the file are
    # flagged (the reference fills them with np.random.rand, which is seed dependent)
    with open(os.path.join(REF, "pre_train", "link_prediction", "CA-GrQc_pre_train.emb")) as f:
        lines = f.readlines()[1:]
    ids = np.asarray([int(l.split()[0]) for l in lines], np.int32)
    q = np.asarray([[int(round(float(x) * 1e6)) for x in l.split()[1:]] for l in lines], np.int32)
    assert np.array_equal(q.astype(np.float64) / 1e6, pre[ids])
    # rows in id order; q + 2**23 fits 24 bits and is stored as its three little-endian byte planes, which
    # compress ~20 % smaller than int32 (the fixture stays below 1 MB; tests/golden/loader.py unpacks them)
    order = np.argsort(ids)
    ids, u = ids[order], q[order].astype(np.int64) + (1 << 23)
    assert u.min() >= 0 and u.max() < (1 << 24)
    planes = np.stack([(u >> s) & 255 for s in (0, 8, 16)]).astype(np.uint8)
    extra = {"test_neg_edges": np.asarray(test_neg, np.int32), "pretrain_ids": ids, "pretrain_q1e6_bytes": planes,
             "pretrain_fill_seed": np.int64(123)}
    # the D-pass trace is cut to the 6002 steps test_t1_teacher_forced_steps replays; d_steps / d_sum_l keep its totals
    run_case(gg_mod, ref_utils, "cagrqc", [tuple(e) for e in train], [tuple(e) for e in test], d=50, seed=2024,
             emb=(pre, pre.copy()), trace_g=False, keep_parent=False, extra=extra, d_trace_steps=6002)


if __name__ == "__main__":
    main()
