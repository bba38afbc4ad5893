"""CPU tests (no GPU): pin the oracles against the reference-generated golden fixtures.

  T0 = oracle/faithful.py  (numpy restatement, reference data structures and RNG stream)
  T1 = oracle/gg_oracle.c  (canonical arithmetic the CUDA kernels replicate)

tests/golden/*.npz come from running the UNMODIFIED reference host code (make_golden.py).
"""
import numpy as np
import pytest

from oracle import canonical as can
from oracle import faithful, updates
from tests.golden import loader


# ----------------------------------------------------------------------------- RNG
def test_philox_known_answers():
    # Random123 kat_vectors, philox4x32-10
    assert can.philox([0, 0, 0, 0], [0, 0]).tolist() == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    ff = 0xffffffff
    assert can.philox([ff, ff, ff, ff], [ff, ff]).tolist() == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert can.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]).tolist() == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_philox_independent_python():
    def ref(ctr, key):
        c, k = list(ctr), list(key)
        for _ in range(10):
            p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
            c = [((p1 >> 32) ^ c[1] ^ k[0]) & 0xffffffff, p1 & 0xffffffff, ((p0 >> 32) ^ c[3] ^ k[1]) & 0xffffffff,
                 p0 & 0xffffffff]
            k = [(k[0] + 0x9E3779B9) & 0xffffffff, (k[1] + 0xBB67AE85) & 0xffffffff]
        return c
    rs = np.random.RandomState(0)
    for _ in range(50):
        ctr = rs.randint(0, 2 ** 32, size=4, dtype=np.uint64).tolist()
        key = rs.randint(0, 2 ** 32, size=2, dtype=np.uint64).tolist()
        assert can.philox(ctr, key).tolist() == ref(ctr, key)


def test_uniform_construction_is_mt19937s():
    # random_sample() = ((a >> 5) * 2^26 + (b >> 6)) / 2^53 from two consecutive 32-bit outputs
    rs = np.random.RandomState(42)
    st = rs.get_state()
    words = np.random.RandomState(42)
    words.set_state(st)
    a, b = (int(x) for x in words.randint(0, 2 ** 32, size=2, dtype=np.uint64))
    assert can.lib().ggo_u53(a, b) == rs.random_sample()


# ----------------------------------------------------------------------------- canonical arithmetic
def test_exp_accuracy_and_edges():
    x = -np.abs(np.random.RandomState(1).normal(0, 12, size=20000)).astype(np.float32)
    x = x[x >= -86]
    got = can.exp_c(x).astype(np.float64)
    want = np.exp(x.astype(np.float64))
    rel = np.abs(got - want) / want
    assert rel.max() < 2.5e-7            # < ~2 ulp
    assert can.exp_c(np.float32(0.0)) == np.float32(1.0)
    assert can.exp_c(np.float32(-86.5)) == 0.0 and can.exp_c(np.float32(-1e30)) == 0.0


def test_dot_matches_float64():
    rs = np.random.RandomState(2)
    for ld in (32, 64, 128, 256):
        a, b = rs.normal(size=ld).astype(np.float32), rs.normal(size=ld).astype(np.float32)
        assert abs(float(can.dot_c(a, b)) - float(a.astype(np.float64) @ b.astype(np.float64))) < 1e-4


def test_choose_is_numpy_legacy_choice():
    """ggo_choose == softmax (utils.py:131-133) + RandomState.choice's cdf/searchsorted, except
    when u falls within fp32 rounding of a cdf edge (then it must be the neighbouring bin)."""
    rs = np.random.RandomState(3)
    mism = 0
    for trial in range(3000):
        n = int(rs.choice([1, 2, 3, 5, 8, 31, 32, 33, 64, 100, 257]))
        s = rs.normal(0, 3, size=n).astype(np.float32)
        u = rs.random_sample()
        p = faithful.softmax(s)
        cdf = p.astype(np.float64).cumsum()
        cdf /= cdf[-1]
        want = int(cdf.searchsorted(u, side="right"))
        got = can.choose(s, u)
        if got != want:
            mism += 1
            assert abs(got - want) == 1 and min(abs(cdf[min(got, want)] - u), 1) < 1e-5
    assert mism <= 2


def test_choose_degenerate_lists():
    assert can.choose(np.float32([3.5]), 0.999999) == 0
    assert can.choose(np.float32([0, 0, 0, 0]), 0.0) == 0
    assert can.choose(np.float32([0, 0, 0, 0]), 0.2500001) == 1
    assert can.choose(np.float32([0, 0, 0, 0]), 0.99999999) == 3
    assert can.choose(np.float32([-200, 0, -200]), 0.5) == 1          # exp underflow -> exact zeros
    big = np.zeros(1000, np.float32)
    assert can.choose(big, 0.5) == 500


# ----------------------------------------------------------------------------- reference golden vectors
def test_window_pairs_docstring_vector():
    # the only golden vector in the reference: graph_gan.py:276-277
    assert faithful.node_pairs_from_path([1, 0, 2, 4, 2], 2) == \
        [[1, 0], [1, 2], [0, 1], [0, 2], [0, 4], [2, 1], [2, 0], [2, 4], [4, 0], [4, 2]]
    c = loader.load("tiny")
    pp, pf, op, of = c.win_paths_ptr, c.win_paths_flat, c.win_pairs_ptr, c.win_pairs_flat
    for k in range(pp.shape[0] - 1):
        got = faithful.node_pairs_from_path(pf[pp[k]:pp[k + 1]].tolist(), 2)
        assert [x for pr in got for x in pr] == of[op[k]:op[k + 1]].tolist()


def test_tree_format_docstring():
    # graph_gan.py:90 + SURVEY section 4: edges 0-1,0-2,1-3,1-2 in file order
    graph = {0: [1, 2], 1: [0, 3, 2], 2: [0, 1], 3: [1]}
    assert faithful.build_trees(graph, [0])[0] == {0: [0, 1, 2], 1: [0, 3], 2: [0], 3: [1]}
    indptr, adj = can.unique_csr([graph[i] for i in range(4)])
    assert can.bfs_parents(indptr, adj, [0])[0].tolist() == [-1, 0, 0, 1]


@pytest.mark.parametrize("name", ["tiny", "rand300", "rand1200"])
def test_t0_reproduces_reference(name):
    c = loader.load(name)
    trees = faithful.build_trees(c.graph, range(c.n))
    if "parent" in c:
        par = np.full((c.n, c.n), -1, np.int32)
        for r in range(c.n):
            for node, lst in trees[r].items():
                if node != r:
                    par[r, node] = lst[0]
        assert np.array_equal(par, c.parent)
    F = faithful.Faithful(c.graph, c.emb_g, c.bias_g, c.emb_d, c.bias_d, rng=np.random.RandomState(int(c.seed)), trees=trees)
    ce, ne, la = F.prepare_data_for_d()
    assert np.array_equal(ce, c.d_center) and np.array_equal(ne, c.d_neighbor) and np.array_equal(la, c.d_labels)
    n1, n2, rw, paths = F.prepare_data_for_g(n_sample_gen=int(c.n_sample_gen), with_paths=True)
    assert len(paths) == int(c.g_n_paths) and len(n1) == int(c.g_n_pairs)
    k = c.g_node_1.shape[0]
    assert np.array_equal(n1[:k], c.g_node_1) and np.array_equal(n2[:k], c.g_node_2)
    assert np.allclose(rw[:k], c.g_reward, rtol=1e-6, atol=1e-7)
    pp, pf = c.g_paths_ptr, c.g_paths_flat
    for i in range(pp.shape[0] - 1):
        assert list(map(int, paths[i])) == pf[pp[i]:pp[i + 1]].tolist()


def _t1_stream(c):
    indptr, adj = can.unique_csr(c.graph)
    pptr, pflat = can.raw_csr(c.graph)
    roots = np.arange(c.n, dtype=np.int32)
    par = can.bfs_parents(indptr, adj, roots)
    E = can.pad_rows(c.emb_g)
    bits = np.zeros((adj.shape[0] + 31) // 32 + 1, np.uint32)
    st = loader.stream(c)
    r = can.walk_pass(E, c.bias_g, indptr, adj, roots, par, np.diff(pptr), True, bits, rng_mode=can.RNG_STREAM, stream=st)
    return indptr, adj, pptr, pflat, roots, par, E, bits, st, r


@pytest.mark.parametrize("name", ["tiny", "rand300", "rand1200", "cagrqc"])
def test_t1_reproduces_reference_on_its_stream(name):
    """Canonical oracle fed the very MT19937 doubles the reference consumed: D rows, the number of
    draws, the set of mutated depth-1 lists, and the G-pass paths must all be the reference's."""
    c = loader.load(name)
    indptr, adj, pptr, pflat, roots, par, E, bits, st, r = _t1_stream(c)
    if "parent" in c:
        assert np.array_equal(par, c.parent)
    ce, ne, la = can.d_rows(r, roots, pptr, pflat)
    assert np.array_equal(ce, c.d_center) and np.array_equal(ne, c.d_neighbor) and np.array_equal(la, c.d_labels)
    assert r.consumed == int(c.d_draws) and r.steps == int(c.d_steps)
    assert r.sum_l == int(c.d_sum_l)
    mut = set()
    for rr in range(c.n):
        for e in range(indptr[rr], indptr[rr + 1]):
            if (bits[e >> 5] >> (e & 31)) & 1:
                mut.add((rr, int(adj[e])))
    assert mut == set(map(tuple, c.mutated.tolist()))
    r2 = can.walk_pass(E, c.bias_g, indptr, adj, roots, par, np.full(c.n, int(c.n_sample_gen)), False, bits,
                       rng_mode=can.RNG_STREAM, stream=st[r.consumed:], max_path=48)
    assert r.consumed + r2.consumed == int(c.total_draws) and r2.path_overflow == 0
    paths = can.paths_list(r2)
    assert len(paths) == int(c.g_n_paths)
    pp, pf = c.g_paths_ptr, c.g_paths_flat
    for i in range(pp.shape[0] - 1):
        assert paths[i] == pf[pp[i]:pp[i + 1]].tolist()
    # every pair the reference derived from those paths (sha over the full list)
    n1, n2 = [], []
    for p in paths:
        for a, b in faithful.node_pairs_from_path(p, int(c.window_size)):
            n1.append(a); n2.append(b)
    assert len(n1) == int(c.g_n_pairs)
    assert loader._sha(np.asarray(n1, np.int32), np.asarray(n2, np.int32)) == c.g_pairs_sha.tobytes()


@pytest.mark.parametrize("name", ["rand300", "cagrqc"])
def test_t1_teacher_forced_steps(name):
    """Per recorded reference step (candidate list, uniform) the canonical softmax/CDF picks the
    reference's node -- measured, not assumed: report the flip rate, require it tiny."""
    c = loader.load(name)
    E = can.pad_rows(c.emb_g)
    st = loader.stream(c)
    cp, cf, ch, sd = c.dtr_cand_ptr, c.dtr_cand_flat, c.dtr_chosen, c.dtr_step_draw
    # the walk position `cur` of each step is the previous chosen node or the root: recover it from the
    # canonical pass instead (same stream => same steps), here only the choice given scores is checked
    indptr, adj, pptr, pflat, roots, par, E, bits, st, r = _t1_stream(c)
    flips = 0
    # rebuild per-step cur by replaying reference order: root changes when a per-root draw happened
    root_draws = set(c.dtr_root_draw.tolist())
    order = sorted([(int(d), "root") for d in c.dtr_root_draw] + [(int(d), "step", k) for k, d in enumerate(sd)])
    root, cur, prev = -1, -1, -1
    for item in order:
        if item[1] == "root":
            root += 1; cur = root; prev = -1
            continue
        k = item[2]
        cand = cf[cp[k]:cp[k + 1]]
        sc = np.asarray([can.dot_c(E[cur], E[v]) + c.bias_g[v] for v in cand], np.float32)
        got = int(cand[can.choose(sc, st[sd[k]])])
        flips += got != int(ch[k])
        nxt = int(ch[k])
        if nxt == prev:
            cur, prev = root, -1      # walk ended; next walk restarts at the root
        else:
            prev, cur = cur, nxt
    assert flips == 0


# ----------------------------------------------------------------------------- update oracle
def test_update_oracle_gradients_match_autograd():
    import torch
    rs = np.random.RandomState(5)
    n, d, B = 40, 12, 16
    emb = rs.normal(0, 0.5, size=(n, d))
    i, j = rs.randint(0, n, B), rs.randint(0, n, B)
    i[3], j[3] = i[0], j[0]      # duplicates
    j[5] = i[5]                  # self pair
    lab = (rs.random_sample(B) < 0.5).astype(np.float32)
    rew = rs.random_sample(B).astype(np.float32) * 3
    bias0 = rs.normal(0, 0.2, n).astype(np.float32)
    for kind in ("d", "g"):
        M = (updates.Discriminator if kind == "d" else updates.Generator)(n, emb, 1e-3, 1e-2, bias0)
        rows, g_rows, g_bias = M.grads(i, j, lab if kind == "d" else rew)
        E = torch.tensor(M.E, dtype=torch.float64, requires_grad=True)
        b = torch.tensor(M.b, dtype=torch.float64, requires_grad=True)
        ti, tj = torch.tensor(i), torch.tensor(j)
        s = (E[ti] * E[tj]).sum(1) + b[tj]
        if kind == "d":
            loss = torch.nn.functional.binary_cross_entropy_with_logits(s, torch.tensor(lab, dtype=torch.float64), reduction="sum") \
                + 1e-2 * 0.5 * ((E[tj] ** 2).sum() + (E[ti] ** 2).sum() + (b[tj] ** 2).sum())
        else:
            p = torch.clamp(torch.sigmoid(s), 1e-5, 1.0)
            loss = -(torch.log(p) * torch.tensor(rew, dtype=torch.float64)).mean() + 1e-2 * 0.5 * ((E[tj] ** 2).sum() + (E[ti] ** 2).sum())
        loss.backward()
        dense = np.zeros((n, d)); dense[rows] = g_rows
        dbias = np.zeros(n); dbias[rows] = g_bias
        assert np.allclose(dense, E.grad.numpy(), rtol=1e-4, atol=1e-6)
        assert np.allclose(dbias, b.grad.numpy(), rtol=1e-4, atol=1e-6)
        assert abs(M.loss(i, j, lab if kind == "d" else rew) - float(loss)) < 1e-6 * max(1, abs(float(loss)))


def test_update_oracle_adam_is_dense_decay():
    rs = np.random.RandomState(6)
    n, d = 10, 4
    M = updates.Discriminator(n, rs.normal(size=(n, d)), 1e-3, 1e-5)
    E0 = M.E.copy()
    M.d_updates([1, 2], [3, 4], [1, 0])
    touched = {1, 2, 3, 4}
    for r in range(n):
        assert (not np.array_equal(M.E[r], E0[r])) == (r in touched)
    E1 = M.E.copy()
    M.d_updates([5], [6], [1])          # rows 1..4 are NOT in this batch but keep moving (momentum decay)
    for r in (1, 2, 3, 4):
        assert not np.array_equal(M.E[r], E1[r])
    for r in (0, 7, 8, 9):
        assert np.array_equal(M.E[r], E0[r])
    # first step of Adam moves every touched coordinate by ~lr (sign of the gradient)
    assert np.allclose(np.abs(E1[[1, 2, 3, 4]] - E0[[1, 2, 3, 4]]), 1e-3, rtol=1e-3)
