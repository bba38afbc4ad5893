"""GPU parity of K1 (walk sampler) and the BFS-tree builder against the oracles.

Everything goes through the C ABI (graphgan_b200._cabi -> libgraphgan_b200.so).  Bars:
bit-exact node indices, statuses, root_ok flags, tree-mutation bits, D rows and paths.
"""
import numpy as np
import pytest

from tests.golden import loader

pytestmark = pytest.mark.gpu


def _setup(case, cuda_device, roots=None, hub_threshold=256, depth1=True):
    import torch
    from graphgan_b200 import graph as G, sampler as S
    from oracle import canonical as can
    edges = case["train_edges"]
    hg = G.HostGraph(edges, case["test_edges"], n_node=case.n)
    assert hg.n_node == case.n
    # host graph == the reference reader's graph (utils.py:12-47)
    ptr, flat = can.raw_csr(case.graph)
    assert np.array_equal(hg.raw_indptr, ptr) and np.array_equal(hg.raw_adj, flat)
    indptr, adj = can.unique_csr(case.graph)
    assert np.array_equal(hg.indptr, indptr) and np.array_equal(hg.adj, adj)
    dg = G.DeviceGraph(hg, cuda_device)
    smp = S.WalkSampler(dg, hub_threshold=hub_threshold, depth1=depth1)
    roots = np.arange(case.n, dtype=np.int32) if roots is None else np.asarray(roots, np.int32)
    trees = smp.build_trees(roots)
    emb = S.pad_embedding(case.emb_g, cuda_device)
    bias = torch.as_tensor(case.bias_g).to(cuda_device)
    return hg, dg, smp, roots, trees, emb, bias


def _bits_to_set(bits, indptr, adj):
    out = set()
    words = np.asarray(bits).view(np.uint32)
    for w in np.flatnonzero(words):
        for b in range(32):
            if (words[w] >> b) & 1:
                e = int(w) * 32 + b
                r = int(np.searchsorted(indptr, e, side="right") - 1)
                out.add((r, int(adj[e])))
    return out


@pytest.mark.parametrize("name", ["tiny", "rand300", "rand1200", "cagrqc"])
def test_bfs_matches_reference_order(name, cuda_device):
    from oracle import canonical as can
    case = loader.load(name)
    rs = np.random.RandomState(1)
    roots = np.arange(case.n) if case.n <= 1200 else np.sort(rs.choice(case.n, 600, replace=False))
    hg, dg, smp, roots, trees, emb, bias = _setup(case, cuda_device, roots)
    got = trees.parent_arrays().cpu().numpy()
    want = can.bfs_parents(hg.indptr, hg.adj, roots)
    assert np.array_equal(got, want)
    if "parent" in case:  # the reference's own dict trees (construct_trees) as parent arrays
        assert np.array_equal(got, case["parent"][roots])


def test_bfs_beyond_the_shared_memory_bitmap(cuda_device):
    """N = 1.8 M nodes: the visited bitmap (N bits) no longer fits in shared memory and lives in the per-CTA global
    scratch (csrc/bfs.cu: bfs_kernel<false>).  Same parents as the sequential FIFO BFS, deep sparse trees included
    (avg degree 3: hundreds of levels of small frontiers)."""
    import torch
    from graphgan_b200 import graph as G, sampler as S, synth
    from oracle import canonical as can
    n = 1_800_000
    edges = synth.power_law(n, 3, seed=9)
    hg = G.HostGraph(edges, None, n_node=n)
    dg = G.DeviceGraph(hg, cuda_device)
    smp = S.WalkSampler(dg)
    roots = synth.pick_roots(hg.degrees(), 6, seed=4)
    trees = smp.build_trees(roots)
    got = trees.parent_arrays().cpu().numpy()
    want = can.bfs_parents(hg.indptr, hg.adj, roots)
    assert np.array_equal(got, want)
    assert (got >= 0).sum() > 6 * 1000            # the roots' components are not trivial


@pytest.mark.parametrize("hub", [0, 8])
@pytest.mark.parametrize("name", ["tiny", "rand300", "rand1200", "cagrqc"])
def test_stream_replay_matches_reference(name, hub, cuda_device):
    """Feed the MT19937 doubles the reference consumed; the GPU must reproduce the reference's
    prepare_data_for_d rows, its tree mutations, and then (G pass on the mutated trees) its paths."""
    import torch
    from graphgan_b200 import sampler as S
    case = loader.load(name)
    hg, dg, smp, roots, trees, emb, bias = _setup(case, cuda_device, hub_threshold=hub)
    st = torch.as_tensor(loader.stream(case)).to(cuda_device)
    out = smp.run(emb, bias, trees, dg.raw_deg, True, rng_mode=S.RNG_STREAM, stream=st)
    c, nb, lb, n_rows = smp.emit_d_rows(out)
    n_rows = int(n_rows.item())
    assert n_rows == case.d_center.shape[0]
    assert np.array_equal(c[:n_rows].cpu().numpy(), case.d_center)
    assert np.array_equal(nb[:n_rows].cpu().numpy(), case.d_neighbor)
    assert np.array_equal(lb[:n_rows].cpu().numpy(), case.d_labels)
    cnt = out.counters_host()
    assert cnt["stream_used"] == int(case.d_draws)
    assert cnt["steps"] == int(case.d_steps)
    assert _bits_to_set(dg.d1_bits.cpu().numpy(), hg.indptr, hg.adj) == set(map(tuple, case.mutated.tolist()))
    # G pass continues on the same stream
    used = cnt["stream_used"]
    out_g = smp.run(emb, bias, trees, int(case.n_sample_gen), False, rng_mode=S.RNG_STREAM, stream=st[used:], max_path=48)
    cg = out_g.counters_host()
    assert cg["path_overflow"] == 0
    assert used + cg["stream_used"] == int(case.total_draws)
    status = out_g.status.cpu().numpy()
    plen = out_g.path_len.cpu().numpy()
    paths = out_g.paths.cpu().numpy()
    got = [paths[w, :plen[w]].tolist() for w in np.flatnonzero(status == S.DONE)]
    assert len(got) == int(case.g_n_paths)
    pp, pf = case.g_paths_ptr, case.g_paths_flat
    for k in range(pp.shape[0] - 1):
        assert got[k] == pf[pp[k]:pp[k + 1]].tolist()


def _philox_compare(case, cuda_device, roots, update_ratio, seed, n_sample_gen, hub_threshold=256, depth1=True):
    import torch
    from graphgan_b200 import sampler as S
    from oracle import canonical as can
    hg, dg, smp, roots, trees, emb, bias = _setup(case, cuda_device, roots, hub_threshold, depth1)
    par = trees.parent_arrays().cpu().numpy()
    E = can.pad_rows(case.emb_g)
    bits = np.zeros(dg.n_bit_words, np.uint32)
    deg = hg.degrees()[roots]
    ref = can.walk_pass(E, case.bias_g, hg.indptr, hg.adj, roots, par, deg, True, bits, seed=seed, pass_tag=3,
                        update_ratio=update_ratio)
    sn = torch.as_tensor(deg.astype(np.int64)).to(cuda_device)
    out = smp.run(emb, bias, trees, sn, True, seed=seed, pass_tag=3, update_ratio=update_ratio)
    assert np.array_equal(out.root_ok.cpu().numpy()[:len(roots)], ref.root_ok)
    assert np.array_equal(out.status.cpu().numpy()[:ref.status.shape[0]], ref.status)
    assert np.array_equal(out.samples.cpu().numpy()[:ref.samples.shape[0]], ref.samples)
    assert np.array_equal(out.wsteps.cpu().numpy()[:ref.wsteps.shape[0]], ref.wsteps)
    assert np.array_equal(out.wsuml.cpu().numpy()[:ref.wsuml.shape[0]], ref.wsuml)
    assert np.array_equal(dg.d1_bits.cpu().numpy().view(np.uint32), bits)
    cnt = out.counters_host()
    assert (cnt["steps"], cnt["sum_l"]) == (ref.steps, ref.sum_l)
    assert cnt["accepted"] == int(sum(deg[k] for k in range(len(roots)) if ref.root_ok[k]))
    c, nb, lb, n_rows = smp.emit_d_rows(out)
    n_rows = int(n_rows.item())
    rc, rn, rl = can.d_rows(ref, roots, hg.raw_indptr, hg.raw_adj)
    assert n_rows == rc.shape[0]
    assert np.array_equal(c[:n_rows].cpu().numpy(), rc) and np.array_equal(nb[:n_rows].cpu().numpy(), rn)
    assert np.array_equal(lb[:n_rows].cpu().numpy(), rl)
    # G pass on the mutated trees
    ref_g = can.walk_pass(E, case.bias_g, hg.indptr, hg.adj, roots, par, np.full(len(roots), n_sample_gen), False, bits,
                          seed=seed, pass_tag=4, update_ratio=update_ratio, max_path=40)
    out_g = smp.run(emb, bias, trees, n_sample_gen, False, seed=seed, pass_tag=4, update_ratio=update_ratio, max_path=40)
    assert np.array_equal(out_g.status.cpu().numpy(), ref_g.status)
    assert np.array_equal(out_g.samples.cpu().numpy(), ref_g.samples)
    assert np.array_equal(out_g.path_len.cpu().numpy(), ref_g.path_len)
    gp, rp = out_g.paths.cpu().numpy(), ref_g.paths
    for w in np.flatnonzero(ref_g.status == can.DONE):
        assert np.array_equal(gp[w, :ref_g.path_len[w]], rp[w, :ref_g.path_len[w]])
    # the start order of the walks (WalkPlan.start_order) must not change anything
    assert smp.hub_first
    smp.hub_first = False
    out2 = smp.run(emb, bias, trees, sn, True, seed=seed, pass_tag=3, update_ratio=update_ratio)
    for name in ("samples", "status", "wsteps", "wsuml", "root_ok", "first_edge"):
        assert torch.equal(getattr(out2, name), getattr(out, name)), name
    cg = out_g.counters_host()
    assert (cg["steps"], cg["sum_l"]) == (ref_g.steps, ref_g.sum_l)
    return cnt, cg


@pytest.mark.parametrize("hub", [0, 8, 256])
@pytest.mark.parametrize("name,ratio", [("tiny", 1.0), ("rand300", 1.0), ("rand300", 0.6), ("rand1200", 1.0), ("cagrqc", 1.0)])
def test_philox_matches_canonical_oracle(name, ratio, hub, cuda_device):
    """hub = 0: every score on demand, root step per walk; hub = 8 / 256: per-pass hub scores and root
    CDFs (csrc/hub.cu).  Identical bits either way."""
    case = loader.load(name)
    _philox_compare(case, cuda_device, None, ratio, seed=0x1234567 + 17, n_sample_gen=int(case.n_sample_gen),
                    hub_threshold=hub)


@pytest.mark.parametrize("name,hub,ratio", [("rand300", 0, 0.6), ("rand1200", 256, 1.0), ("cagrqc", 8, 1.0)])
def test_philox_without_depth1_reuse(name, hub, ratio, cuda_device):
    """One warp per walk WITHOUT the depth-1 CDF reuse agrees bit for bit with the oracle (and so with the default
    path)."""
    case = loader.load(name)
    _philox_compare(case, cuda_device, None, ratio, seed=4242, n_sample_gen=int(case.n_sample_gen), hub_threshold=hub,
                    depth1=False)


@pytest.mark.parametrize("hub", [0, 64, 256])
def test_hub_lists_use_global_scratch(hub, cuda_device):
    """A power-law graph whose hub has > SMEM_CAP neighbours: the long-list (global scratch) path
    and multi-tile softmax must agree bit-for-bit with the oracle as well."""
    from graphgan_b200 import synth
    n, d = 12000, 128
    edges = synth.power_law(n, 20, seed=3)
    case = loader.Case(n=n, dim=d, train_edges=edges, test_edges=np.zeros((0, 2), np.int64),
                       emb_g=synth.embeddings(n, d, seed=5, sigma=0.3), bias_g=np.zeros(n, np.float32))
    from graphgan_b200 import graph as G
    hg = G.HostGraph(edges, None, n_node=n)
    assert hg.max_deg > 400
    case["graph"] = [hg.neighbors(i).tolist() for i in range(n)]
    rs = np.random.RandomState(0)
    roots = np.sort(rs.choice(np.flatnonzero(hg.degrees() > 0), 400, replace=False))
    cnt, cg = _philox_compare(case, cuda_device, roots, 1.0, seed=99, n_sample_gen=6, hub_threshold=hub)
    assert cnt["steps"] > 0
    if hub:   # the reuse must actually remove row gathers
        assert cnt["rows_gathered"] < cnt["raw_sum_l"]


BFS_MODES = {"top_down": (0.0, 0), "default": (-1.0, 0), "bottom_up_forced": (1e9, 1)}


def _trees_in_mode(smp, roots, mode):
    smp.bfs_bottom_up_ratio, smp.bfs_flags = BFS_MODES[mode]
    return smp.build_trees(roots)


def test_reverse_entries_match_numpy(cuda_device):
    """gg_reverse_entries: rev[e] of e = (u -> v) is the index of (v -> u); an asymmetric CSR is reported, not used."""
    import torch
    from graphgan_b200 import graph as G, synth
    n = 20000
    hg = G.HostGraph(synth.power_law(n, 12, seed=21), None, n_node=n)
    dg = G.DeviceGraph(hg, cuda_device)
    rev = dg.reverse_entries()
    assert rev is not None
    rev = rev.cpu().numpy()
    src = np.repeat(np.arange(n), np.diff(hg.indptr))
    assert np.array_equal(hg.adj[rev], src) and np.array_equal(src[rev], hg.adj)
    # one direction of an edge removed: that entry has no reverse
    keep = np.ones(hg.adj.shape[0], bool)
    keep[hg.indptr[5]] = False
    bad = G.HostGraph.from_arrays(n, hg.raw_indptr, hg.raw_adj,
                                  np.concatenate([[0], np.cumsum(np.bincount(src[keep], minlength=n))]), hg.adj[keep])
    assert G.DeviceGraph(bad, cuda_device).reverse_entries() is None


@pytest.mark.parametrize("graph", ["rand1200", "power_law_12k", "hub_30k", "path_tail"])
def test_bfs_bottom_up_levels_build_the_same_trees(graph, cuda_device):
    """The direction-optimising builder (csrc/bfs.cu: bottom_up_level) against the top-down sweep and the FIFO oracle:
    identical tree rows bit for bit, with the bottom-up form forced at every level it can run at (ratio 1e9, the small
    sorted form off), at the library default, and off.  hub_30k: a 30 000-leaf hub two hops from the roots -- more
    undiscovered nodes than one staging round holds (phase A), a frontier node with more children than the child stage
    holds and ~940 words of tree bits (phase B long-node path).  path_tail: hundreds of one-node levels."""
    import torch
    from graphgan_b200 import graph as G, sampler as S, synth
    from oracle import canonical as can
    rs = np.random.RandomState(3)
    if graph == "rand1200":
        case = loader.load("rand1200")
        hg = G.HostGraph(case["train_edges"], case["test_edges"], n_node=case.n)
        roots = np.arange(case.n, dtype=np.int32)
    elif graph == "power_law_12k":
        n = 12000
        hg = G.HostGraph(synth.power_law(n, 10, seed=5), None, n_node=n)
        roots = synth.pick_roots(hg.degrees(), 96, seed=6)
    elif graph == "hub_30k":
        n = 42000
        hub = 7
        leaves = rs.permutation(np.arange(100, 30100))
        star = np.stack([np.full(leaves.shape[0], hub, np.int64), leaves], 1)
        extra = synth.power_law(n, 4, seed=8)
        edges = np.concatenate([star[:9000], extra, star[9000:], np.asarray([[41999, 41998], [41998, hub]])])
        hg = G.HostGraph(edges, None, n_node=n)
        roots = np.asarray([41999, 41998, hub, 100, 20000, 35000], np.int32)
    else:
        n = 5000
        path = np.stack([np.arange(3000, 3400), np.arange(3001, 3401)], 1)
        edges = np.concatenate([synth.power_law(n, 6, seed=11), path, np.asarray([[3000, 17]])])
        hg = G.HostGraph(edges, None, n_node=n)
        roots = np.asarray([3400, 3200, 17, 4000], np.int32)
    dg = G.DeviceGraph(hg, cuda_device)
    assert dg.reverse_entries() is not None
    smp = S.WalkSampler(dg)
    want = can.bfs_parents(hg.indptr, hg.adj, roots)
    rows = {}
    for mode in BFS_MODES:
        t = _trees_in_mode(smp, roots, mode)
        assert np.array_equal(t.parent_arrays().cpu().numpy(), want), mode
        rows[mode] = t.tree_bits.cpu().numpy()
    assert np.array_equal(rows["top_down"], rows["default"]) and np.array_equal(rows["top_down"], rows["bottom_up_forced"])


def test_bfs_bottom_up_with_the_global_bitmap(cuda_device):
    """N = 1.8 M (visited bitmap in global scratch, bfs_kernel<false>), bottom-up forced: hundreds of sparse levels."""
    from graphgan_b200 import graph as G, sampler as S, synth
    from oracle import canonical as can
    n = 1_800_000
    hg = G.HostGraph(synth.power_law(n, 3, seed=9), None, n_node=n)
    dg = G.DeviceGraph(hg, cuda_device)
    smp = S.WalkSampler(dg)
    roots = synth.pick_roots(hg.degrees(), 4, seed=4)
    want = can.bfs_parents(hg.indptr, hg.adj, roots)
    for mode in ("bottom_up_forced", "default"):
        assert np.array_equal(_trees_in_mode(smp, roots, mode).parent_arrays().cpu().numpy(), want), mode


@pytest.mark.parametrize("hub", [0, 256])
def test_giant_hub_lists_beyond_the_smem_score_buffer(hub, cuda_device):
    """A 3000+-neighbour hub: candidate lists longer than the 2048-score shared buffer and than the 64 tiles
    whose running totals the draw tracks (global-scratch scores, linear tail scan), at ld = 32 (CPL = 1)."""
    import torch
    from graphgan_b200 import graph as G, sampler as S, synth
    from oracle import canonical as can
    n, d = 3600, 32
    rs = np.random.RandomState(8)
    star = np.stack([np.zeros(n - 1, np.int64), rs.permutation(np.arange(1, n))], 1)
    extra = synth.power_law(n, 6, seed=9)
    edges = np.concatenate([star[:1500], extra, star[1500:]])
    hg = G.HostGraph(edges, None, n_node=n)
    assert hg.max_deg >= n - 1
    emb_h = synth.embeddings(n, d, seed=10, sigma=0.4)
    dg = G.DeviceGraph(hg, cuda_device)
    smp = S.WalkSampler(dg, hub_threshold=hub, depth1=True)
    roots = np.asarray([0, 3, 11, 200, 1999, 3599], np.int32)
    trees = smp.build_trees(roots)
    par = trees.parent_arrays().cpu().numpy()
    assert np.array_equal(par, can.bfs_parents(hg.indptr, hg.adj, roots))
    emb = S.pad_embedding(emb_h, cuda_device)
    bias_h = rs.normal(0, 0.2, n).astype(np.float32)
    bias = torch.as_tensor(bias_h).to(cuda_device)
    sample_num = np.asarray([120, 40, 40, 40, 40, 40], np.int64)
    bits = np.zeros(dg.n_bit_words, np.uint32)
    E = can.pad_rows(emb_h)
    for for_d, tag in ((True, 1), (False, 2)):
        ref = can.walk_pass(E, bias_h, hg.indptr, hg.adj, roots, par, sample_num, for_d, bits, seed=5, pass_tag=tag, max_path=16)
        out = smp.run(emb, bias, trees, torch.as_tensor(sample_num).to(cuda_device), for_d, seed=5, pass_tag=tag, max_path=16)
        assert ref.max_l > 2100
        assert np.array_equal(out.status.cpu().numpy(), ref.status)
        assert np.array_equal(out.samples.cpu().numpy(), ref.samples)
        assert np.array_equal(out.wsuml.cpu().numpy(), ref.wsuml)
        assert np.array_equal(dg.d1_bits.cpu().numpy().view(np.uint32), bits)
        if hub and not for_d:   # cp.async.bulk staging of the hub's adjacency / cached scores vs plain loads: same bits
            got = {k: getattr(out, k).clone() for k in ("samples", "status", "wsteps", "wsuml", "path_len")}
            smp.tma = False
            out2 = smp.run(emb, bias, trees, torch.as_tensor(sample_num).to(cuda_device), for_d, seed=5, pass_tag=tag, max_path=16)
            smp.tma = True
            for k, v in got.items():
                assert torch.equal(getattr(out2, k), v), k


def test_partition_invariance(cuda_device):
    """Philox is keyed by (root, walk, step): the rows of a root do not depend on which other roots share its
    batch (or its GPU).  Two half batches == one full batch, row for row (SURVEY 8e)."""
    import torch
    from graphgan_b200 import sampler as S
    case = loader.load("rand1200")
    hg, dg, smp, roots, trees, emb, bias = _setup(case, cuda_device)
    full = smp.run(emb, bias, trees, dg.raw_deg, True, seed=77, pass_tag=9)
    fc, fn, fl, fk = (x.clone() for x in smp.emit_d_rows(full))
    fk = int(fk.item())
    bits_full = dg.d1_bits.clone()
    dg.reset_tree_mutations()
    parts = []
    for lo, hi in ((0, 500), (500, 1200)):
        t = trees.slice(lo, hi)
        o = smp.run(emb, bias, t, dg.raw_deg[lo:hi].contiguous(), True, seed=77, pass_tag=9)
        c, nb, lb, k = smp.emit_d_rows(o)
        k = int(k.item())
        parts.append((c[:k].clone(), nb[:k].clone(), lb[:k].clone()))
    assert torch.equal(torch.cat([p[0] for p in parts]), fc[:fk])
    assert torch.equal(torch.cat([p[1] for p in parts]), fn[:fk])
    assert torch.equal(torch.cat([p[2] for p in parts]), fl[:fk])
    assert torch.equal(dg.d1_bits, bits_full)


@pytest.mark.parametrize("d,hub", [(256, 16), (200, 0), (64, 256)])
def test_wide_and_odd_embeddings(d, hub, cuda_device):
    """n_emb = 256 (ld 256, 8 float4 chunks per lane), 200 (padded to 224? no: to 256 -> zero columns take part
    in the canonical dot) and 64, against the canonical oracle."""
    from graphgan_b200 import graph as G, synth
    n = 1500
    edges = synth.power_law(n, 8, seed=12)
    hg = G.HostGraph(edges, None, n_node=n)
    case = loader.Case(n=n, dim=d, train_edges=edges, test_edges=np.zeros((0, 2), np.int64),
                       emb_g=synth.embeddings(n, d, seed=13, sigma=0.25), bias_g=np.random.RandomState(14).normal(0, 0.3, n).astype(np.float32))
    case["graph"] = [hg.neighbors(i).tolist() for i in range(n)]
    roots = np.sort(np.random.RandomState(1).choice(np.flatnonzero(hg.degrees() > 0), 300, replace=False))
    _philox_compare(case, cuda_device, roots, 0.8, seed=321, n_sample_gen=7, hub_threshold=hub)


def test_empty_and_degenerate_batches(cuda_device):
    """Zero roots, roots without walks (isolated nodes, sample_num 0), update_ratio 0: nothing crashes, nothing
    is accepted, counters stay zero."""
    import torch
    from graphgan_b200 import sampler as S
    case = loader.load("tiny")
    hg, dg, smp, roots, trees, emb, bias = _setup(case, cuda_device)
    # (a) no roots at all
    t0 = trees.slice(0, 0)
    out = smp.run(emb, bias, t0, dg.raw_deg[:0].contiguous(), True, seed=1)
    assert out.n_walks == 0 and out.counters_host()["accepted"] == 0
    c, nb, lb, k = smp.emit_d_rows(out)
    assert int(k.item()) == 0
    # (b) only the isolated node 9 and the self-loop-only node 10 (graph_gan.py:252-253)
    sel = torch.as_tensor([9, 10]).to(cuda_device)
    t1 = trees.select(sel)
    out = smp.run(emb, bias, t1, dg.raw_deg[sel].contiguous(), True, seed=1)
    assert out.root_ok.cpu().tolist()[:2] == [0, 0] and out.counters_host()["accepted"] == 0
    out = smp.run(emb, bias, t1, 3, False, seed=1, max_path=8)       # G mode: paths_from_i is None
    assert (out.status.cpu().numpy()[:6] != S.DONE).all()
    # (c) update_ratio = 0 skips every root
    out = smp.run(emb, bias, trees, dg.raw_deg, True, seed=1, update_ratio=0.0)
    assert out.counters_host()["accepted"] == 0 and (out.status.cpu().numpy()[:out.n_walks] == S.SKIPPED).all()


def test_bench_dump_outputs_are_reproducible(cuda_device, tmp_path):
    """`bench.py --dump-outputs DIR`: the D rows of the last timed step, float64, the same from run to run with the
    same arguments; --steps sets the number of timed steps; the oracle parity of that step is clean."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for k in range(2):
        d = tmp_path / ("run%d" % k)
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "powerlaw_100k", "--roots", "512",
                              "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--g-steps", "0", "--verify", "4",
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=root)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout)
        assert line["steps"] == 3 and line["parity"]["mismatches"] == 0 and line["parity"]["tree_mismatches"] == 0
        names = sorted(p.name for p in d.iterdir())
        assert names == ["center.npy", "label.npy", "n_rows.npy", "neighbor.npy", "row_index.npy"]
        assert sum(p.stat().st_size for p in d.iterdir()) <= 64 << 20
        a = {p.stem: np.load(p) for p in d.iterdir()}
        assert all(v.dtype == np.float64 for v in a.values())
        n = int(a["n_rows"][0])
        assert n > 0 and np.array_equal(a["row_index"], np.arange(n))       # small enough to be dumped whole
        assert a["center"].shape == a["neighbor"].shape == a["label"].shape == (n,)
        assert 2 * int(a["label"].sum()) == n                                # one negative row per positive row
        assert ((a["neighbor"] >= 0) & (a["neighbor"] < 100_000)).all()
        dumps.append(a)
    for name in dumps[0]:
        assert np.array_equal(dumps[0][name], dumps[1][name]), name
