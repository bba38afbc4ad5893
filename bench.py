#!/usr/bin/env python
"""bench.py -- sampled negative edges / second of the D-sampling pass (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of synthetic input: every walk of
``prepare_data_for_d`` (reference src/GraphGAN/graph_gan.py:182-202 -> sample :225-270) for R
resident roots -- K1 (walk kernel) + finalize + row emission.  Workload at N=1: BASELINE.json
configs[2], synthetic power-law N=1M, avg-deg 20, n_emb=128 (the configuration the metric is
quoted on).  Multi-GPU: every rank holds the replicated graph/embeddings and its own R roots
(weak scaling, no data-path collective -- SURVEY.md section 8e).

  python bench.py [--gpus N --steps K --warmup W]         # one JSON line on rank 0
  python bench.py --impl reference ...                    # the reference's CPU path (oracle T0, all host threads)

The CUDA path never touches oracle/; only the cpu_baseline / --impl reference legs do.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (generator, N, avg_deg, d)
    "powerlaw_1m": ("power_law", 1_000_000, 20, 128),     # BASELINE.json configs[2] / [3]
    "er_100k": ("erdos_renyi", 100_000, 10, 128),         # configs[1]
    "powerlaw_100k": ("power_law", 100_000, 10, 128),     # smoke-sized
    "powerlaw_10m": ("power_law", 10_000_000, 8, 256),    # configs[4] (per-GPU share; R is capped by the memory rule)
    "c1_cagrqc": ("fixture", 5242, 5, 50),                # configs[0]: the shipped CA-GrQc graph + pretrain embeddings
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=50)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="powerlaw_1m", choices=sorted(WORKLOADS))
    p.add_argument("--roots", type=int, default=16384,
                   help="resident roots per GPU (R); the tree rows take R * nnz / 8 bytes (41 GB at C3), capped at half of the "
                        "device memory")
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--hub-threshold", type=int, default=128, help="degree from which adjacency scores are cached per pass")
    p.add_argument("--file-order", action="store_true", help="start the walks in root order instead of hub-neighbourhoods first")
    p.add_argument("--no-depth1", dest="depth1", action="store_false",
                   help="disable the per-(root, depth-1 child) CDF reuse (csrc/walk.cu: step1_cdf_kernel)")
    p.add_argument("--no-tma", action="store_true", help="enumerate hub lists with plain loads instead of cp.async.bulk staging (A/B)")
    p.add_argument("--flat-steps", type=int, default=None,
                   help="level-synchronous walk steps before the persistent kernel (csrc/walk.cu: flat_*_kernel); default: the sampler's")
    p.add_argument("--verify", type=int, default=12, help="roots of the last timed pass re-derived with the C oracle (0 = off)")
    p.add_argument("--verify-seconds", type=float, default=45.0, help="time budget of --verify")
    p.add_argument("--g-steps", type=int, default=5, help="timed generator-mode passes (0 = skip)")
    p.add_argument("--pairs", type=int, default=1 << 22, help="--phase reward: pairs per launch")
    p.add_argument("--bfs-roots", type=int, default=1184, help="--phase bfs: roots per launch (8 per SM)")
    p.add_argument("--score-mode", default="lazy", choices=["lazy", "literal"],
                   help="--impl reference: 'literal' recomputes the whole N x N all_score per root exactly as graph_gan.py:238 does "
                        "(only feasible at C1); 'lazy' scores the candidates on demand (the only form that exists at N >= 1e5)")
    p.add_argument("--transport", default="nccl", choices=["nccl", "p2p"],
                   help="--phase update: gradient exchange by ncclAllGather or by peer-memory stores fused into the gradient kernel")
    p.add_argument("--adam-path", default="ldg", choices=["ldg", "tma", "tma256x2", "tma512x3", "ws16", "ws8"],
                   help="K3 sweep: cp.async.bulk (TMA) pipeline or the per-thread-load kernel (A/B; sets GG_ADAM_PATH)")
    p.add_argument("--phase", default="sample", choices=["sample", "reward", "adam", "bfs", "update"],
                   help="what to time: the D-sampling pass (the BASELINE metric) or one of the other kernels of the path")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the (center, neighbor, label) rows of the last timed D-sampling step as DIR/<name>.npy "
                        "(float64; a fixed sample of %d rows when there are more), to compare two builds output for output"
                        % DUMP_ROWS)
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.phase != "sample"):
        p.error("--dump-outputs writes the D-sampling pass of --impl b200 --phase sample")
    return args


DUMP_ROWS = 1 << 20      # 4 float64 arrays of this many rows: 32 MiB, half of the 64 MB a dump may take


def dump_rows(dirname, out):
    """The rows prepare_data_for_d returns (graph_gan.py:192-201) as the last step of `out` left them in its plan's
    buffers, plus row_index.npy (which rows: all of them, or a fixed seeded sample) and n_rows.npy."""
    p = out.plan
    n = int(p.n_rows.item())
    idx = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    os.makedirs(dirname, exist_ok=True)
    arrays = {"n_rows": np.array([n]), "row_index": idx}
    for name, rows in zip(("center", "neighbor", "label"), p.rows):
        arrays[name] = rows[:n].cpu().numpy()[idx]
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a.astype(np.float64))


def make_inputs(args, rank):
    from graphgan_b200 import graph as G, synth
    gen, n, deg, d = WORKLOADS[args.workload]
    if gen == "fixture":      # BASELINE.json configs[0]: tests/golden/cagrqc.npz holds the reference's own data files
        from tests.golden import loader
        c = loader.load("cagrqc")
        hg = G.HostGraph(c.train_edges, c.test_edges)
        roots = np.flatnonzero(hg.degrees() > 0).astype(np.int32)
        args.roots = len(roots)
        return hg, np.asarray(c.emb_g, np.float64).astype(np.float32), roots, d
    cache = "/tmp/gg_bench_cache/%s_seed%d.npz" % (args.workload, args.seed)
    try:       # the CSR arrays of an earlier process on this box (the reference arm, another rank, an ncu pass)
        z = np.load(cache)
        hg = G.HostGraph.from_arrays(n, z["raw_indptr"], z["raw_adj"], z["indptr"], z["adj"])
    except (OSError, ValueError, KeyError, AssertionError):
        hg = G.HostGraph(getattr(synth, gen)(n, deg, seed=args.seed), None, n_node=n)
        try:   # best effort
            os.makedirs(os.path.dirname(cache), exist_ok=True)
            tmp = "%s.%d.tmp.npz" % (cache, os.getpid())
            np.savez(tmp, raw_indptr=hg.raw_indptr, raw_adj=hg.raw_adj, indptr=hg.indptr, adj=hg.adj)
            os.replace(tmp, cache)
        except OSError:
            pass
    emb = synth.embeddings(n, d, seed=args.seed + 1)
    n_roots = args.roots
    if args.impl == "b200":      # SURVEY 8d: "R chosen so the trees fit"
        import torch
        total = torch.cuda.mem_get_info()[1]
        n_roots = max(1, min(n_roots, int(total // 2 // (hg.adj.shape[0] // 8 + 8))))
        args.roots = n_roots
    # one seeded pool of R * world roots in ascending id order, dealt out round-robin: node ids follow the degree
    # ranking in the synthetic graphs, so every rank gets the same degree mix (the roots of a real pass would be
    # partitioned degree-balanced too, SURVEY 8e) -- with independent random sets the slowest rank's set costs ~5 % more
    world = max(1, int(os.environ.get("WORLD_SIZE", "1")))
    roots = synth.pick_roots(hg.degrees(), n_roots * world, seed=args.seed)[rank % world::world]
    return hg, emb, roots, d


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_first(self, timeout=5.0):
        """nvidia-smi takes a moment to print its first row; do not start a short timed region before it."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        rows = [r for (t, r) in self.rows if t0 - 0.02 <= t <= t1 + 0.12]
        if not rows and self.rows:   # region shorter than the sampling period: take the sample nearest to it
            rows = [min(self.rows, key=lambda tr: abs(tr[0] - 0.5 * (t0 + t1)))[1]]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU legs (oracle; checker only)
_SH = {}   # inherited by forked workers: graph, embeddings, parent arrays of the sample


class _AdjView:
    def __init__(self, indptr, adj):
        self.indptr, self.adj = indptr, adj

    def __getitem__(self, i):
        return self.adj[self.indptr[i]:self.indptr[i + 1]]


class _GraphView:
    """graph[i] for the sampled roots only: prepare_data_for_d needs the list and its length."""

    def __init__(self, hg, roots):
        self.d = {int(r): hg.neighbors(int(r)).tolist() for r in roots}

    def __getitem__(self, i):
        return self.d[i]

    def __len__(self):
        return len(self.d)


def _bfs_chunk(rng):
    from oracle import canonical as can
    lo, hi = rng
    hg = _SH["hg"]
    _SH["par"][lo:hi] = can.bfs_parents(hg.indptr, hg.adj, _SH["sample"][lo:hi])
    return hi - lo


def _one_thread():
    """Pool initializer: one BLAS/OpenMP thread per worker process (the pool already uses every core; without this each
    of the C workers starts C BLAS threads and the box thrashes -- measured 50x slower per core on 128 cores)."""
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    try:
        import threadpoolctl
        _SH["_limit"] = threadpoolctl.threadpool_limits(limits=1)
    except Exception:      # noqa: BLE001 -- best effort
        pass


def _sample_roots(job):
    """The reference's prepare_data_for_d -> sample(for_d=True) (oracle T0, lazy score) over sample[idx]."""
    from oracle import faithful
    idx, seed = job
    idx = np.atleast_1d(np.asarray(idx, np.int64))
    hg, emb, roots, par = _SH["hg"], _SH["emb"], _SH["sample"][idx], _SH["par"]
    trees = faithful.ParentTrees(_AdjView(hg.indptr, hg.adj), {int(r): par[int(i)] for i, r in zip(idx, roots)})
    F = faithful.Faithful(_GraphView(hg, roots), emb, bias_g=_SH["bias"], rng=np.random.RandomState(seed),
                          score_mode=_SH.get("score_mode", "lazy"), trees=trees)
    t0 = time.time()
    F.prepare_data_for_d(roots=[int(r) for r in roots])
    return os.getpid(), F.stats["neg_edges"], F.stats["steps"], F.stats["sum_l"], time.time() - t0


class CpuReference:
    """Bounded sample of the workload's roots, trees built once (the reference caches them too), then timed passes
    of the reference sampling logic on `workers` host processes (one fork pool, created before the timed passes).

    The reference walks all `sample_num` walks of a root inside one `sample()` call, so a root is the smallest unit
    of work, and on a power-law graph one root can hold thousands of walks: the wall clock of a bounded sample is
    set by its largest root, not by the core count.  The value reported is therefore the STEADY-STATE rate of the
    pool -- the sum over worker processes of (edges sampled / seconds busy), roots handed out one at a time, largest
    first -- which is what a long pass over all roots converges to (and is the generous reading for the CPU side).
    Roots whose expected time alone exceeds the per-step budget are left out of the sample."""

    TREE_BYTES = 4 << 30     # parent arrays of the sample (4*N bytes per root) stay below this

    def __init__(self, hg, emb, roots, seconds, workers, parent_rows=None):
        import multiprocessing as mp
        self.mp, self.workers, self.pool, self.path, self.seconds = mp.get_context("fork"), workers, None, None, seconds
        _SH.update(hg=hg, emb=emb, bias=np.zeros(hg.n_node, np.float32))
        deg = hg.degrees()
        # calibrate on 2 roots (evenly spaced: roots are sorted by id and low ids are the hubs)
        cal = roots[[len(roots) // 3, (2 * len(roots)) // 3]]
        _SH["sample"] = cal
        if parent_rows is not None:
            _SH["par"] = parent_rows(cal)
        else:
            _SH["par"] = np.empty((2, hg.n_node), np.int32); _bfs_chunk((0, 2))
        _, e, st, sl, dt = _sample_roots((np.arange(2), 12345))
        per_root = max(dt / 2, 1e-4)
        per_walk = max(dt / max(int(deg[cal].sum()), 1), 1e-6)
        cap = max(64, int(seconds / per_walk))               # a root with more walks than this overruns a step alone
        cand = roots[deg[roots] <= cap] if workers > 1 else roots
        n = int(min(len(cand), max(2 * workers, workers * seconds / per_root)))
        # bound the tree memory and, when the trees are built here, the BFS time of the sample
        n = min(n, max(2, self.TREE_BYTES // (4 * hg.n_node)), 1024 if parent_rows is not None else 96 * workers)
        self.sample = cand[np.unique(np.linspace(0, len(cand) - 1, n).astype(np.int64))]
        n = len(self.sample)
        self.order = np.argsort(-deg[self.sample], kind="stable")      # largest roots first
        _SH["sample"] = self.sample
        par = None
        for d in ("/dev/shm", "/tmp"):
            try:
                self.path = "%s/gg_bench_par_%d.npy" % (d, os.getpid())
                par = np.lib.format.open_memmap(self.path, mode="w+", dtype=np.int32, shape=(n, hg.n_node))
                break
            except OSError:
                par = None
        if par is None:
            raise RuntimeError("no room for the parent arrays of the CPU sample")
        _SH["par"] = par
        self.chunks = [(int(c[0]), int(c[-1]) + 1) for c in np.array_split(np.arange(n), min(workers, n)) if len(c)]
        if len(self.chunks) > 1:
            self.pool = self.mp.Pool(len(self.chunks), initializer=_one_thread)   # forked AFTER _SH is complete
        if parent_rows is not None:
            par[:] = parent_rows(self.sample)
        elif self.pool is None:
            _bfs_chunk((0, n))
        else:
            self.pool.map(_bfs_chunk, self.chunks)
            par.flush()

    def run(self, seed):
        t0 = time.time()
        if self.pool is None:
            res = [_sample_roots((self.order, seed))]
        else:
            res = list(self.pool.imap_unordered(_sample_roots, [(int(i), seed * 100003 + int(i)) for i in self.order], chunksize=1))
        dt = time.time() - t0
        busy, done = {}, {}
        for pid, e, st, sl, b in res:
            busy[pid] = busy.get(pid, 0.0) + b
            done[pid] = done.get(pid, 0) + e
        edges = sum(done.values())
        value = sum(done[p] / busy[p] for p in busy if busy[p] > 0)
        out = {"value": value, "unit": "neg_edges/s", "cores": len(busy), "kind": "port",
               "wall_clock_value": edges / max(dt, 1e-9), "score_mode": _SH.get("score_mode", "lazy"),
               "sample": "%d of the workload's roots (%d neg edges, %d walk steps, %d candidates), %.1f core-seconds in "
                         "%.1f s wall on %d processes; value = sum over processes of edges / busy seconds (steady-state "
                         "rate; the wall clock of a bounded sample is set by its largest root); oracle T0 lazy-score: "
                         "the reference's sample()/prepare_data_for_d logic (graph_gan.py:182-270) with numpy standing "
                         "in for TF1.8, trees prebuilt" % (len(self.sample), edges, sum(r[2] for r in res),
                                                           sum(r[3] for r in res), sum(busy.values()), dt, len(busy))}
        return out, dt

    def close(self):
        if self.pool is not None:
            self.pool.close(); self.pool.join(); self.pool = None
        try:
            os.unlink(self.path)
        except (OSError, TypeError):
            pass


# ----------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    hg, emb, roots, d = make_inputs(args, 0)
    _SH["score_mode"] = args.score_mode
    workers = os.cpu_count() or 1
    per_step_seconds = max(0.5, min(args.cpu_seconds, 150.0 / max(args.steps + args.warmup, 1)))   # whole run: a few minutes
    ref = CpuReference(hg, emb, roots, per_step_seconds, workers)
    times, vals, last = [], [], None
    for s in range(args.warmup + args.steps):
        res, dt = ref.run(args.seed + s)
        if s >= args.warmup:
            times.append(dt); vals.append(res["value"])
        last = res
    ref.close()
    v = float(np.mean(vals)) if vals else last["value"]
    last["value"] = v
    line = {"impl": "reference", "metric": "sampled negative edges/sec (D-sampling pass)", "value": v,
            "unit": "neg_edges/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * float(np.mean(times)) if times else None, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": data_kind(args),
            "config": workload_config(args, hg, d), "cpu_baseline": last,
            "e2e": {"value": v, "unit": "neg_edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


def data_kind(args):
    return "reference data files (CA-GrQc, tests/golden/cagrqc.npz)" if WORKLOADS[args.workload][0] == "fixture" else "synthetic"


def workload_config(args, hg, d):
    gen, n, deg, _ = WORKLOADS[args.workload]
    return {"workload": "%s N=%d avg_deg=%d n_emb=%d, D-sampling pass over R=%d resident roots per GPU "
                        "(sample_num = deg(root), Philox RNG, update_ratio=1)" % (gen, n, deg, d, args.roots),
            "nnz": int(hg.adj.shape[0]), "max_deg": int(hg.max_deg),
            "l2_policy": "inputs larger than L2 (embedding matrix %d MB, tree rows %d MB)" % (
                n * d * 4 >> 20, args.roots * (int(hg.adj.shape[0]) // 8) >> 20),
            "parallelism": "roots sharded over %d GPU(s), replicated graph+embeddings" % args.gpus}


# ----------------------------------------------------------------------------- B200 arm
def _peak():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        if "hbm_gbs" in peaks:
            return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except (OSError, ValueError):
        pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _ncu_traffic(kernel, key):
    """DRAM bytes per launch of `kernel` from the committed ncu capture -- only when that capture was taken from the
    library that is running now (content hash of csrc/ + include/); a stale capture reports null."""
    try:
        from graphgan_b200 import _build
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        if t.get("source_hash") != _build.source_hash():
            return None, "profiles/ncu_traffic.json was captured from other kernel sources (hash mismatch): not used"
        v = t.get("kernels", {}).get(key, {}).get(kernel)
        return (float(v), "profiles/ncu_traffic.json (%s)" % t.get("capture", "?")) if v is not None else (None, "no capture for %s" % key)
    except (OSError, ValueError):
        return None, "no ncu capture committed for these kernel sources"


def _verify(args, hg, emb_h, roots, trees, out, smp, dev, seed, tag):
    """Re-derive K roots of the LAST TIMED pass with the C oracle (oracle/gg_oracle.c: BFS tree + every walk of the root,
    same Philox key) and compare the sampled nodes / statuses bit for bit."""
    import torch
    from oracle import canonical as can
    K = min(args.verify, len(roots))
    if K <= 0:
        return None
    deg = hg.degrees()[roots]
    order = np.argsort(deg, kind="stable")
    pick = np.unique(np.concatenate([np.linspace(0, len(roots) - 1, K - 1).astype(np.int64) if K > 1 else [],
                                     [order[-1]]]).astype(np.int64))            # a spread of roots + the largest one
    budget = float(args.verify_seconds)
    t0 = time.time()
    E = can.pad_rows(emb_h, smp_ld(emb_h))
    bias0 = np.zeros(hg.n_node, np.float32)
    wp = out.walk_ptr.cpu().numpy()
    samples, status = out.samples.cpu().numpy(), out.status.cpu().numpy()
    checked = walks = mism = tree_mism = 0
    skipped = 0
    for k in pick:
        if time.time() - t0 > budget and checked > 0:
            skipped += 1
            continue
        r = roots[k:k + 1]
        par = can.bfs_parents(hg.indptr, hg.adj, r)
        got_par = trees.parent_arrays(torch.as_tensor([int(k)], device=dev)).cpu().numpy()
        tree_mism += int(not np.array_equal(par, got_par))
        bits = np.zeros((hg.adj.shape[0] + 31) // 32 + 1, np.uint32)
        ref = can.walk_pass(E, bias0, hg.indptr, hg.adj, r, par, deg[k:k + 1], True, bits, seed=seed, pass_tag=tag)
        w0, w1 = int(wp[k]), int(wp[k + 1])
        ok = bool(ref.root_ok[0])
        if ok:
            mism += int(np.count_nonzero(samples[w0:w1] != ref.samples)) + int(np.count_nonzero(status[w0:w1] != ref.status))
        else:       # the reference voids the whole root: finalize blanks the walks after the first void
            mism += int(out.root_ok[k].item() != 0)
        checked += 1
        walks += w1 - w0
    return {"roots_checked": checked, "walks_checked": walks, "mismatches": mism, "tree_mismatches": tree_mism,
            "roots_skipped_over_budget": skipped, "seconds": round(time.time() - t0, 2),
            "oracle": "oracle/gg_oracle.c (T1): ggo_bfs_parent + ggo_walk_pass on the roots of the last timed pass"}


def smp_ld(emb_h):
    d = int(emb_h.shape[1])
    ld = 32
    while ld < d:
        ld *= 2
    return ld


def run_b200(args):
    import torch
    import torch.distributed as dist
    from graphgan_b200 import graph as G, sampler as S
    from graphgan_b200.sampler import CNT
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    hg, emb_h, roots, d = make_inputs(args, rank)
    dg = G.DeviceGraph(hg, dev)
    smp = S.WalkSampler(dg, hub_threshold=args.hub_threshold, depth1=args.depth1, hub_first=not args.file_order, tma=not args.no_tma)
    if args.flat_steps is not None:
        smp.flat_steps = args.flat_steps
    emb = S.pad_embedding(emb_h, dev)
    bias = torch.zeros(hg.n_node, dtype=torch.float32, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    # ---- tree construction (outside the metric: "trees resident", SURVEY 8d) -- timed on the device, reported
    smp.build_trees(roots[:min(len(roots), 296)])                     # warm-up (allocates the builder's scratch)
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    e0.record()
    trees = smp.build_trees(roots)
    e1.record()
    torch.cuda.synchronize()
    bfs_ms = e0.elapsed_time(e1)
    sample_num = dg.raw_deg[trees.roots.long()]
    W = int(sample_num.sum().item())

    # pinned host buffers of the plugin-level call
    roots_pin = torch.from_numpy(roots.copy()).pin_memory()
    rows_pin = [torch.empty(2 * W, dtype=torch.int32).pin_memory() for _ in range(3)]
    nrows_pin = torch.zeros(1, dtype=torch.int64).pin_memory()

    t0 = time.time()
    plan = smp.plan(trees, sample_num, True)
    reuse = smp.hub_threshold > 0
    if reuse:
        dg.hub_tiles(smp.hub_threshold)
        if smp.depth1:
            plan.depth1_buffers(smp)
    if smp.hub_first:
        plan.start_order(smp)
    torch.cuda.synchronize()
    plan_ms = 1e3 * (time.time() - t0)

    def step(tag, e2e=False, events=None):
        if e2e:
            trees.roots.copy_(roots_pin, non_blocking=True)          # H2D: this step's root ids
        if events is not None:
            events[0].record()
        if reuse:                                                    # per-pass reuse: depends on the embeddings,
            smp.precompute(emb, bias, plan)                          # so it is part of every pass
        if events is not None:                                       # (breakdown only: the two stages of gg_walk_sample
            events[1].record()                                       # as two calls, so that each can be timed)
            smp.run(emb, bias, trees, sample_num, True, seed=args.seed, pass_tag=tag, finalize=False, plan=plan,
                    precompute=False, phase_mask=1)
            events[2].record()
            out = smp.run(emb, bias, trees, sample_num, True, seed=args.seed, pass_tag=tag, finalize=False, plan=plan,
                          precompute=False, phase_mask=2, zero_counters=False)
            events[3].record()
        else:
            out = smp.run(emb, bias, trees, sample_num, True, seed=args.seed, pass_tag=tag, finalize=False, plan=plan,
                          precompute=False)
        smp.finalize(out)
        c, nb, lb, n_rows = smp.emit_d_rows(out)
        if events is not None:
            events[4].record()
        if e2e:
            rows_pin[0].copy_(c, non_blocking=True); rows_pin[1].copy_(nb, non_blocking=True)
            rows_pin[2].copy_(lb, non_blocking=True); nrows_pin.copy_(n_rows, non_blocking=True)
            torch.cuda.current_stream().synchronize()                # the caller reads the rows
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(e2e):
        for s in range(args.warmup):
            step(1000 + s, e2e)
        barrier()
        b0, b1 = ev(), ev()
        t_start = time.time()
        b0.record()
        cnts_live, out = [], None
        for s in range(args.steps):
            out = step(2000 + s, e2e)
            cnts_live.append(out.counters.clone())                   # device-side copy, read after the region
        b1.record()
        barrier()
        t_end = time.time()
        ms = b0.elapsed_time(b1)
        cnts = [{k: int(c[i]) for k, i in CNT.items()} for c in (x.cpu().numpy() for x in cnts_live)]
        return ms, cnts, t_start, t_end, out

    clocks = ClockSampler(local)
    clocks.wait_first()
    ms, cnts, t_start, t_end, last_out = timed(False)
    clk = clocks.stop(t_start, t_end)
    if rank == 0 and args.dump_outputs:         # before the e2e passes below overwrite the plan's row buffers
        dump_rows(args.dump_outputs, last_out)
    parity = None
    if rank == 0 and args.verify > 0:
        parity = _verify(args, hg, emb_h, roots, trees, last_out, smp, dev, args.seed, 2000 + args.steps - 1)
    ms_e2e, cnts_e2e, _, _, _ = timed(True)

    # ---- per-kernel breakdown (separate, untimed-for-the-headline passes; same work, stage boundaries evented)
    nb_ = max(3, min(10, args.steps))
    evs = [[ev() for _ in range(5)] for _ in range(nb_)]
    bcnt = []
    for s in range(nb_):
        o = step(3000 + s, False, evs[s])
        bcnt.append(o.counters.clone())
    torch.cuda.synchronize()
    stage = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(4)] for e in evs]).mean(0)   # pre, depth1, walk, finalize+emit
    brows = float(np.mean([int(c[CNT["rows_gathered"]]) for c in bcnt]))                       # walk_kernel only (phase 2)

    # ---- generator-mode pass (prepare_data_for_g's walks: n_sample_gen per root, paths recorded)
    g_stats = None
    if args.g_steps > 0:
        plan_g = smp.plan(trees, 20, False, 64)
        def gstep(tag):
            if reuse:
                smp.precompute(emb, bias, plan_g)
            return smp.run(emb, bias, trees, 20, False, seed=args.seed, pass_tag=tag, max_path=64, plan=plan_g, precompute=False)
        for s in range(2):
            gstep(4000 + s)
        torch.cuda.synchronize()
        g0, g1 = ev(), ev()
        g0.record()
        for s in range(args.g_steps):
            og = gstep(4100 + s)
        g1.record()
        torch.cuda.synchronize()
        gms = g0.elapsed_time(g1) / args.g_steps
        gc = og.counters_host()
        done = int((og.status == S.DONE).sum().item())
        g_stats = {"samples_per_s": done / (gms * 1e-3), "ms_per_pass": gms, "walks": int(og.n_walks), "done": done,
                   "steps_per_s": gc["steps"] / (gms * 1e-3), "path_overflow": gc["path_overflow"],
                   "note": "G mode: 20 walks per root (config.n_sample_gen), paths recorded (max_path 64), trees as left by the D passes"}

    accepted = sum(c["accepted"] for c in cnts)
    accepted_e2e = sum(c["accepted"] for c in cnts_e2e)
    tot = torch.tensor([float(accepted), float(accepted_e2e), float(sum(c["steps"] for c in cnts)), float(W * args.steps)],
                       dtype=torch.float64, device=dev)
    tmax = torch.tensor([ms, ms_e2e, bfs_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tot, tmax = tot.cpu().numpy(), tmax.cpu().numpy()

    if rank == 0:
        peak, peak_src = _peak()
        ld = int(emb.shape[1])
        c0 = cnts[-1]
        row_b = 4 * ld + 8
        pre_ms, d1_ms, walk_ms, fin_ms = (float(x) for x in stage)
        k1_ms = pre_ms + d1_ms + walk_ms
        # SURVEY 8d algorithmic bytes (every candidate row counted at every visit) -- an upper bound on the work a
        # literal implementation would do, NOT what these kernels move (hub scores once per pass, one CDF per root,
        # one per (root, child) pair): reported as the reuse ratio, never as a roofline fraction
        survey_bytes = float(np.mean([W * 4 * ld + c["sum_l"] * row_b for c in cnts]))
        hub_edges = dg.hub_tiles(smp.hub_threshold)[3] if reuse else 0
        deg_w = np.diff(hg.indptr)[roots]
        root_rows = int(deg_w[deg_w < smp.hub_threshold].sum() + len(roots)) if reuse else 0
        all_rows = float(np.mean([c["rows_gathered"] for c in cnts])) + hub_edges + root_rows     # whole K1 stage
        key = "%s@R%d" % (args.workload, args.roots)
        flat = smp.flat_steps if (reuse and smp.depth1) else 0
        traffic, traffic_src = _ncu_traffic("walk_stage" if flat else "walk_kernel", key)
        stage_traffic, _ = _ncu_traffic("k1_stage", key)
        choose_us, _ = _ncu_traffic("flat_choose_kernel_ncu_us_per_pass", key)
        stage_us, _ = _ncu_traffic("walk_stage_ncu_us", key)
        if flat:
            kname = ("walk stage = gg::flat_start_kernel + %d x (gg::flat_enum_kernel + gg::flat_choose_kernel<%d>) + gg::walk_kernel<%d> "
                     "tail (dominant stage: %.0f %% of the K1 stage%s)" % (
                         flat, ld // 32, ld // 32, 100 * walk_ms / k1_ms,
                         "; flat_choose_kernel = %.0f %% of it in the ncu launch list" % (100 * choose_us / stage_us) if choose_us and stage_us else ""))
        else:
            kname = "gg::walk_kernel<%d> (dominant: %.0f %% of the K1 stage)" % (ld // 32, 100 * walk_ms / k1_ms)
        useful = brows * row_b                                       # embedding rows + bias + id the dominant kernel gathered
        achieved = useful / (walk_ms * 1e-3) / 1e9
        line = {
            "metric": "sampled negative edges/sec (D-sampling pass)", "value": float(tot[0] / (tmax[0] * 1e-3)),
            "unit": "neg_edges/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": float(tmax[0] / args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": data_kind(args), "config": workload_config(args, hg, d),
            "clocks": clk,
            "e2e": {"value": float(tot[1] / (tmax[1] * 1e-3)), "unit": "neg_edges/s",
                    "h2d_bytes_per_step": int(roots_pin.numel() * 4),
                    "d2h_bytes_per_step": int(3 * 2 * W * 4 + 8),
                    "call": "WalkSampler.precompute + run + finalize + emit_d_rows with pinned host roots in / rows out",
                    "note": "trees and the walk plan of these roots are resident (SURVEY 8d); a NEW root batch also costs "
                            "gg_bfs_build + the plan -- see full_pass"},
            "gpu_launches": (((11 if smp.depth1 else 9) if reuse else 7) + ((1 + 2 * flat) if flat else 0)) * args.steps,
            "parity": parity,
            "roofline": {"bound": "hbm", "kernel": kname, "flat_steps": flat,
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel_ms": walk_ms,
                         "useful_bytes_per_launch": useful, "useful_frac": achieved / peak,
                         "dram_frac": (traffic / (walk_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "k1_stage": {"ms": k1_ms, "hub_scores_root_cdf_ms": pre_ms, "root_step_step1_cdf_ms": d1_ms,
                                      "walk_kernel_ms": walk_ms, "finalize_emit_ms": fin_ms,
                                      "useful_bytes": all_rows * row_b,
                                      "useful_frac": all_rows * row_b / (k1_ms * 1e-3) / 1e9 / peak,
                                      "dram_bytes": stage_traffic,
                                      "dram_frac": (stage_traffic / (k1_ms * 1e-3) / 1e9 / peak) if stage_traffic else None},
                         "survey_algorithmic_bytes_per_launch": survey_bytes,
                         "algorithmic_reuse_ratio": survey_bytes / max(all_rows * row_b, 1.0),
                         "bytes_per_neg_edge_survey": survey_bytes / max(c0["accepted"], 1),
                         "note": "achieved = (embedding row + bias + id) bytes the walk stage gathers on demand per pass / its "
                                 "event-timed duration (frac = useful_frac); dram_frac uses ncu dram__bytes of the same kernels when "
                                 "a capture of THESE sources is committed.  With flat_steps > 0 the stage is a sequence of "
                                 "level-synchronous kernels (the row gathers sit in flat_choose_kernel) and is timed as a whole.  "
                                 "SURVEY 8d's formula counts every candidate row at every visit; the kernels fetch "
                                 "algorithmic_reuse_ratio x fewer bytes (exact reuse, DESIGN.md 5)"},
            "rates": {"walks_per_s": float(tot[3] / (tmax[0] * 1e-3)), "walk_steps_per_s": float(tot[2] / (tmax[0] * 1e-3)),
                      "g_mode": g_stats},
            "full_pass": {"neg_edges_per_s": c0["accepted"] / ((tmax[2] + plan_ms + tmax[0] / args.steps) * 1e-3),
                          "bfs_build_ms": float(tmax[2]), "bfs_ms_per_root": float(tmax[2]) / len(roots), "plan_ms": plan_ms,
                          "sampling_ms": float(tmax[0] / args.steps),
                          "note": "one NEW root batch end to end: gg_bfs_build (device-timed) + walk plan (host wall clock, torch "
                                  "plumbing) + one sampling pass; the headline metric keeps trees resident (SURVEY 8d)"},
            "walk": {"walks_per_step": W, "steps_per_neg_edge": c0["steps"] / max(c0["accepted"], 1),
                     "cands_per_neg_edge": c0["sum_l"] / max(c0["accepted"], 1), "ok_roots": c0["ok_roots"],
                     "warp_cycle_share": {k[4:]: round(c0[k] / max(c0["cyc_walk"], 1), 4) for k in
                                          ("cyc_enum", "cyc_score", "cyc_choose", "cyc_step0", "cyc_step1", "cyc_step2p")}},
        }
        if not args.no_cpu_baseline and world >= 1:
            def parent_rows(rs):   # reuse the GPU-built trees (checked against the oracle BFS in tests/ and in `parity`)
                idx = np.searchsorted(roots, rs)
                return trees.parent_arrays(torch.as_tensor(idx, device=dev)).cpu().numpy()
            ref = CpuReference(hg, emb_h, roots, args.cpu_seconds, 1, parent_rows=parent_rows)
            line["cpu_baseline"] = ref.run(args.seed)[0]
            # the same roots on the GPU, so that the two numbers of this block describe identical inputs
            idx = torch.as_tensor(np.searchsorted(roots, ref.sample), device=dev)
            sub = trees.select(idx)
            sn = dg.raw_deg[sub.roots.long()]
            psub = smp.plan(sub, sn, True)
            for s in range(3):
                osub = smp.run(emb, bias, sub, sn, True, seed=args.seed, pass_tag=5000 + s, plan=psub)
            torch.cuda.synchronize()
            s0, s1 = ev(), ev()
            s0.record()
            for s in range(5):
                osub = smp.run(emb, bias, sub, sn, True, seed=args.seed, pass_tag=5100 + s, plan=psub)
            s1.record()
            torch.cuda.synchronize()
            line["cpu_baseline"]["gpu_same_roots"] = {
                "value": osub.counters_host()["accepted"] / (s0.elapsed_time(s1) / 5 * 1e-3), "unit": "neg_edges/s",
                "note": "this GPU on exactly the cpu_baseline's root sample (%d roots: too few walks to fill 148 SMs)" % len(ref.sample)}
            ref.close()
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


# ----------------------------------------------------------------------------- other kernels of the path
def run_phase(args):
    """One JSON line for a kernel of the path other than the D-sampling pass (not the BASELINE metric; these lines
    exist so that every number quoted in DESIGN.md section 8 can be reproduced by a command):
      --phase bfs     gg_bfs_build             trees/s        (graph_gan.py:84-108)
      --phase reward  gg_pair_reward           pairs/s        (discriminator.py:33-34, called at graph_gan.py:220-222)
      --phase adam    gg_adam_apply            steps/s        (TF1.8 dense Adam, generator.py:30-31)
      --phase update  one data-parallel optimizer step: pair-grad slice -> NCCL all-gather -> merge -> Adam sweep"""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from graphgan_b200 import _cabi, graph as G, sampler as S
    from graphgan_b200._cabi import ptr
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    gen, n, deg, d = WORKLOADS[args.workload]
    peak, peak_src = _peak()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    lib = _cabi.lib()
    st = lambda: torch.cuda.current_stream(dev).cuda_stream
    ld = smp_ld(np.empty((1, d)))
    clocks = ClockSampler(local)
    clocks.wait_first()

    def time_steps(fn, flush=None):
        for s in range(args.warmup):
            fn(s)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.time()
        tot = 0.0
        for s in range(args.steps):
            if flush is not None:
                flush()
            a, b = ev(), ev()
            a.record(); fn(args.warmup + s); b.record()
            torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        if world > 1:
            dist.barrier()
        t = torch.tensor([tot], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), t0, time.time()

    line = {"n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "phase": args.phase}
    if args.phase == "bfs":
        hg, emb_h, roots, d = make_inputs(args, rank)
        dg = G.DeviceGraph(hg, dev)
        smp = S.WalkSampler(dg)
        R = min(len(roots), args.bfs_roots)
        rr = roots[np.linspace(0, len(roots) - 1, R).astype(np.int64)]
        holder = {}
        def fn(s):
            holder["t"] = smp.build_trees(rr)
        ms, t0, t1 = time_steps(fn)
        nnz = int(hg.adj.shape[0])
        alg = R * (4.0 * nnz + nnz / 8.0 + 8.0 * n)          # adjacency once + tree row + queue write/read, per root
        k_ms = ms / args.steps
        line.update({"metric": "BFS trees built/sec (gg_bfs_build)", "value": R * world * args.steps / (ms * 1e-3), "unit": "trees/s",
                     "ms_per_step": k_ms, "scaling": "weak",
                     "config": {"workload": "%s N=%d avg_deg=%d: gg_bfs_build_ex of %d roots per GPU" % (gen, n, deg, R), "nnz": nnz,
                                "bottom_up_ratio": smp.bfs_bottom_up_ratio, "reverse_entries": dg.reverse_entries() is not None,
                                "l2_policy": "tree rows (%d MB per step) exceed L2; the adjacency (%d MB) is shared by all roots and stays in L2"
                                             % (R * (nnz // 8) >> 20, nnz * 4 >> 20)},
                     "ms_per_root": k_ms / R, "gpu_launches": args.steps,
                     "roofline": {"bound": "hbm", "kernel": "gg::bfs_kernel", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak,
                                  "unit": "GB/s", "frac": alg / (k_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                                  "algorithmic_bytes_per_launch": alg,
                                  "note": "bytes = per root: adjacency 4*nnz (the top-down sweep's read-once figure; bottom-up levels read "
                                          "less) + tree row nnz/8 + queue 8*N; the builder is latency / issue bound, not HBM bound"}})
    elif args.phase in ("reward", "adam", "update"):
        g = torch.Generator(device=dev); g.manual_seed(args.seed + 5)
        emb = torch.empty((n, ld), dtype=torch.float32, device=dev).normal_(0, 0.5, generator=g)
        if ld > d:
            emb[:, d:] = 0
        bias = torch.zeros(n, dtype=torch.float32, device=dev)
        flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        flush = lambda: flush_buf.zero_()
        if args.phase == "reward":
            # every row is read exactly ONCE per launch (a random perfect matching of the nodes): the algorithmic bytes
            # are then also the compulsory DRAM bytes -- with uniform random pairs each row was read ~8 times per
            # launch and L2 hits pushed "achieved" above the HBM peak
            M = min(args.pairs, n // 2)
            perm = torch.randperm(n, device=dev, generator=g).to(torch.int32)
            i, j = perm[:M].contiguous(), perm[M:2 * M].contiguous()
            out = torch.empty(M, dtype=torch.float32, device=dev)
            def fn(s):
                _cabi.check(lib.gg_pair_reward(M, ptr(i), ptr(j), ptr(emb), ptr(bias), ld, ptr(out), st()), "gg_pair_reward")
            ms, t0, t1 = time_steps(fn, flush)
            k_ms = ms / args.steps
            alg = M * (8.0 * ld + 12)
            line.update({"metric": "discriminator.reward pairs/sec (gg_pair_reward)", "value": M * world * args.steps / (ms * 1e-3),
                         "unit": "pairs/s", "ms_per_step": k_ms, "scaling": "weak", "gpu_launches": args.steps,
                         "config": {"workload": "N=%d n_emb=%d, %d disjoint random pairs per launch (every row read once)" % (n, d, M),
                                    "l2_policy": "L2 flushed between launches (256 MB memset); embedding matrix %d MB" % (n * ld * 4 >> 20)},
                         "roofline": {"bound": "hbm", "kernel": "gg::reward_kernel", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak,
                                      "unit": "GB/s", "frac": alg / (k_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                                      "algorithmic_bytes_per_launch": alg, "note": "8*ld + 12 bytes per pair (two rows, two ids, one bias-free score out)"}})
        else:
            from graphgan_b200.discriminator import Discriminator
            from graphgan_b200 import config as cfg
            cfg.device = str(dev)
            m = Discriminator(n, emb[:, :d], device=dev)
            B = 64
            i = torch.randint(0, n, (B,), device=dev, dtype=torch.int32, generator=g)
            j = torch.randint(0, n, (B,), device=dev, dtype=torch.int32, generator=g)
            lab = (torch.rand(B, device=dev, generator=g) < 0.5).float()
            alg = 24.0 * n * ld
            if args.phase == "adam":
                m.step(i, j, lab)
                def fn(s):
                    m.apply_adam()
                ms, t0, t1 = time_steps(fn)
                k_ms = ms / args.steps
                line.update({"metric": "TF1.8 dense Adam sweeps/sec (gg_adam_apply)", "value": world * args.steps / (ms * 1e-3), "unit": "steps/s",
                             "ms_per_step": k_ms, "scaling": "weak", "gpu_launches": args.steps,
                             "config": {"workload": "N=%d n_emb=%d (ld %d): one dense Adam sweep over E, m, v per step" % (n, d, ld),
                                        "l2_policy": "inputs larger than L2 (E, m, v = %d MB)" % (3 * n * ld * 4 >> 20)},
                             "roofline": {"bound": "hbm", "kernel": "gg::adam_tma_kernel (%s)" % args.adam_path if args.adam_path != "ldg" else "gg::adam_kernel", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": peak,
                                          "unit": "GB/s", "frac": alg / (k_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                                          "algorithmic_bytes_per_launch": alg, "note": "24 * N * ld bytes per step: read + write of E, m, v"}})
            else:
                from graphgan_b200.parallel import DataParallelStep
                dp = DataParallelStep(m, transport=args.transport) if world > 1 else None
                def fn(s):
                    if dp is not None:
                        dp.step(i, j, lab)
                    else:
                        m.step(i, j, lab)
                ms, t0, t1 = time_steps(fn)
                k_ms = ms / args.steps
                extra = dp.stats() if dp is not None else {}
                line.update({"metric": "optimizer steps/sec (64-pair discriminator step, data parallel)", "value": args.steps / (ms * 1e-3),
                             "unit": "steps/s", "ms_per_step": k_ms, "scaling": "strong",
                             "gpu_launches": (4 if world > 1 else 2) * args.steps,
                             "config": {"workload": "N=%d n_emb=%d (ld %d): one 64-pair d_updates step = pair-grad on this rank's slice -> "
                                                    "%s -> merge -> dense Adam sweep" % (n, d, ld, ("ncclAllGather of the compact gradients (C ABI: gg_dp_step)" if args.transport == "nccl" else "peer-memory stores from the gradient kernel + flag wait (C ABI: gg_dp_step, p2p)") if world > 1 else "no collective (1 GPU)"),
                                        "l2_policy": "inputs larger than L2 (E, m, v = %d MB)" % (3 * n * ld * 4 >> 20),
                                        "parallelism": "replicated parameters, batch rows split over %d GPU(s)" % world},
                             "collective": extra,
                             "roofline": {"bound": "hbm", "kernel": "gg::adam_kernel (the sweep dominates the step)", "achieved": alg / (k_ms * 1e-3) / 1e9,
                                          "peak": peak, "unit": "GB/s", "frac": alg / (k_ms * 1e-3) / 1e9 / peak, "traffic": None,
                                          "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                                          "note": "whole step time against the sweep's 24 * N * ld bytes: the collective and the 64-pair gradient are the difference to --phase adam"}})
    line["clocks"] = clocks.stop(t0, t1)
    line["e2e"] = {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "note": "device-resident kernel line (not the BASELINE metric); the plugin-level e2e number is the default --phase sample"}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


_RESULT_FD = None


def emit(line):
    """The ONE JSON line goes to the real stdout; anything libraries print meanwhile (NCCL's version banner on some
    boxes, torchrun notices) was routed to stderr by main()."""
    sys.stdout.flush()
    if _RESULT_FD is not None:
        os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())
    else:
        print(json.dumps(line))
        sys.stdout.flush()


def main():
    global _RESULT_FD
    args = parse()
    try:       # keep fd 1 for the result line only
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)
    except OSError:
        _RESULT_FD = None
    os.environ["GG_ADAM_PATH"] = args.adam_path
    if args.impl == "reference":
        return run_reference(args)
    if args.phase != "sample":
        return run_phase(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
