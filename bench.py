#!/usr/bin/env python
"""bench.py -- the hot path's headline metric on B200: sampled edges/s and gathered-feature GB/s.

One "step" = one mini-batch through the hot path: k-hop neighbour sampling (quiver.pyg.GraphSageSampler.sample) followed
by the feature gather of the sampled nodes (quiver.Feature.__getitem__) -- the two calls of the reference's training
loop (examples/pyg/reddit_quiver.py:116-122) and of its benchmarks (benchmarks/sample/bench_sampler.py:35-46,
benchmarks/feature/bench_feature.py:36-46, whose metric definitions are reused: SEPS counts adj.edge_index columns,
feature bandwidth counts OUTPUT bytes only).

Workloads (--config; BASELINE.json):
  ns  (default) the workload `north_star` states its target on: synthetic power-law CSR, 100 M nodes / ~1 B edges
      (pareto(2) degrees, neighbours drawn in proportion to degree), 256-d fp32 features (1 KiB rows, 102 GB), 1024 seeds,
      fan-out [15,10,5].  N=1: whole table in one GPU's HBM.  N>1: every rank holds a CSR replica (the sampler does not
      shard, SURVEY 8(e)) and the table is placed by ACCESS PROBABILITY (sample_prob -> storage order): the hottest
      --hot-frac (default 40 %) of the rows replicated on every GPU (NCCL broadcast at setup), the rest striped over the N GPUs and read
      one-sidedly over NVLink inside the gather kernel; every rank runs its own batches (weak scaling, no data-path
      collective).
  c1  Reddit-shaped (232 965 nodes, mean degree 492, 602-d, fan-out [25,10]) -- configs[0], the reference's CPU-runnable case
  c2  ogbn-products-shaped (2 449 029 nodes, mean degree 50.5, 100-d, [15,10,5]) -- configs[1], round 1's headline
  c3  R-MAT 10 M nodes / 160 M edges, 256-d, 2 GPUs: 50/50 HBM shard + NVLink P2P gather -- configs[2]
  c4  papers100M-shaped (111 M nodes / 1.6 B edges, 128-d, [20,15,10]), 4 GPUs: hot rows replicated + cold rows in
      pinned host memory -- configs[3]
  c5  mag240m-scale (244 M nodes / 1.7 B edges, 768-d, [25,15]), 8 GPUs: 8-way shard built in place -- configs[4]
Features are a closed formula of (original row id, column), so every rank can recompute any row: every run ASSERTS that the
rows it gathered in a timed batch equal the formula (`parity_checked_rows`) and that n_id / edge_index of the fused call
equal the two-call path.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own CPU sampler + CPU gather on the host cores

Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "torch-quiver_b200"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

# torch's caching allocator: every step returns fresh tensors whose sizes vary with the batch (n_id, edge_index, the gathered
# rows: 0.1-1 GB); with unlimited splitting a large cached block gets carved up by a smaller request and the next large one
# pays a cudaMalloc (13-33 ms next to a 100 GB table).  Blocks above 256 MB are kept whole (a documented PyTorch knob).
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "max_split_size_mb:256")

import torch  # noqa: E402

CONFIGS = {
    "ns": dict(title="north-star: synthetic power-law CSR, 100M nodes / ~1B edges (pareto(2) degrees, degree-proportional "
                     "neighbours), 1024 seeds, fanout [15,10,5], 256-d fp32 features",
               n_nodes=100_000_000, mean_deg=10.0, graph="pareto_degree", feat_dim=256, sizes=[15, 10, 5], batch=1024,
               legacy=False, min_gpus=1),
    "c1": dict(title="Reddit-shaped synthetic CSR (232965 nodes, pareto(2) mean-deg 492), 1024 seeds, fanout [25,10], "
                     "602-d fp32 features",
               n_nodes=232_965, mean_deg=492.0, graph="pareto_uniform", feat_dim=602, sizes=[25, 10], batch=1024,
               legacy=True, min_gpus=1),
    "c2": dict(title="ogbn-products-shaped synthetic CSR (2449029 nodes, pareto(2) mean-deg 50.5), 1024 seeds, fanout "
                     "[15,10,5], 100-d fp32 features",
               n_nodes=2_449_029, mean_deg=50.5, graph="pareto_uniform", feat_dim=100, sizes=[15, 10, 5], batch=1024,
               legacy=True, min_gpus=1),
    "c3": dict(title="synthetic R-MAT (0.57,0.19,0.19,0.05) 10M nodes / 160M edges, 1024 seeds, fanout [15,10,5], 256-d fp32 "
                     "features",
               n_nodes=10_000_000, n_edges=160_000_000, graph="rmat", feat_dim=256, sizes=[15, 10, 5], batch=1024,
               legacy=False, min_gpus=1),
    "c4": dict(title="ogbn-papers100M-shaped synthetic CSR (111059956 nodes, pareto(2) mean-deg 14.5 ~ 1.6B edges, "
                     "degree-proportional neighbours), 1024 seeds, fanout [20,15,10], 128-d fp32 features",
               n_nodes=111_059_956, mean_deg=14.5, graph="pareto_degree", feat_dim=128, sizes=[20, 15, 10], batch=1024,
               legacy=False, min_gpus=1),
    "c5": dict(title="mag240m-scale synthetic CSR (244160499 nodes, pareto(2) mean-deg 7 ~ 1.7B edges, degree-proportional "
                     "neighbours), 1024 seeds, fanout [25,15], 768-d fp32 features",
               n_nodes=244_160_499, mean_deg=7.0, graph="pareto_degree", feat_dim=768, sizes=[25, 15], batch=1024,
               legacy=False, min_gpus=8),
}
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r2_gather_traffic.json")  # ncu dram bytes of the shipped gather kernel


def env_int(name, default):
    return int(os.environ.get(name, default))


# ----------------------------------------------------------------------------------------------------------------------
# synthetic workload (device-side generation; identical on every rank)
# ----------------------------------------------------------------------------------------------------------------------
def _pareto_degrees(n_nodes, mean_deg, g, device):
    raw = (1.0 - torch.rand(n_nodes, generator=g, device=device, dtype=torch.float64)).pow(-0.5)  # pareto(alpha=2)
    deg = (raw * (mean_deg / raw.mean())).floor().long().clamp_(max=n_nodes - 1)
    indptr = torch.zeros(n_nodes + 1, dtype=torch.long, device=device)
    indptr[1:] = deg.cumsum(0)
    return deg, indptr


def make_graph_legacy(device, n_nodes, mean_deg, seed=0):
    """Round 1's generator (kept bit for bit so c1 / c2 numbers stay comparable): uniform neighbours, one sort."""
    g = torch.Generator(device=device).manual_seed(seed)
    deg, indptr = _pareto_degrees(n_nodes, mean_deg, g, device)
    n_edges = int(indptr[-1])
    row = torch.repeat_interleave(torch.arange(n_nodes, device=device), deg)
    col = torch.randint(0, n_nodes, (n_edges, ), generator=g, device=device)
    key, _ = torch.sort(row * n_nodes + col)  # columns sorted inside each row, as scipy's COO->CSR gives the reference
    return indptr, key % n_nodes


def make_graph_pareto(device, n_nodes, mean_deg, by_degree, seed=0, chunk_edges=1 << 26):
    """Power-law CSR built chunk by chunk (a 1 B-edge graph never needs more than a few GB of scratch).  by_degree: a
    neighbour is the owner of a uniformly drawn edge slot, i.e. node v is picked with probability deg(v)/E (Chung-Lu
    style), so high-degree nodes are also the frequently SAMPLED ones, as in real power-law graphs."""
    g = torch.Generator(device=device).manual_seed(seed)
    deg, indptr = _pareto_degrees(n_nodes, mean_deg, g, device)
    n_edges = int(indptr[-1])
    indices = torch.empty(n_edges, dtype=torch.long, device=device)
    cuts = torch.searchsorted(indptr, torch.arange(0, n_edges, chunk_edges, device=device), right=True) - 1
    cuts = torch.unique(torch.cat([cuts.clamp_(min=0), torch.tensor([n_nodes], device=device)])).tolist()
    if cuts[0] != 0:
        cuts = [0] + cuts
    for a, b in zip(cuts[:-1], cuts[1:]):
        ea, eb = int(indptr[a]), int(indptr[b])
        if eb == ea:
            continue
        row = torch.repeat_interleave(torch.arange(a, b, device=device), deg[a:b])
        if by_degree:
            slot = torch.randint(0, n_edges, (eb - ea, ), generator=g, device=device)
            col = torch.searchsorted(indptr, slot, right=True) - 1
            del slot
        else:
            col = torch.randint(0, n_nodes, (eb - ea, ), generator=g, device=device)
        key, _ = torch.sort(row * n_nodes + col)
        indices[ea:eb] = key % n_nodes
        del row, col, key
    return indptr, indices


def make_graph_rmat(device, n_nodes, n_edges, seed=2, abcd=(0.57, 0.19, 0.19, 0.05)):
    """R-MAT over 2^ceil(log2 n) ids, trimmed to n_nodes (ids beyond are dropped and regenerated until n_edges remain);
    duplicate edges kept (sampling is by CSR position).  Same recursion as tests/graphs.py:rmat_csr, on the device."""
    g = torch.Generator(device=device).manual_seed(seed)
    scale = (n_nodes - 1).bit_length()
    a, b, c, _ = abcd
    keys = []
    have = 0
    while have < n_edges:
        m = min(1 << 26, int((n_edges - have) * 1.6) + 1024)
        src = torch.zeros(m, dtype=torch.long, device=device)
        dst = torch.zeros(m, dtype=torch.long, device=device)
        for _ in range(scale):
            r = torch.rand(m, generator=g, device=device)
            down = r >= a + b
            right = ((r >= a) & (r < a + b)) | (r >= a + b + c)
            src = (src << 1) | down
            dst = (dst << 1) | right
        keep = (src < n_nodes) & (dst < n_nodes)
        k = (src * n_nodes + dst)[keep][:n_edges - have]
        keys.append(k)
        have += k.numel()
    key, _ = torch.sort(torch.cat(keys))
    del keys
    src = key // n_nodes
    indptr = torch.searchsorted(src, torch.arange(n_nodes + 1, device=device))
    return indptr, key % n_nodes


def make_graph(device, cfg, seed=0):
    if cfg["graph"] == "rmat":
        return make_graph_rmat(device, cfg["n_nodes"], cfg["n_edges"])
    if cfg["legacy"]:
        return make_graph_legacy(device, cfg["n_nodes"], cfg["mean_deg"], seed)
    return make_graph_pareto(device, cfg["n_nodes"], cfg["mean_deg"], cfg["graph"] == "pareto_degree", seed)


def make_seed_batches(n_batches, n_nodes, batch, seed=1, legacy=False):
    """Unique seeds per batch.  legacy: round 1's randperm (fine up to a few M nodes); else draw-and-dedup (a randperm
    of 100 M ids per batch would take seconds)."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_batches):
        if legacy:
            b = torch.randperm(n_nodes, generator=g)[:batch]
        else:
            b = torch.empty(0, dtype=torch.long)
            while b.numel() < batch:
                cand = torch.unique(torch.cat([b, torch.randint(0, n_nodes, (batch + 64, ), generator=g)]))
                b = cand[torch.randperm(cand.numel(), generator=g)][:batch]
        out.append(b.pin_memory() if torch.cuda.is_available() else b)
    return out


def feat_formula(ids, dim, device):
    """Feature row of ORIGINAL node id i: x[i, j] = ((i * 1000003 + j * 7919) mod 2^20) / 2^20 -- exact in fp32, cheap to
    evaluate anywhere (GPU fill, CPU fill, per-rank parity check)."""
    ids = ids.to(device=device, dtype=torch.long)
    v = (ids[:, None] * 1000003 + torch.arange(dim, device=device, dtype=torch.long)[None, :] * 7919) & 0xFFFFF
    return v.to(torch.float32) * (1.0 / 1048576.0)


DUMP_BYTES = 60 << 20  # --dump-outputs: all arrays together, under 64 MB (10^6 bytes) with the .npy headers


def last_step_outputs(n_id, adjs, x):
    """What the timed call returned in its last step, as host arrays: ids and sizes as float64 (exact below 2^53), the
    gathered rows as float32."""
    out = {"n_id": n_id.cpu().double().numpy()}
    for i, a in enumerate(adjs):
        out[f"adj{i}_edge_index"] = a.edge_index.cpu().double().numpy()
        out[f"adj{i}_size"] = torch.as_tensor(a.size).double().numpy()
    out["x"] = x.cpu().float().numpy()
    return out


def dump_outputs(path, arrays, budget=DUMP_BYTES, seed=0):
    """Write every array as path/<name>.npy, smallest first, each within an even share of what is left of `budget`.  An
    array larger than its share is replaced by a sample along its longest axis, drawn by a generator with a fixed seed;
    <name>_index.npy (float64) holds the sampled positions, so that two runs with the same arguments write the same files."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    left = budget
    for i, (name, a) in enumerate(sorted(arrays.items(), key=lambda t: t[1].nbytes)):
        share = left // (len(arrays) - i)
        if a.nbytes > share:
            axis = int(np.argmax(a.shape))
            m = share // (a.nbytes // a.shape[axis] + 8)
            pick = np.sort(np.random.default_rng(seed).choice(a.shape[axis], m, replace=False))
            np.save(os.path.join(path, f"{name}_index.npy"), pick.astype(np.float64))
            a = np.take(a, pick, axis=axis)
            left -= pick.nbytes
        np.save(os.path.join(path, f"{name}.npy"), a)
        left -= a.nbytes


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md)."""
    FIELDS = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index, self.samples, self.stop_flag = gpu_index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.check_output(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                               "-i", str(self.gpu_index)], text=True, timeout=5)
                self.samples.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i] == "Active" for s in self.samples)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": int(self.samples[0][1]),
                "reasons": reasons, "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's own CPU implementation of the path (oracle/_ref when built)
# ----------------------------------------------------------------------------------------------------------------------
def host_threads():
    """All the host threads this process may use.  torchrun exports OMP_NUM_THREADS=1, which would leave the reference's
    CPU gather (and its OpenMP build) on one core: undo that for the reference arm."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


def reference_cpu_setup(indptr_cpu, indices_cpu):
    """The reference CPU classes compiled from its own sources (oracle/_ref).  Preference: a reference build that is
    already imported (one process can hold only one: they register the same pybind types), else the CUDA build (it carries
    the same CPU classes and lets `ref_gpu_baseline` run in the same process), else the as-shipped CPU build (its
    at::parallel_for runs serially without -fopenmp, setup.py:58-69); QV_REF_VARIANT=omp asks for the -fopenmp build.
    Returns None when no build of the reference is present."""
    from oracle import oracle
    host_threads()
    ext, openmp = None, False
    if os.environ.get("QV_REF_VARIANT", "") == "omp":
        ext, openmp = oracle.load_reference(openmp=True), True
        openmp = ext is not None and ext.__name__.endswith("_omp")
    if ext is None:
        ext = oracle.load_reference_cuda() or oracle.load_reference(openmp=False)
    if ext is None:
        return None
    return {"ext": ext, "openmp": openmp, "kind": "reference", "module": ext.__name__,
            "quiver": ext.cpu_quiver_from_csr_array(indptr_cpu, indices_cpu)}


class _OraclePort:
    """sample_neighbor / reindex_single of oracle/qv_oracle.c behind the reference extension's call shapes."""

    def __init__(self, oracle, indptr, indices):
        self.o, self.indptr, self.indices = oracle, indptr.numpy(), indices.numpy()

    def sample_neighbor(self, nodes, k):
        out, cnt = self.o.sample_neighbor(self.indptr, self.indices, nodes.numpy(), int(k))
        return torch.from_numpy(out), torch.from_numpy(cnt)

    def reindex_single(self, nodes, out, cnt):
        return tuple(torch.from_numpy(a) for a in self.o.reindex(nodes.numpy(), out.numpy(), cnt.numpy()))


def oracle_port_setup(indptr_cpu, indices_cpu):
    from oracle import oracle
    host_threads()
    return {"ext": None, "openmp": False, "kind": "port", "module": "oracle/qv_oracle.c",
            "quiver": _OraclePort(oracle, indptr_cpu, indices_cpu)}


def host_table(n_nodes, dim, cap_bytes=32 << 30):
    """The CPU arm's feature table: the formula's values do not matter for timing, its SIZE does (random 4*dim-byte rows
    out of a table far larger than the caches).  Up to cap_bytes are materialised (first-touched by a parallel fill);
    larger tables are folded: row id -> id mod rows."""
    rows = int(min(n_nodes, cap_bytes // (dim * 4)))
    x = torch.empty(rows, dim)
    x.fill_(0.5)
    return x, rows


def reference_cpu_step(ref, seeds, x_cpu, sizes, fold):
    """GraphSageSampler.sample restated over the reference's C++ bindings (sage_sampler.py:118-147, mode='CPU') +
    the CPU gather of bench_feature.py:62-66.  Returns (edges, rows, t_sample, t_gather)."""
    t0 = time.perf_counter()
    nodes, edges = seeds, 0
    for size in sizes:
        out, cnt = ref["quiver"].sample_neighbor(nodes, size)
        frontier, row_idx, col_idx = ref["quiver"].reindex_single(nodes, out, cnt)
        edges += out.numel()
        nodes = frontier
    t1 = time.perf_counter()
    rows = x_cpu[nodes % fold] if fold < (1 << 62) else x_cpu[nodes]
    t2 = time.perf_counter()
    return edges, rows.shape[0], t1 - t0, t2 - t1


def _describe(ref, x_rows, n_nodes):
    what = (f"reference CPU classes compiled from its sources ({ref['module']}: "
            + ("-fopenmp" if ref["openmp"] else "as shipped, at::parallel_for serial") + ")"
            if ref["kind"] == "reference" else "oracle/qv_oracle.c port, 1 core (oracle/_ref not built)")
    table = "full host table" if x_rows >= n_nodes else f"host table folded to {x_rows} rows (ids mod rows)"
    return f"{what} for sample+reindex; torch CPU gather on {torch.get_num_threads()} threads, {table}; " \
           f"host has {os.cpu_count()} cores"


def cpu_baseline_sample(cfg, indptr_cpu, indices_cpu, batches_host, n_b=4, budget_s=25.0):
    """The `cpu_baseline` object of the N=1 line: the reference's CPU path timed on a bounded sample (up to n_b batches of
    the same workload, stopping after ~budget_s of CPU work) on this box's host cores."""
    ref = reference_cpu_setup(indptr_cpu, indices_cpu) or oracle_port_setup(indptr_cpu, indices_cpu)
    x_cpu, rows = host_table(cfg["n_nodes"], cfg["feat_dim"])
    fold = rows if rows < cfg["n_nodes"] else (1 << 62)
    e = r = done = 0
    ts = tg = 0.0
    reference_cpu_step(ref, batches_host[0], x_cpu, cfg["sizes"], fold)
    t0 = time.perf_counter()
    for b in batches_host[1:1 + n_b]:
        ee, rr, a, gg = reference_cpu_step(ref, b, x_cpu, cfg["sizes"], fold)
        e, r, ts, tg, done = e + ee, r + rr, ts + a, tg + gg, done + 1
        if time.perf_counter() - t0 > budget_s:
            break
    tt = time.perf_counter() - t0
    return {"value": e / tt, "unit": "edges/s", "cores": torch.get_num_threads() if ref["openmp"] else 1,
            "kind": ref["kind"], "sample": f"{done} batches of the same workload; " + _describe(ref, rows, cfg["n_nodes"]),
            "seps_sampler_only": e / ts, "feature_gather_GiBps": r * cfg["feat_dim"] * 4 / tg / 2**30,
            "gather_threads": torch.get_num_threads()}


def run_reference(args, cfg, rank, world):
    if rank != 0:
        return None
    torch.manual_seed(0)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    indptr, indices = make_graph(dev, cfg)
    indptr_cpu, indices_cpu = indptr.cpu(), indices.cpu()
    del indptr, indices
    if dev == "cuda":
        torch.cuda.empty_cache()
    batches = make_seed_batches(args.steps + args.warmup, cfg["n_nodes"], cfg["batch"], seed=1, legacy=cfg["legacy"])
    ref = reference_cpu_setup(indptr_cpu, indices_cpu)
    note = None
    if ref is None:
        # bench contract for this tier: the oracle always exists -- but a line measured on OUR port must say so loudly
        ref = oracle_port_setup(indptr_cpu, indices_cpu)
        note = "oracle/_ref (the reference's own code) was not built: this line times oracle/qv_oracle.c, the repo's " \
               "single-core restatement of the reference GPU algorithm -- NOT the reference's code"
    x_cpu, rows = host_table(cfg["n_nodes"], cfg["feat_dim"])
    fold = rows if rows < cfg["n_nodes"] else (1 << 62)
    for b in batches[:args.warmup]:
        reference_cpu_step(ref, b, x_cpu, cfg["sizes"], fold)
    edges = n_rows = done = 0
    ts = tg = 0.0
    t0 = time.perf_counter()
    for b in batches[args.warmup:]:
        e, r, a, g = reference_cpu_step(ref, b, x_cpu, cfg["sizes"], fold)
        edges, n_rows, ts, tg, done = edges + e, n_rows + r, ts + a, tg + g, done + 1
    total = time.perf_counter() - t0
    cores = torch.get_num_threads() if ref["openmp"] else 1
    value = edges / total
    base = {"kind": ref["kind"], "cores": cores, "value": value, "unit": "edges/s",
            "sample": f"{done} batches of the full workload; " + _describe(ref, rows, cfg["n_nodes"]),
            "seps_sampler_only": edges / ts, "feature_gather_GiBps": n_rows * cfg["feat_dim"] * 4 / tg / 2**30,
            "gather_threads": torch.get_num_threads()}
    out = {"metric": "sampled_edges_per_s (k-hop sample + feature gather per step)", "value": value, "unit": "edges/s",
           "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "int64", "data": "synthetic",
           "config": {"workload": cfg["title"], "config_key": args.config, "where": "host CPU"},
           "reference_procs": 1,
           "reference_procs_note": "ONE CPU process whatever --gpus says (rank 0 runs, the other ranks exit): at N GPUs the "
                                   "driver's ratio compares N GPUs with one CPU process, not N with N",
           "cpu_baseline": base, "gpu_launches": 0,
           "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if note:
        out["reference_unavailable"] = note
    return out


# ----------------------------------------------------------------------------------------------------------------------
# the reference's CUDA kernels on the same GPU (oracle/_ref/torch_quiver_ref_cuda*.so, N=1 only)
# ----------------------------------------------------------------------------------------------------------------------
def ref_gpu_baseline(cfg, dev, indptr, indices, batches_dev, nid_list, n_batches=5):
    """SURVEY 2.2's bar: the reference's own kernels recompiled for sm_100a, same GPU, same batches.  Sampler = the hop loop
    of sage_sampler.py:118-147 over Quiver.sample_neighbor / reindex_single; gather = ShardTensor.__getitem__ over a
    bounded HBM table (ids folded modulo its rows: the reference can only create shards from CPU tensors)."""
    from oracle import oracle
    ref = oracle.load_reference_cuda()
    if ref is None:
        return {"unavailable": "oracle/_ref/torch_quiver_ref_cuda*.so not built"}
    q = ref.device_quiver_from_csr_array(indptr, indices, torch.zeros(1, dtype=torch.long), dev.index, True)

    def sample(seeds):
        nodes, edges = seeds, 0
        for size in cfg["sizes"]:
            out, cnt = q.sample_neighbor(0, nodes, size)
            nodes, _, _ = q.reindex_single(nodes, out, cnt)
            edges += out.numel()
        return nodes, edges

    sample(batches_dev[0])
    torch.cuda.synchronize()
    edges, per_batch = 0, []
    for b in batches_dev[1:1 + n_batches]:
        t0 = time.perf_counter()
        e = sample(b)[1]
        torch.cuda.synchronize()
        per_batch.append((time.perf_counter() - t0, e))
        edges += e
    # the reference allocates ~10 thrust vectors per hop with cudaMalloc/cudaFree; next to a 100 GB table single calls take
    # 10-30 ms now and then, so the figure is the MEDIAN batch (min / max alongside)
    per_batch.sort(key=lambda t: t[0] / max(t[1], 1))
    t_med, e_med = per_batch[len(per_batch) // 2]
    t_sample = t_med * n_batches * (edges / max(e_med * n_batches, 1))
    dim = cfg["feat_dim"]
    rows = int(min(cfg["n_nodes"], (4 << 30) // (dim * 4)))
    x = torch.empty(rows, dim).fill_(0.25)
    st = ref.ShardTensor(dev.index)
    st.append(x, dev.index)
    ids = [(n % rows) if rows < cfg["n_nodes"] else n for n in nid_list[:n_batches]]
    st[ids[0]]
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    n_rows = 0
    for i in ids:
        st[i]
        n_rows += i.numel()
    e1.record()
    torch.cuda.synchronize()
    t_gather = e0.elapsed_time(e1) * 1e-3
    del st, q
    return {"what": "the reference's CUDA extension compiled unmodified for sm_100a (oracle/build_ref_cuda.py), same GPU, "
                    "same seed batches", "seps_sampler_only": edges / t_sample, "sample_ms_per_step": t_sample / n_batches * 1e3,
            "feature_gather_GBps": n_rows * dim * 4 / t_gather / 1e9, "gather_ms_per_step": t_gather / n_batches * 1e3,
            "edges_per_s_step": edges / (t_sample + t_gather),
            "gather_table": f"{rows} rows in HBM" + ("" if rows >= cfg["n_nodes"] else " (ids folded modulo rows)"),
            "batches": n_batches, "seps_sampler_min_max": [min(e / t for t, e in per_batch), max(e / t for t, e in per_batch)],
            "timing": "sampler: wall clock around synchronising calls (the reference blocks on the host several times per "
                      "hop and allocates with cudaMalloc per call), median batch; gather: CUDA events"}


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
def build_feature(args, cfg, dev, rank, world, indptr, indices, sampler):
    """Place the feature table; returns (feature, store-or-feature for the fused call, feature_order (device) or None,
    placement text, info dict, x_cpu or None)."""
    import quiver
    from quiver.shard_tensor import build_tiered_inplace
    n, dim = cfg["n_nodes"], cfg["feat_dim"]
    small = n * dim * 4 <= (4 << 30)
    if world == 1 and small and not args.device_build:
        # the reference-facing path: CPU tensor -> quiver.Feature.from_cpu_tensor (degree order, budget, tiers)
        topo = sampler.csr_topo
        x_cpu = feat_formula(torch.arange(n), dim, "cpu")
        feature = quiver.Feature(rank=dev.index, device_list=[dev.index], device_cache_size="8G",
                                 cache_policy="device_replicate", csr_topo=topo)
        feature.from_cpu_tensor(x_cpu)
        return feature, feature, feature.feature_order, \
            "1 GPU: whole table in local HBM via Feature.from_cpu_tensor, degree-ordered (feature_order folded into the " \
            "gather)", {"hot": (0, 0), "stripe": (0, n), "striped": (0, n), "cold": (n, n), "world": 1}, x_cpu
    # ---- storage order --------------------------------------------------------------------------------------------
    order_kind = args.order
    if order_kind == "auto":
        order_kind = "prob" if world > 1 or cfg["graph"] != "pareto_uniform" else "degree"
    if order_kind == "prob":
        # access probability of every node after len(sizes) hops from uniformly drawn seeds (sample_prob: the cal_next
        # kernel; sage_sampler.py:149-157) -> hottest rows first
        # (GraphSageSampler.sample_prob marks a train set with probability 1; here every node is a seed with the same small
        #  probability -- 100 batches' worth -- so the seeds themselves do not jump the queue)
        score = torch.full((n, ), min(1.0, 100.0 * cfg["batch"] / n), device=dev)
        for size in cfg["sizes"]:
            cur = torch.zeros(n, device=dev)
            sampler.quiver.cal_neighbor_prob(0, score, cur, size)
            score = cur
        del cur
    elif order_kind == "degree":
        score = (indptr[1:] - indptr[:-1]).to(torch.float32)
    else:
        score = None
    if score is not None:
        inv_order = torch.sort(score, descending=True, stable=True)[1]  # storage row -> original id
        del score
        feature_order = torch.empty_like(inv_order)
        feature_order[inv_order] = torch.arange(n, device=dev)
    else:
        inv_order, feature_order = None, None

    def fill(view, lo, hi):
        ids = inv_order[lo:hi] if inv_order is not None else torch.arange(lo, hi, device=dev)
        view.copy_(feat_formula(ids, dim, dev))

    hot = int(n * args.hot_frac) if world > 1 else 0
    cold = int(n * args.cold_frac)
    store, info = build_tiered_inplace(dev.index, n, [dim], torch.float32, fill, hot_rows=hot, cold_rows=cold)
    del inv_order
    torch.cuda.empty_cache()
    feature = quiver.Feature.from_tiered_store(dev.index, store, feature_order)
    placement = (f"{order_kind}-ordered rows built in place on the GPUs: "
                 + (f"hottest {args.hot_frac:.0%} replicated on every GPU (NCCL broadcast at setup), " if hot else "")
                 + (f"{1 - args.hot_frac - args.cold_frac if world > 1 else 1 - args.cold_frac:.0%} "
                    f"{'striped over the ' + str(world) + ' GPUs (CUDA IPC peer mappings, one-sided NVLink reads)' if world > 1 else 'in local HBM'}")
                 + (f", coldest {args.cold_frac:.0%} in one pinned host copy (zero-copy over PCIe)" if cold else ""))
    return feature, feature, feature_order, placement, info, None


def run_ours(args, cfg, rank, world, local_rank):
    import torch.distributed as dist

    import quiver
    from torch_quiver import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    n, dim, sizes, batch = cfg["n_nodes"], cfg["feat_dim"], cfg["sizes"], cfg["batch"]
    row_bytes = dim * 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- setup (untimed) ---------------------------------------------------------------------------------------------
    t_setup = time.perf_counter()
    indptr, indices = make_graph(dev, cfg)
    n_edges = indices.numel()
    torch.cuda.empty_cache()
    if args.uva:  # indices stay in (pinned) host memory, read zero-copy
        topo = quiver.CSRTopo(indptr=indptr.cpu(), indices=indices.cpu())
        del indices
    else:  # device tensors go straight in: no host round trip of a 9 GB CSR
        topo = quiver.CSRTopo(indptr=indptr, indices=indices)
    sampler = quiver.pyg.GraphSageSampler(topo, sizes, device=local_rank, mode="UVA" if args.uva else "GPU")
    sampler.overlap = args.overlap  # opt-in pipelining of sample(i+1) with gather(i) on a private stream (default off)
    sampler.inputs_ready = True  # the device-resident seed batches below are materialised before the timed region
    if world > 1:
        quiver.init_p2p(list(range(world)))
    feature, fuse_target, feature_order, placement, info, x_cpu = build_feature(args, cfg, dev, rank, world, indptr,
                                                                                 indices if not args.uva else None, sampler)
    feature._my_store().shard_tensor.gather_variant = args.gather_variant
    n_rep = max(1, args.repeats)
    n_batches = args.warmup + n_rep * args.steps
    batches_host = make_seed_batches(n_batches, n, batch, seed=1 + rank, legacy=cfg["legacy"])
    batches_dev = [b.to(dev) for b in batches_host]
    timed = [batches_dev[args.warmup + r * args.steps: args.warmup + (r + 1) * args.steps] for r in range(n_rep)]
    timed_host = batches_host[args.warmup: args.warmup + args.steps]
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t_setup

    # ---- warm-up -----------------------------------------------------------------------------------------------------
    # torch's caching allocator first: `feature[n_id]` returns a fresh [rows, dim] tensor per call and rows varies per batch,
    # so without two cached blocks of the largest possible size a step now and then pays a cudaMalloc (13-33 ms measured
    # next to a 100 GB table) -- steady state for a training loop, noise for a 20-step timed region
    cap_rows = min(batch * int(torch.tensor([1 + s_ for s_ in sizes]).prod()), n + batch)
    _warm = [torch.empty(cap_rows, dim, device=dev) for _ in range(2)]
    del _warm
    clocks = ClockSampler(local_rank)
    clocks.start()
    for b in batches_dev[:args.warmup]:
        n_id, _, adjs = sampler.sample(b)
        res = feature[n_id]
    barrier()
    # The timed regions below last ~10 ms -- shorter than one nvidia-smi poll.  Keep the SAME step loop running for
    # ~0.7 s first (untimed) so the clock / throttle record is taken under this workload's load.  Same batches, same order
    # and the same tensor lifetimes as region A (`res` of step i-1 is alive while step i allocates): an unsplit cached block
    # serves a request only when it is < 20 MB larger, so the allocator's cache must have seen exactly this sequence -- or a
    # step of the per-phase region pays a cudaMalloc now and then (gather_ms_per_step 2.3 ms instead of 0.15 in one c2 run).
    t_probe = time.perf_counter()
    while time.perf_counter() - t_probe < 0.7:
        for b in timed[0]:
            n_id, _, adjs = sampler.sample(b)
            res = feature[n_id]
    barrier()

    # ---- timed region A: K steps as the reference's two calls, inputs resident in HBM, with per-phase events -------------
    want_overlap = sampler.overlap
    sampler.overlap = False
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * args.steps + 1)]
    launches_s0 = _lib.launch_count()
    edges = rows = 0
    hop_bytes = 0  # SURVEY 8(d): B_hop = 40*E + 40*S + 8*F algorithmic bytes per hop
    nid_keep, adj_keep = [], None
    # the timed batches' node lists are kept (parity check, roofline loop) in ONE buffer allocated up front: tensors created
    # and kept inside the loop would pin the remainders of torch's cached blocks and force a cudaMalloc per step
    keep_cap = min(batch * int(torch.tensor([1 + s_ for s_ in sizes]).prod()), n + batch)
    keep_buf = torch.empty(args.steps * keep_cap, dtype=torch.long, device=dev)
    dbg = os.environ.get("QV_BENCH_DEBUG")
    if dbg:
        print("[dbg] device allocs before region A:", torch.cuda.memory_stats().get("num_device_alloc"), file=sys.stderr)
    barrier()
    ev[0].record()
    for i, b in enumerate(timed[0]):
        n_id, _, adjs = sampler.sample(b)
        ev[3 * i + 1].record()
        th0 = time.perf_counter()
        res = feature[n_id]
        th1 = time.perf_counter()
        ev[3 * i + 2].record()
        if dbg:
            torch.cuda.synchronize()
            print(f"[dbg] step {i}: feature[n_id] host {1e3 * (th1 - th0):.3f} ms, then sync {1e3 * (time.perf_counter() - th1):.3f} ms, "
                  f"rows {n_id.numel()}", file=sys.stderr)
        edges += sum(a.edge_index.shape[1] for a in adjs)
        hop_bytes += sum(40 * a.edge_index.shape[1] + 40 * int(a.size[1]) + 8 * int(a.size[0]) for a in adjs)
        rows += n_id.numel()
        keep = keep_buf[i * keep_cap: i * keep_cap + n_id.numel()]
        keep.copy_(n_id)
        nid_keep.append(keep)
        if i == args.steps - 1:
            adj_keep = adjs
        ev[3 * i + 3].record()
    barrier()
    launches_serial = _lib.launch_count() - launches_s0
    if dbg:
        print("[dbg] device allocs after region A:", torch.cuda.memory_stats().get("num_device_alloc"), file=sys.stderr)
    serial_ms = ev[0].elapsed_time(ev[3 * args.steps])
    sample_ms = sum(ev[3 * i].elapsed_time(ev[3 * i + 1]) for i in range(args.steps))
    gather_ms = sum(ev[3 * i + 1].elapsed_time(ev[3 * i + 2]) for i in range(args.steps))
    sampler.overlap = want_overlap

    # ---- parity, inside the run: gathered rows == the closed formula of (original id, column), on every rank; fused call
    #      == two calls (n_id, every edge_index, rows) ------------------------------------------------------------------
    parity_rows = 0
    for j in (0, args.steps - 1):
        got = feature[nid_keep[j]]
        want = feat_formula(nid_keep[j], dim, dev)
        assert torch.equal(got, want), f"rank {rank}: gathered rows differ from the feature formula (batch {j})"
        parity_rows += got.shape[0]
        del got, want
    tier_rows = None
    if feature_order is not None and info["world"] >= 1:
        srow = feature_order[nid_keep[0]]
        lo, hi = info["stripe"]
        h0, h1 = info["hot"]
        c0, c1 = info["cold"]
        tier_rows = {"hot_local": int(((srow >= h0) & (srow < h1)).sum()), "stripe_local": int(((srow >= lo) & (srow < hi)).sum()),
                     "host": int(((srow >= c0) & (srow < c1)).sum()), "total": int(srow.numel())}
        tier_rows["peer"] = tier_rows["total"] - tier_rows["hot_local"] - tier_rows["stripe_local"] - tier_rows["host"]
        del srow

    # ---- timed region A': the same K steps through sample_and_gather (gather enqueued behind the last hop, frontier size
    #      read on the device: no GPU idle while the host learns the sizes) -- `value`.  n_rep repeats on distinct batches. --
    rep_ms = []
    fused = not args.no_fuse and not want_overlap
    launches = launches_serial
    if fused:
        for b in batches_dev[:args.warmup]:
            sampler.sample_and_gather(b, fuse_target)
        n_id_f, _, adjs_f, res_f = sampler.sample_and_gather(timed[0][-1], fuse_target)
        assert torch.equal(n_id_f, nid_keep[-1]) and torch.equal(res_f, feature[nid_keep[-1]])
        assert all(torch.equal(a.edge_index, b_.edge_index) for a, b_ in zip(adjs_f, adj_keep))
        del n_id_f, adjs_f, res_f
    del adj_keep
    for r in range(n_rep):
        launches0 = _lib.launch_count()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        edges_r = 0
        barrier()
        a0.record()
        for b in timed[r]:
            if fused:
                n_id, _, adjs, res = sampler.sample_and_gather(b, fuse_target)
            else:
                n_id, _, adjs = sampler.sample(b)
                res = feature[n_id]
            edges_r += sum(a.edge_index.shape[1] for a in adjs)
        a1.record()
        barrier()
        rep_ms.append((a0.elapsed_time(a1), edges_r))
        launches = _lib.launch_count() - launches0
    # the last step's results are copied to the host here, between timed regions, and written at the end of the run
    last_outputs = last_step_outputs(n_id, adjs, res) if args.dump_outputs and rank == 0 else None
    rep_rates = sorted(e / (ms * 1e-3) for ms, e in rep_ms)
    # the reported K-step region is the median repeat (by rate)
    med = sorted(rep_ms, key=lambda t: t[1] / t[0])[len(rep_ms) // 2]
    total_ms, edges_val = med

    # ---- timed region B: end to end through the public API with HOST seeds -------------------------------------------
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_edges = 0
    d2h = 0
    e0.record()
    for b in timed_host:
        n_id, _, adjs = sampler.sample(b)  # pinned host seeds -> H2D inside the call
        res = feature[n_id]
        probe = res[-1, :1].cpu()  # completes the step on the host (4 bytes) + the sampler's size read-back
        d2h = 4 + 8 * 4 * 9
        e2e_edges += sum(a.edge_index.shape[1] for a in adjs)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    e2e_fused_ms = 0.0
    if fused:  # the same end-to-end loop through the call `value` uses
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        probe_host = torch.empty(1, dtype=torch.float32).pin_memory()
        e0.record()
        for b in timed_host:
            n_id, _, adjs, res = sampler.sample_and_gather(b, fuse_target)
            probe_host.copy_(res[-1, :1], non_blocking=True)  # the step's result reaches the host (4 bytes + the sampler's
            torch.cuda.current_stream().synchronize()          # size read-back) before the next step starts
        e1.record()
        barrier()
        e2e_fused_ms = e0.elapsed_time(e1)
    clock_summary = clocks.summary()
    del res

    # ---- roofline of the dominant kernel (the gather): back-to-back launches over the timed batches' node lists -------
    alg_bytes_per_row = 2 * row_bytes + 8 + (8 if feature_order is not None else 0)  # SURVEY 8(d): read + write + index (+ order)
    barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # (outputs are pre-allocated and the C-ABI call is issued directly so the host never starves the queue: the interval
    #  between the two events is back-to-back executions of the gather kernel and nothing else)
    st_raw = feature._my_store().shard_tensor
    max_rows = max(x.numel() for x in nid_keep)
    outs = [torch.empty(max_rows, dim, device=dev) for _ in range(2)]
    for j, x in enumerate(nid_keep[:2]):
        st_raw.gather(x, feature_order, out=outs[j][:x.numel()])
    barrier()
    reps = 0
    r0.record()
    for _ in range(3):
        for j, x in enumerate(nid_keep):
            st_raw.gather(x, feature_order, out=outs[j % 2][:x.numel()])
            reps += 1
    r1.record()
    barrier()
    kern_ms = r0.elapsed_time(r1) / reps
    if dbg:
        print(f"[dbg] rank {rank}: gather kernel {kern_ms:.3f} ms per launch, tiers {tier_rows}", file=sys.stderr)
    rows_per_launch = rows / args.steps
    achieved = rows_per_launch * alg_bytes_per_row / (kern_ms * 1e-3) / 1e9
    del outs

    # ---- a large-batch point (64 k seeds): the sampler where bandwidth, not launch latency, matters (SURVEY 8(d)) -------
    big = None
    if not args.no_large_batch:
        big_batches = [b.to(dev) for b in make_seed_batches(3, n, 65536, seed=99 + rank, legacy=cfg["legacy"])]
        try:
            sampler.sample(big_batches[0])
            barrier()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            big_edges = big_bytes = 0
            b0.record()
            for bb in big_batches:
                _, _, adjs = sampler.sample(bb)
                big_edges += sum(a.edge_index.shape[1] for a in adjs)
                big_bytes += sum(40 * a.edge_index.shape[1] + 40 * int(a.size[1]) + 8 * int(a.size[0]) for a in adjs)
            b1.record()
            barrier()
            big_ms = b0.elapsed_time(b1)
            big = {"seeds": 65536, "seps": big_edges / (big_ms * 1e-3), "algorithmic_GBps": big_bytes / (big_ms * 1e-3) / 1e9,
                   "frac_of_hbm_peak": big_bytes / (big_ms * 1e-3) / 1e9 / hbm_peak, "ms_per_batch": big_ms / 3}
        except torch.OutOfMemoryError:
            big = {"skipped": "out of memory next to the feature table"}
            barrier()
        del big_batches

    # ---- informational: the opt-in fast (non-reference-stream) sampler on the same batches ------------------------------
    fast = None
    if not args.no_large_batch:
        sampler.quiver.set_fast(True)
        for b in batches_dev[:2]:
            sampler.sample(b)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fe = 0
        f0.record()
        for b in timed[0]:
            _, _, adjs = sampler.sample(b)
            fe += sum(a.edge_index.shape[1] for a in adjs)
        f1.record()
        barrier()
        fast = {"seps_sampler_only": fe / (f0.elapsed_time(f1) * 1e-3), "sample_ms_per_step": f0.elapsed_time(f1) / args.steps,
                "note": "qv_sampler_set_fast: O(k) per row, NOT the reference's random stream; not part of `value`"}
        sampler.quiver.set_fast(False)

    # ---- reduce over ranks -------------------------------------------------------------------------------------------
    stats = torch.tensor([total_ms, sample_ms, gather_ms, e2e_ms, kern_ms, serial_ms, e2e_fused_ms], dtype=torch.float64,
                         device=dev)
    sums = torch.tensor([edges_val, rows, e2e_edges, launches, edges, parity_rows, hop_bytes] +
                        ([tier_rows[k] for k in ("hot_local", "stripe_local", "peer", "host", "total")] if tier_rows else [0] * 5),
                        dtype=torch.float64, device=dev)
    mins = torch.tensor(rep_rates[:1] + rep_rates[-1:], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        dist.all_reduce(mins, op=dist.ReduceOp.SUM)
    total_ms, sample_ms, gather_ms, e2e_ms, kern_ms, serial_ms, e2e_fused_ms = stats.tolist()
    edges_val_all, rows_all, e2e_edges_all, launches_all, edges_all, parity_all, hop_bytes_all, t_hot, t_stripe, t_peer, \
        t_host, t_total = sums.tolist()
    if rank != 0:
        return None

    value = edges_val_all / (total_ms * 1e-3)
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(TRAFFIC_FILE))
        ent = tj.get(args.config)
        if ent and world == 1:
            traffic, traffic_src = ent["dram_bytes_per_launch"], ent["source"]
    except Exception:
        pass
    hot_frac_now = args.hot_frac if world > 1 else 0.0
    out = {
        "metric": "sampled_edges_per_s (k-hop sample + feature gather per step)",
        "value": value, "unit": "edges/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": cfg["title"], "config_key": args.config, "n_nodes": n, "n_edges": n_edges,
                   "feature_table_GB": n * row_bytes / 1e9, "placement": placement,
                   "sampler_mode": ("UVA (indices in pinned host memory)" if args.uva else "GPU (CSR replica in HBM)") +
                                   ", reference-exact XORWOW sampling (rand_seed 0)",
                   "pipelining": ("sampler on its own high-priority stream: sample(i+1) overlaps the feature gather of "
                                  "step i" if want_overlap else
                                  ("sample_and_gather (qv_khop_gather): the gather is enqueued behind the last hop with the "
                                   "frontier size read on the device; one stream, one host wait per step"
                                   if fused else "none: sampler and gather on one stream")),
                   "l2": f"inputs larger than L2 ({n_edges * 8 / 1e9:.1f} GB CSR + {n * row_bytes / 1e9:.1f} GB feature table vs "
                         "126 MB L2); fresh seeds every step and every repeat",
                   "torch_allocator": os.environ.get("PYTORCH_CUDA_ALLOC_CONF"),
                   "edges_per_step": edges_all / args.steps / world, "rows_per_step": rows_all / args.steps / world,
                   "setup_s": setup_s},
        "spread": {"repeats": n_rep, "edges_per_s_min": mins.tolist()[0], "edges_per_s_max": mins.tolist()[1],
                   "note": "each repeat = K steps on its own seed batches; `value` is the median repeat (max over ranks of "
                           "its time); min / max = sum over ranks of each rank's slowest / fastest repeat"},
        "parity_checked_rows": int(parity_all),
        "parity": "asserted in this run on every rank: gathered rows == closed formula of (original id, column) for 2 timed "
                  "batches; fused call == two calls (n_id, edge_index, rows)",
        "seps_sampler_only": edges_all / (sample_ms * 1e-3),
        "feature_gather_GBps": rows_all * row_bytes / (gather_ms * 1e-3) / 1e9,
        "feature_gather_GiBps": rows_all * row_bytes / (gather_ms * 1e-3) / 2**30,
        "feature_gather_kernel_GBps": rows_per_launch * world * row_bytes / (kern_ms * 1e-3) / 1e9,
        "sample_ms_per_step": sample_ms / args.steps, "gather_ms_per_step": gather_ms / args.steps,
        "serial_ms_per_step": serial_ms / args.steps, "serial_edges_per_s": edges_all / (serial_ms * 1e-3),
        "sampler_roofline": {"bound": "hbm (nominally; at 1024 seeds the hops are launch/latency bound)",
                             "algorithmic_bytes_per_step": hop_bytes_all / args.steps / world,
                             "formula": "sum over hops 40E+40S+8F",
                             "achieved": hop_bytes_all / world / (sample_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": hop_bytes_all / world / (sample_ms * 1e-3) / 1e9 / hbm_peak, "large_batch": big},
        "fast_mode": fast,
        "gpu_launches": int(launches_all),
        # e2e = the SAME call `value` is measured through (sample_and_gather), now with pinned HOST seeds copied in and a host
        # read of the result inside every step; the reference's two calls (sample, then feature[n_id]) are reported next to it
        "e2e": ({"value": e2e_edges_all / (e2e_fused_ms * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": batch * 8,
                 "d2h_bytes_per_step": d2h, "ms_per_step": e2e_fused_ms / args.steps,
                 "api": "sampler.sample_and_gather(host seeds, feature) + host read of the result -- the call `value` uses",
                 "two_call_value": e2e_edges_all / (e2e_ms * 1e-3), "two_call_ms_per_step": e2e_ms / args.steps,
                 "two_call_api": "sampler.sample(host seeds) then feature[n_id] -- the reference's two calls"}
                if e2e_fused_ms > 0 else
                {"value": e2e_edges_all / (e2e_ms * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": batch * 8,
                 "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps,
                 "api": "sampler.sample(host seeds) then feature[n_id] -- the reference's two calls"}),
        "clocks": clock_summary,
        "roofline": {"kernel": "feature gather (qv_gather.cu: gather_batch_flat_kernel / gather_batch_kernel; "
                               "gather_tma_kernel from 2 KiB rows)", "bound": "hbm",
                     "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src, "algorithmic_bytes_per_row": alg_bytes_per_row,
                     "rows_per_launch": rows_per_launch, "kernel_ms": kern_ms,
                     "how": "CUDA events around back-to-back launches of the timed batches' gathers (3 passes)"
                            + ("; at N>1 part of the rows arrive over NVLink, see `nvlink`" if world > 1 else "")},
    }
    if tier_rows:
        out["tier_rows_first_batch"] = {"hot_replica_local": t_hot / t_total, "stripe_local": t_stripe / t_total,
                                        "peer_nvlink": t_peer / t_total, "host_pcie": t_host / t_total,
                                        "note": "fractions of gathered rows by tier, summed over ranks"}
    if world > 1:
        remote_frac = t_peer / t_total if t_total else 1.0 - 1.0 / world
        nv = rows_per_launch * remote_frac * row_bytes / (kern_ms * 1e-3) / 1e9
        out["nvlink"] = {"achieved_GBps_per_gpu_ingress": nv, "peak": 770.0, "frac": nv / 770.0,
                         "peak_source": "measured peer-copy 770 GB/s per direction (B200_PROFILING.md)",
                         "remote_row_fraction": remote_frac, "hot_frac_replicated": hot_frac_now,
                         "how": "peer rows x row bytes / event-timed gather launch (all tiers in one kernel, so this is a "
                                "lower bound on the link rate while the kernel also copies local rows); counter-based "
                                "figures: profiles/"}
    if world == 1 and not args.no_cpu_baseline:
        indptr_cpu, indices_cpu = topo.indptr.cpu(), topo.indices.cpu()
        if not args.no_ref_gpu:
            try:
                out["ref_gpu_baseline"] = ref_gpu_baseline(cfg, dev, topo.indptr, topo.indices, timed[0], nid_keep)
            except Exception as e:  # the reference calls exit(1) on CUDA errors; anything catchable is reported
                out["ref_gpu_baseline"] = {"unavailable": f"{type(e).__name__}: {e}"}
        out["cpu_baseline"] = cpu_baseline_sample(cfg, indptr_cpu, indices_cpu, timed_host)
    if last_outputs is not None:
        dump_outputs(args.dump_outputs, last_outputs)
    return out


def main():
    sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree, which may be read-only
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("QV_BENCH_CONFIG", "ns"), choices=sorted(CONFIGS))
    ap.add_argument("--repeats", type=int, default=3, help="timed K-step regions (distinct batches); value = median")
    ap.add_argument("--hot-frac", type=float, default=None,
                    help="N>1: fraction of rows (hottest first) replicated on every GPU (default: 0.4; c3: 0; c4: 0.3; c5: 0)")
    ap.add_argument("--cold-frac", type=float, default=None,
                    help="fraction of rows (coldest) kept in pinned host memory (default 0; c4 at N>1: 0.5)")
    ap.add_argument("--order", default="auto", choices=["auto", "prob", "degree", "none"],
                    help="storage order of the feature rows: access probability (sample_prob), degree, or original ids")
    ap.add_argument("--device-build", action="store_true", help="build small tables in place on the device too")
    ap.add_argument("--feat-dim", type=int, default=None, help="override the config's feature width (experiments)")
    ap.add_argument("--gather-variant", type=int, default=0, help="qv_gather variant: 0 auto, 1 SIMT, 2 TMA bulk copies")
    ap.add_argument("--uva", action="store_true", help="sampler mode UVA: indices in pinned host memory")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--no-large-batch", action="store_true")
    ap.add_argument("--no-fuse", action="store_true",
                    help="`value` from sample() + feature[n_id] as two calls instead of sample_and_gather")
    ap.add_argument("--overlap", action="store_true",
                    help="run the sampler on its own high-priority stream so sample(i+1) overlaps gather(i)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed call returned in its last step as DIR/<name>.npy (float32 / float64, at "
                         "most 64 MB in all; a seeded sample of larger outputs), to compare two builds on the same inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    cfg = dict(CONFIGS[args.config])
    if args.feat_dim:
        cfg["feat_dim"] = args.feat_dim
        cfg["title"] += f" [feature width overridden: {args.feat_dim}]"
    if args.hot_frac is None:
        args.hot_frac = {"c3": 0.0, "c4": 0.3, "c5": 0.0}.get(args.config, 0.4)
    if args.cold_frac is None:
        args.cold_frac = 0.5 if args.config == "c4" else 0.0
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner with printf on
    # the first communicator), so file descriptor 1 is pointed at stderr for the whole run and the result line goes to a
    # private duplicate of the real stdout.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        res = run_reference(args, cfg, rank, world)
    else:
        if world < cfg["min_gpus"]:
            res = {"unavailable": f"config {args.config} needs {cfg['min_gpus']} GPUs (its table does not fit fewer)"} \
                if rank == 0 else None
        else:
            if world > 1:
                import torch.distributed as dist
                torch.cuda.set_device(local_rank)
                dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            res = run_ours(args, cfg, rank, world, local_rank)
            if world > 1:
                import torch.distributed as dist
                dist.destroy_process_group()
    if res is not None:
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(res) + "\n").encode())
    os.close(real_stdout)


if __name__ == "__main__":
    main()
