"""CPU suite, part 5: bench.py's host-side pieces -- the synthetic workload generators (run here on CPU tensors at toy
sizes), the closed-formula features every rank checks its gathered rows against, and the reference / cpu_baseline arm
(the reference's CPU classes from oracle/_ref when built, else the oracle port, and the line says which)."""
import json
import types

import numpy as np
import pytest
import torch

import bench


def test_configs_cover_baseline_json():
    import os
    base = json.load(open(os.path.join(bench.ROOT, "BASELINE.json")))
    assert len(base["configs"]) == 5
    assert set(bench.CONFIGS) == {"ns", "c1", "c2", "c3", "c4", "c5"}
    ns = bench.CONFIGS["ns"]  # the workload north_star states its target on
    assert ns["n_nodes"] == 100_000_000 and ns["feat_dim"] == 256 and round(ns["n_nodes"] * ns["mean_deg"]) == 1_000_000_000
    assert bench.CONFIGS["c1"]["feat_dim"] == 602 and bench.CONFIGS["c1"]["sizes"] == [25, 10]
    assert bench.CONFIGS["c2"]["feat_dim"] == 100 and bench.CONFIGS["c5"]["feat_dim"] == 768


@pytest.mark.parametrize("by_degree", [True, False])
def test_pareto_graph_is_a_valid_sorted_csr(by_degree):
    n = 30000
    indptr, indices = bench.make_graph_pareto("cpu", n, 10.0, by_degree, seed=3, chunk_edges=1 << 15)  # many chunks
    assert indptr.shape == (n + 1, ) and indptr[0] == 0 and indices.numel() == int(indptr[-1])
    assert int(indices.min()) >= 0 and int(indices.max()) < n
    deg = indptr[1:] - indptr[:-1]
    row = torch.repeat_interleave(torch.arange(n), deg)
    key = row * n + indices
    assert bool((key[1:] >= key[:-1]).all())  # rows in order, columns sorted inside each row
    indeg = torch.bincount(indices, minlength=n).float()
    corr = torch.corrcoef(torch.stack([deg.float(), indeg]))[0, 1].item()
    assert (corr > 0.8) if by_degree else (abs(corr) < 0.2)  # neighbours drawn in proportion to degree, or uniformly
    again = bench.make_graph_pareto("cpu", n, 10.0, by_degree, seed=3, chunk_edges=1 << 15)
    assert torch.equal(again[0], indptr) and torch.equal(again[1], indices)  # every rank builds the same graph


def test_rmat_graph():
    indptr, indices = bench.make_graph_rmat("cpu", 5000, 60000)
    assert indices.numel() == 60000 == int(indptr[-1]) and indptr.shape == (5001, )
    assert int(indices.max()) < 5000 and bool((indptr[1:] >= indptr[:-1]).all())
    deg = indptr[1:] - indptr[:-1]
    assert int(deg.max()) > 20 * float(deg.float().mean())  # heavy skew


def test_seed_batches_are_unique_and_reproducible():
    a = bench.make_seed_batches(3, 100000, 1024, seed=5)
    b = bench.make_seed_batches(3, 100000, 1024, seed=5)
    for x, y in zip(a, b):
        assert x.numel() == 1024 and x.unique().numel() == 1024 and torch.equal(x, y)
    legacy = bench.make_seed_batches(2, 5000, 256, seed=1, legacy=True)
    assert all(x.unique().numel() == 256 for x in legacy)


def test_feature_formula_is_exact_and_position_independent():
    ids = torch.tensor([0, 1, 12345678, 99_999_999, 244_160_498])
    x = bench.feat_formula(ids, 7, "cpu")
    want = ((ids.numpy()[:, None].astype(np.int64) * 1000003 + np.arange(7)[None, :] * 7919) & 0xFFFFF) / 1048576.0
    assert x.dtype == torch.float32 and np.array_equal(x.numpy().astype(np.float64), want)  # exact in fp32
    assert torch.equal(bench.feat_formula(ids[[3, 0]], 7, "cpu"), x[[3, 0]])


def _tiny():
    cfg = dict(title="tiny", n_nodes=20000, mean_deg=8.0, graph="pareto_degree", feat_dim=16, sizes=[5, 3], batch=128,
               legacy=False, min_gpus=1)
    args = types.SimpleNamespace(steps=2, warmup=1, gpus=1, config="tiny")
    return cfg, args


def test_reference_arm_line_and_cpu_baseline():
    cfg, args = _tiny()
    bench.CONFIGS["tiny"] = cfg
    try:
        line = bench.run_reference(args, cfg, 0, 1)
        assert bench.run_reference(args, cfg, 1, 2) is None  # under torchrun only rank 0 runs the CPU arm
    finally:
        del bench.CONFIGS["tiny"]
    json.dumps(line)
    assert line["impl"] == "reference" and line["unit"] == "edges/s" and line["higher_is_better"] is True
    assert line["reference_procs"] == 1 and line["gpu_launches"] == 0
    assert line["e2e"]["value"] == line["value"] == line["cpu_baseline"]["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["workload"] == "tiny"
    kind = line["cpu_baseline"]["kind"]
    assert kind in ("reference", "port")
    # a line measured on OUR port (oracle/_ref missing) must say so at the top level; the reference's own code must not
    assert ("reference_unavailable" in line) == (kind == "port")
    indptr, indices = bench.make_graph("cpu", cfg)
    base = bench.cpu_baseline_sample(cfg, indptr, indices, bench.make_seed_batches(4, cfg["n_nodes"], cfg["batch"]), n_b=2)
    assert base["kind"] in ("reference", "port") and base["value"] > 0 and base["cores"] >= 1 and "batches" in base["sample"]


def test_host_table_folds_large_tables():
    x, rows = bench.host_table(1000, 8, cap_bytes=100 * 32)
    assert rows == 100 and x.shape == (100, 8)
    x, rows = bench.host_table(50, 8)
    assert rows == 50


def test_dump_outputs_fit_the_budget_and_repeat(tmp_path):
    rng = np.random.default_rng(0)
    arrays = {"n_id": np.arange(1000, dtype=np.float64), "adj0_edge_index": rng.integers(0, 1000, (2, 30000)).astype(np.float64),
              "x": rng.random((20000, 16), dtype=np.float32)}
    budget = 600_000
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, budget=budget)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["adj0_edge_index.npy", "adj0_edge_index_index.npy", "n_id.npy", "x.npy", "x_index.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= budget + 5 * 128  # + the .npy headers
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)  # same arguments, same files
    load = lambda f: np.load(tmp_path / "a" / f)  # noqa: E731
    assert np.array_equal(load("n_id.npy"), arrays["n_id"])  # within its share: whole
    pick = load("x_index.npy").astype(np.int64)
    assert np.array_equal(load("x.npy"), arrays["x"][pick]) and len(np.unique(pick)) == len(pick)
    pick = load("adj0_edge_index_index.npy").astype(np.int64)
    assert np.array_equal(load("adj0_edge_index.npy"), arrays["adj0_edge_index"][:, pick])
