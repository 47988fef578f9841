"""CPU suite, part 1: pin the oracle (oracle/qv_oracle.c) against the reference's own artefacts.

  * XORWOW restatement  == NVIDIA curand_kernel.h run on the host            (tests/golden/xorwow_kat.json)
  * counts / verbatim rows / reindex == the reference CPU extension           (tests/golden/ref_cpu_kat.json)
  * structural validity == the reference's only sampler assertion             (tests/cpp/test_quiver_cpu.cpp:32-75)
When oracle/_ref/ holds the live builds, the same checks also run against them directly; without them,
test_live_reference_cpu_extension checks the outputs of that build stored in tests/golden/ref_cpu_ext_kat.json.
"""
import json
import os

import numpy as np
import pytest

from graphs import MINI, powerlaw_csr, simple_graph
from reference_outputs import ReferenceOutputs


def _golden_graph(name, meta):
    if name == "mini":
        return np.array(MINI["indptr"]), np.array(MINI["indices"])
    if name == "powerlaw_300":
        return powerlaw_csr(**meta["powerlaw_300"])
    return simple_graph(**meta["simple_100_10"])


def test_xorwow_matches_curand_golden(oracle, golden_dir):
    kat = json.load(open(os.path.join(golden_dir, "xorwow_kat.json")))
    assert len(kat["cases"]) >= 10
    for c in kat["cases"]:
        state, draws = oracle.xorwow_stream(c["seed"], c["subseq"], len(c["draws"]))
        assert state == c["state"], c
        assert draws == c["draws"], c


def test_xorwow_matches_live_curand_probe(oracle):
    rng = np.random.default_rng(5)
    pairs = [(int(rng.integers(0, 2**40)), int(rng.integers(0, 128))) for _ in range(12)]
    live = oracle.curand_probe(8, pairs)
    if live is None:
        pytest.skip("oracle/_ref/curand_probe not built on this machine")
    for c in live:
        state, draws = oracle.xorwow_stream(c["seed"], c["subseq"], 8)
        assert (state, draws) == (c["state"], c["draws"])


def test_xorwow_subsequence_matrix_is_consistent(oracle):
    # P_q applied to a seed state must equal curand_init(seed, q, 0): this is the table the product caches
    for q in (1, 2, 31, 127):
        m = oracle.xorwow_seq_matrix(q)
        base, _ = oracle.xorwow_stream(77, 0, 0)
        want, _ = oracle.xorwow_stream(77, q, 0)
        v = np.zeros(5, np.uint32)
        for w in range(5):
            for j in range(32):
                if (base[1 + w] >> j) & 1:
                    v ^= m[w * 32 + j]
        assert [base[0]] + v.tolist() == want


def test_reference_cpu_golden(oracle, golden_dir):
    kat = json.load(open(os.path.join(golden_dir, "ref_cpu_kat.json")))
    assert len(kat["cases"]) >= 12
    for c in kat["cases"]:
        indptr, indices = _golden_graph(c["graph"], kat["graphs"])
        seeds = np.array(c["seeds"])
        counts, out_ptr, tot = oracle.sample_counts(indptr, seeds, c["k"])
        assert counts.tolist() == c["counts"]
        assert tot == len(c["draw"])
        # the reference's own (unseeded) draw is structurally valid, and rows with deg <= k are verbatim CSR rows
        assert oracle.validate_sample(indptr, indices, seeds, c["k"], np.array(c["counts"]), np.array(c["draw"])) == 0
        ours, _ = oracle.sample_neighbor(indptr, indices, seeds, c["k"])
        assert oracle.validate_sample(indptr, indices, seeds, c["k"], counts, ours) == 0
        deg = indptr[seeds + 1] - indptr[seeds]
        for i in np.nonzero(deg <= c["k"])[0]:
            a, b = out_ptr[i], out_ptr[i] + counts[i]
            assert ours[a:b].tolist() == c["draw"][a:b] == indices[indptr[seeds[i]]:indptr[seeds[i] + 1]].tolist()
        # reindex is deterministic: identical to the reference given the reference's draw
        frontier, row, col = oracle.reindex(seeds, np.array(c["draw"], dtype=np.int64), np.array(c["counts"]))
        assert frontier.tolist() == c["frontier"]
        assert row.tolist() == c["row_idx"]
        assert col.tolist() == c["col_idx"]


def test_mini_known_answer(oracle):
    m = MINI
    counts, _, _ = oracle.sample_counts(np.array(m["indptr"]), np.array(m["seeds"]), m["k"])
    assert counts.tolist() == m["counts"]
    frontier, row, col = oracle.reindex(np.array(m["seeds"]), np.array(m["draw"]), np.array(m["counts"]))
    assert (frontier.tolist(), row.tolist(), col.tolist()) == (m["frontier"], m["row_idx"], m["col_idx"])


@pytest.mark.parametrize("n,nbr,k", [(10, 5, 10), (100, 10, 5), (1000, 10, 10)])  # test_quiver_cpu.cpp:70-75
def test_reference_structural_cases(oracle, n, nbr, k):
    indptr, indices = simple_graph(n, nbr)
    seeds = np.arange(n)
    out, counts = oracle.sample_neighbor(indptr, indices, seeds, k)
    assert counts.tolist() == [min(nbr, k)] * n
    assert oracle.validate_sample(indptr, indices, seeds, k, counts, out) == 0
    # the validator really rejects: duplicate a position
    if k < nbr:
        bad = out.copy()
        bad[1] = bad[0]
        assert oracle.validate_sample(indptr, indices, seeds, k, counts, bad) != 0


def test_sampler_is_uniform(oracle):
    # chi-square over which positions of a degree-40 row get picked (k = 8), across generator seeds
    indptr = np.array([0, 40], dtype=np.int64)
    indices = np.arange(100, 140, dtype=np.int64)
    hits = np.zeros(40)
    trials = 1500
    for s in range(trials):
        out, _ = oracle.sample_neighbor(indptr, indices, np.array([0]), 8, rand_seed=s + 1)
        assert len(set(out.tolist())) == 8
        hits[out - 100] += 1
    expect = trials * 8 / 40
    chi2 = ((hits - expect) ** 2 / expect).sum()
    assert chi2 < 80.0  # 39 dof: p(chi2 > 80) ~ 1e-4


def test_live_reference_cpu_extension(oracle, golden_dir):
    live = oracle.load_reference()
    ref = ReferenceOutputs(os.path.join(golden_dir, "ref_cpu_ext_kat.json"), live,
                           "the reference's CPU extension compiled unmodified (oracle/build_ref.py)", deterministic=False)
    import torch
    indptr, indices = powerlaw_csr(2000, 20.0, seed=9)
    cq = live.cpu_quiver_from_csr_array(torch.from_numpy(indptr), torch.from_numpy(indices)) if live else None
    seeds = np.random.default_rng(1).permutation(2000)[:256]
    for k in (3, 10, 2000):
        reindexed = None
        if live is not None:
            out, cnt = cq.sample_neighbor(torch.from_numpy(seeds), k)
            f, r, c = cq.reindex_single(torch.from_numpy(seeds), out, cnt)
            reindexed = {"frontier": f, "row_idx": r, "col_idx": c}
        drawn = ref.arrays(f"k={k}", {"out": out, "cnt": cnt} if live is not None else None)
        out, cnt = drawn["out"], drawn["cnt"]
        counts, _, tot = oracle.sample_counts(indptr, seeds, k)
        assert cnt.tolist() == counts.tolist() and out.size == tot
        assert oracle.validate_sample(indptr, indices, seeds, k, counts, out) == 0
        of, orow, ocol = oracle.reindex(seeds, out, counts)
        ref.check(f"k={k}/reindex_single", {"frontier": of, "row_idx": orow, "col_idx": ocol}, reindexed)
    ref.save()


def test_gather_oracle_is_tensor_indexing(oracle):
    rng = np.random.default_rng(2)
    x = rng.integers(0, 10, (500, 37)).astype(np.float32)  # integer-valued floats as in test_features.py:310-313
    idx = rng.integers(0, 500, 300)
    shards = [x[:120], x[120:121], x[121:]]
    assert np.array_equal(oracle.gather(shards, idx), x[idx])
    order = rng.permutation(500)
    assert np.array_equal(oracle.gather(shards, idx, feature_order=order), x[order[idx]])
    bad = np.array([0, -1, 500, 499, 10**12])
    got = oracle.gather(shards, bad)
    assert np.array_equal(got[[0, 3]], x[[0, 499]]) and not got[[1, 2, 4]].any()


def test_cal_next_oracle_formula(oracle):
    indptr, indices = powerlaw_csr(200, 6.0, seed=4)
    p = np.random.default_rng(0).random(200).astype(np.float32)
    cur = oracle.cal_next(p, 3, indptr, indices)
    deg = np.diff(indptr)
    for v in (0, 17, 199):
        if deg[v] == 0:
            assert cur[v] == 0
            continue
        acc = 1.0
        for u in indices[indptr[v]:indptr[v + 1]]:
            if deg[u] == 0:
                continue
            acc *= (1 - p[u]) if deg[u] <= 3 else (1 - p[u] + p[u] * (deg[u] - 3) / deg[u])
        assert abs(cur[v] - (1 - (1 - p[v]) * acc)) < 1e-5


def test_gpu_path_golden_khop(oracle, golden_dir):
    """The frozen k-hop vectors (tests/golden/gpu_path_kat.json): the oracle must keep producing exactly these ids."""
    import json
    from graphs import powerlaw_csr
    kat = json.load(open(os.path.join(golden_dir, "gpu_path_kat.json")))
    assert len(kat["cases"]) >= 3
    for c in kat["cases"]:
        g = c["graph"]
        indptr, indices = powerlaw_csr(g["n_nodes"], g["mean_deg"], seed=g["seed"])
        n_id, bs, adjs = oracle.khop(indptr, indices, np.array(c["seeds"], np.int64), c["sizes"])
        assert n_id.tolist() == c["n_id"] and bs == len(c["seeds"])
        for (ei, size), want in zip(adjs, c["adjs"]):
            assert ei.tolist() == want["edge_index"] and list(map(int, size)) == want["size"]


@pytest.mark.parametrize("mega_draws,seg", [(0, 1), (2, 3), (8, 4), (64, 256)])
def test_chain_splitting_equals_the_sequential_walk(oracle, mega_draws, seg):
    """Executable statement of the product's mega-row scheme (qo_sample_neighbor_gpu_split): cutting a lane's generator
    chain into segments positioned by offset skip-ahead, evaluated in reverse order and merged by max, gives exactly the
    sequential reservoir walk -- for every threshold / segment length, several long rows per warp, rows at the end of a
    warp's list, k = 1 .. 32."""
    rng = np.random.default_rng(7)
    n = 3000
    deg = rng.integers(0, 40, n)
    deg[rng.permutation(n)[:25]] = rng.integers(2000, 9000, 25)
    indptr = np.zeros(n + 1, np.int64)
    np.cumsum(deg, out=indptr[1:])
    indices = rng.integers(0, n, int(indptr[-1])).astype(np.int64)
    heavy = np.flatnonzero(deg >= 2000)
    seeds = np.concatenate([heavy[:12], rng.permutation(n)[:150], heavy[12:]]).astype(np.int64)
    for k in (1, 5, 15, 32):
        want, want_cnt = oracle.sample_neighbor(indptr, indices, seeds, k)
        got, got_cnt = oracle.sample_neighbor_split(indptr, indices, seeds, k, mega_draws, seg)
        assert np.array_equal(got_cnt, want_cnt) and np.array_equal(got, want), (k, mega_draws, seg)
