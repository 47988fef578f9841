"""L1 parity against the reference's OWN CUDA kernels EXECUTING on the same B200.

oracle/build_ref_cuda.py compiles the reference's unmodified CUDA extension (quiver_sample.cu, quiver_feature.cu,
cuda_random.cu.hpp, reindex.cu.hpp, shard_tensor.cu.hpp ...) for sm_100a into oracle/_ref/torch_quiver_ref_cuda*.so.
Here both extensions run on the same inputs and must agree bit for bit:
  * Quiver.sample_neighbor ids + counts over the (k, S) matrix of test_sample_neighbor_bit_exact, hub rows, many blocks
    (reference: srcs/cpp/src/quiver/cuda/quiver_sample.cu:113-200, CSRRowWiseSampleKernel cuda_random.cu.hpp:7-69);
  * Quiver.reindex_single (quiver_sample.cu:305-357);
  * the k-hop loop of sage_sampler.py:118-147 driven over the reference bindings vs our fused qv_khop;
  * ShardTensor.__getitem__ fp32 / fp16, GPU shard + pinned-host tier (quiver_feature.cu:246-302).
This closes the gap between "two readings of the same source" (the C oracle) and "two executions".
Without that build, the same tests compare with the reference's outputs stored in tests/golden/ref_cuda_kat.json
(tests/reference_outputs.py): written by `QV_RECORD_REF_GOLDEN=1 pytest tests/test_gpu_vs_reference_cuda.py` on a B200
where oracle/_ref holds the build.
"""
import os

import numpy as np
import pytest
import torch

from graphs import powerlaw_csr
from reference_outputs import ReferenceOutputs

pytestmark = pytest.mark.gpu
_KEEP = []


@pytest.fixture(scope="module")
def ref(golden_dir):
    from oracle import oracle
    r = ReferenceOutputs(os.path.join(golden_dir, "ref_cuda_kat.json"),
                         oracle.load_reference_cuda(),
                         "the reference's CUDA extension compiled unmodified for sm_100a (oracle/build_ref_cuda.py), "
                         "run on a B200")
    yield r
    r.save()


def _both(ref, indptr, indices):
    import torch_quiver as qv
    ip, ix = torch.from_numpy(indptr), torch.from_numpy(indices)
    ours = qv.device_quiver_from_csr_array(ip, ix, torch.zeros(1, dtype=torch.long), 0, True)
    theirs = ref.live.device_quiver_from_csr_array(ip, ix, torch.zeros(1, dtype=torch.long), 0, True) if ref.live else None
    return ours, theirs


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).cuda()


@pytest.fixture(scope="module")
def g2k(ref):
    indptr, indices = powerlaw_csr(2000, 30.0, seed=7)
    return (indptr, indices) + _both(ref, indptr, indices)


@pytest.mark.parametrize("k", [1, 2, 5, 25, 33, 64, 2000])
@pytest.mark.parametrize("S", [1, 63, 64, 65, 1000])
def test_sample_neighbor_equals_reference_kernel(ref, g2k, k, S):
    indptr, indices, ours, theirs = g2k
    seeds = _dev(np.random.default_rng(S * 131 + k).integers(0, 2000, S))
    out, cnt = ours.sample_neighbor(0, seeds, k)
    want = None
    if theirs is not None:
        r_out, r_cnt = theirs.sample_neighbor(0, seeds, k)
        want = {"counts": r_cnt, "out": r_out}
    torch.cuda.synchronize()
    ref.check(f"sample_neighbor/k={k},S={S}", {"counts": cnt, "out": out}, want)


def test_hubs_many_blocks_and_reindex(ref):
    indptr, indices = powerlaw_csr(60000, 40.0, seed=8, alpha=1.3)
    assert np.diff(indptr).max() > 3000
    ours, theirs = _both(ref, indptr, indices)
    hubs = np.argsort(-np.diff(indptr))[:300].copy()
    rest = np.random.default_rng(5).permutation(60000)[:20000]
    seeds = _dev(np.concatenate([hubs, rest[~np.isin(rest, hubs)]]))  # unique, hubs first: long chains + 300+ blocks
    for k in (5, 10, 25):
        out, cnt = ours.sample_neighbor(0, seeds, k)
        f, row, col = ours.reindex_single(seeds, out, cnt)
        want = None
        if theirs is not None:
            r_out, r_cnt = theirs.sample_neighbor(0, seeds, k)
            rf, rrow, rcol = theirs.reindex_single(seeds, r_out, r_cnt)
            want = {"counts": r_cnt, "out": r_out, "frontier": rf, "row_idx": rrow, "col_idx": rcol}
        torch.cuda.synchronize()
        ref.check(f"hubs/k={k}", {"counts": cnt, "out": out, "frontier": f, "row_idx": row, "col_idx": col}, want)


def test_khop_equals_reference_loop(ref):
    """sage_sampler.py:118-147 over the reference's bindings vs our one-call fused k-hop (and our per-hop calls)."""
    import quiver
    indptr, indices = powerlaw_csr(40000, 25.0, seed=11)
    _, theirs = _both(ref, indptr, indices)
    topo = quiver.CSRTopo(indptr=torch.from_numpy(indptr), indices=torch.from_numpy(indices))
    sizes = [15, 10, 5]
    sampler = quiver.pyg.GraphSageSampler(topo, sizes, device=0, mode="GPU")
    for batch in range(3):
        seeds = _dev(np.random.default_rng(100 + batch).permutation(40000)[:1024])
        want = None
        if theirs is not None:
            nodes, ref_adjs = seeds, []
            for size in sizes:
                out, cnt = theirs.sample_neighbor(0, nodes, size)
                frontier, row_idx, col_idx = theirs.reindex_single(nodes, out, cnt)
                ref_adjs.append((torch.stack([col_idx, row_idx]), (frontier.numel(), nodes.numel())))
                nodes = frontier
            torch.cuda.synchronize()
            want = {"n_id": nodes}
            for i, (r_ei, r_size) in enumerate(ref_adjs[::-1]):
                want[f"adj{i}_edge_index"], want[f"adj{i}_size"] = r_ei, np.array(r_size, np.int64)
        n_id, bs, adjs = sampler.sample(seeds)
        assert bs == 1024
        got = {"n_id": n_id}
        for i, adj in enumerate(adjs):
            got[f"adj{i}_edge_index"], got[f"adj{i}_size"] = adj.edge_index, np.array(adj.size.tolist(), np.int64)
        ref.check(f"khop/batch={batch}", got, want)


@pytest.mark.parametrize("dtype,d", [(torch.float32, 100), (torch.float32, 602), (torch.float16, 256), (torch.float32, 256)])
def test_gather_equals_reference_kernel(ref, dtype, d):
    import torch_quiver as qv
    n = 30000
    x = torch.from_numpy(np.random.default_rng(d).standard_normal((n, d)).astype(np.float32)).to(dtype)
    cold, cold_ref = x[20000:].clone(), x[20000:].clone()  # one pinned-host tier each (both libraries register theirs)
    idx = torch.from_numpy(np.random.default_rng(1).integers(0, n, 50000)).cuda()
    ours = qv.ShardTensor(0)
    ours.append(x[:20000], 0)  # HBM shard
    ours.append(cold, -1)      # pinned-host tier, aliased
    got = ours[idx]
    want = None
    if ref.live is not None:
        theirs = ref.live.ShardTensor(0)
        theirs.append(x[:20000], 0)
        theirs.append(cold_ref, -1)
        want = {"rows": theirs[idx]}
    torch.cuda.synchronize()
    ref.check(f"gather/{dtype},d={d}", {"rows": got}, want)  # 0 ULP: byte identity, same dtype and shape
    assert torch.equal(got.cpu(), x[idx.cpu()])
    if ref.live is None:
        return
    if dtype == torch.float32:
        theirs.unregister(cold_ref)  # the reference reads data_ptr<float>() here (quiver_feature.cu:354-360): fp32 only
    else:
        _KEEP.append(cold_ref)       # a registration must not outlive its memory: keep the half tensor for the process
