"""GPU: building an index twice from the same input gives the same index, and searching it gives the same answers.

The builds sum k-means centroids and PQ codebook entries, rank rows inside IVF lists and collect CAGRA reverse edges in input
order, never in the order atomics happen to run, so two builds compare equal bit for bit; a benchmark run can then be
compared output for output with the next one."""
import numpy as np
import pytest
import torch

from tests.util import clustered

pytestmark = pytest.mark.gpu


def _data(n, d, nq):
    ds, centers = clustered(n, d, seed=11, n_centers=200)
    qs, _ = clustered(nq, d, seed=12, centers=centers)
    return torch.from_numpy(ds).cuda(), torch.from_numpy(qs).cuda()


def _lists(index):
    return [index.list_indices(l).cpu() for l in range(index.n_lists)]


def _same(a, b):
    return bool(torch.equal(a.cpu(), b.cpu()))


def _build_twice(build, search):
    out = []
    for _ in range(2):
        index = build()
        first = [t.clone() for t in search(index)]
        again = search(index)
        assert all(_same(x, y) for x, y in zip(first, again)), "a second search of the same index answered differently"
        out.append((index, first))
    return out


@pytest.mark.parametrize("codebook", ["subspace", "cluster"])
def test_ivf_pq_build_is_deterministic(codebook):
    from cuvs_b200.neighbors import ivf_pq
    ds, qs = _data(200_000, 64, 2_000)
    params = ivf_pq.IndexParams(n_lists=256, pq_dim=32, kmeans_n_iters=10, codebook_kind=codebook)
    sp = ivf_pq.SearchParams(n_probes=32, lut_dtype=np.float16)
    (a, ra), (b, rb) = _build_twice(lambda: ivf_pq.build(params, ds), lambda i: ivf_pq.search(sp, i, qs, 10))
    assert _same(a.centers, b.centers)
    assert _same(a.pq_centers, b.pq_centers)
    assert all(_same(x, y) for x, y in zip(_lists(a), _lists(b)))
    assert all(_same(x, y) for x, y in zip(ra, rb))


def test_ivf_flat_build_is_deterministic():
    from cuvs_b200.neighbors import ivf_flat
    ds, qs = _data(200_000, 64, 2_000)
    params = ivf_flat.IndexParams(n_lists=256, kmeans_n_iters=10)
    sp = ivf_flat.SearchParams(n_probes=16)
    (a, ra), (b, rb) = _build_twice(lambda: ivf_flat.build(params, ds), lambda i: ivf_flat.search(sp, i, qs, 10))
    assert _same(a.centers, b.centers)
    assert all(_same(x, y) for x, y in zip(_lists(a), _lists(b)))
    assert all(_same(x, y) for x, y in zip(ra, rb))


def test_cagra_build_is_deterministic():
    from cuvs_b200.neighbors import cagra
    ds, qs = _data(50_000, 32, 2_000)
    params = cagra.IndexParams(graph_degree=32)
    sp = cagra.SearchParams(itopk_size=64)
    (a, ra), (b, rb) = _build_twice(lambda: cagra.build(params, ds), lambda i: cagra.search(sp, i, qs, 10))
    assert _same(a.graph, b.graph)
    assert all(_same(x, y) for x, y in zip(ra, rb))
