"""GPU: inserting the same rows by different routes gives the same index.

A build from a device tensor, a build from a host tensor, and an empty build followed by extend() from the device and then
from the host label every row the same way and place it in input order inside its list, so the saved index files are
byte-identical and the searches answer the same.  The large cases hold more rows than one 512 MiB insertion chunk, so both
passes over the chunks cross a chunk boundary, and the split point of the extend route is not on one."""
import hashlib

import pytest
import torch

from tests.util import clustered

pytestmark = pytest.mark.gpu


def _digest(mod, index, path):
    mod.save(path, index)
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for block in iter(lambda: f.read(1 << 24), b""):
            h.update(block)
    path.unlink()
    return h.hexdigest()


def _check_routes(mod, make_params, sp, n, d, a, tmp_path):
    ds, centers = clustered(n, d, seed=21, n_centers=500)
    qs, _ = clustered(1000, d, seed=22, centers=centers)
    host, qs = torch.from_numpy(ds), torch.from_numpy(qs).cuda()
    dev = host.cuda()
    routes = {
        "device": lambda: mod.build(make_params(True), dev),
        "host": lambda: mod.build(make_params(True), host),
        "extend": lambda: mod.extend(mod.extend(mod.build(make_params(False), dev), dev[:a], None), host[a:], None),
    }
    out = {}
    for name, build in routes.items():
        index = build()
        assert len(index) == n
        dist, nbr = mod.search(sp, index, qs, 10)
        out[name] = (_digest(mod, index, tmp_path / f"{name}.bin"), dist.cpu(), nbr.cpu())
        del index
    ref = out["device"]
    for name in ("host", "extend"):
        assert out[name][0] == ref[0], f"{name}: the saved index differs from the device build"
        assert torch.equal(out[name][1], ref[1]) and torch.equal(out[name][2], ref[2]), f"{name}: search answers differ"


@pytest.mark.parametrize("metric,n,d,a", [("sqeuclidean", 1_100_000, 128, 40_001), ("inner_product", 200_000, 64, 70_001),
                                          ("cosine", 200_000, 64, 70_001)])
def test_ivf_flat_insert_routes_agree(metric, n, d, a, tmp_path):
    from cuvs_b200.neighbors import ivf_flat

    def params(add):
        return ivf_flat.IndexParams(n_lists=256, metric=metric, kmeans_n_iters=10, add_data_on_build=add)
    _check_routes(ivf_flat, params, ivf_flat.SearchParams(n_probes=16), n, d, a, tmp_path)


@pytest.mark.parametrize("codebook,n,d,a", [("subspace", 1_100_000, 128, 40_001), ("cluster", 200_000, 64, 70_001)])
def test_ivf_pq_insert_routes_agree(codebook, n, d, a, tmp_path):
    from cuvs_b200.neighbors import ivf_pq

    def params(add):
        return ivf_pq.IndexParams(n_lists=256, pq_dim=d // 2, kmeans_n_iters=10, codebook_kind=codebook, add_data_on_build=add)
    _check_routes(ivf_pq, params, ivf_pq.SearchParams(n_probes=32), n, d, a, tmp_path)
