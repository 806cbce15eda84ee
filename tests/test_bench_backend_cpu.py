"""BASELINE configs[0] — "kNN via cuvs_bench, 10k x 128 f32, k=10 (CPU path, plumbing, no GPU)" — and the plugin surface of
cuvs_b200/bench_backend.py against the reference's benchmark package (python/cuvs_bench/cuvs_bench/backends/base.py).

The reference's C0 algorithm is hnswlib, a third-party library that is not in this image; the plumbing under test is the
harness (dataset -> build -> batched search -> recall -> Google-Benchmark-style JSON records), so it is driven here with a
test-only CPU backend whose searcher is the oracle's exact kNN (test infrastructure; the product backend serves GPU algorithms
only and never imports the oracle)."""
import importlib
import inspect
import itertools
import json
import os
import sys

import numpy as np
import pytest

import oracle
from cuvs_b200 import bench_backend as bb
from oracle.make_golden_cuvs_bench import BUILD_RESULT, SEARCH_RESULT, recall_inputs

REF_PKG = "/root/reference/python/cuvs_bench"


class OracleExactBackend(bb.HarnessMixin, bb.BenchmarkBackend):
    """CPU stand-in for the reference's hnswlib wrapper: build = keep the vectors, search = exact fp32 kNN (oracle)."""

    def _build_one(self, algo, metric, vectors, build_param):
        return (np.ascontiguousarray(vectors, dtype=np.float32), metric)

    def _search_batch(self, handle, algo, queries, k, search_param, dataset):
        ds, metric = handle
        return oracle.knn(ds, np.ascontiguousarray(queries, dtype=np.float32), k, metric)


def _dataset(n=10_000, d=128, nq=500, k=10, seed=7):
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((n, d)).astype(np.float32)
    queries = rng.standard_normal((nq, d)).astype(np.float32)
    # ground truth by an independent float64 computation (not the oracle)
    d2 = (queries.astype(np.float64) ** 2).sum(1)[:, None] - 2.0 * queries.astype(np.float64) @ base.astype(np.float64).T \
        + (base.astype(np.float64) ** 2).sum(1)[None, :]
    gt = np.argsort(d2, axis=1, kind="stable")[:, :k]
    return bb.Dataset(name="synthetic-128-euclidean", training_vectors=base, query_vectors=queries, groundtruth_neighbors=gt,
                      distance_metric="euclidean")


def _c0_dataset_with_the_reference_ground_truth():
    """10k x 128 f32, k = 10, with the ground truth the REFERENCE's CPU path computed (cuvs_bench generate_groundtruth
    calc_truth, run by oracle/make_golden_cuvs_bench.py; tests/golden/cuvs_bench_cpu_groundtruth.json, case c0_10k_x_128_l2)."""
    case = [c for c in json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                                                   "cuvs_bench_cpu_groundtruth.json")))["cases"] if c["name"] == "c0_10k_x_128_l2"][0]
    rng = np.random.default_rng(case["seed"])
    base = rng.standard_normal((case["n"], case["d"]), dtype=np.float32)
    queries = rng.standard_normal((case["nq"], case["d"]), dtype=np.float32)
    return bb.Dataset(name="c0-10k-128-euclidean", training_vectors=base, query_vectors=queries,
                      groundtruth_neighbors=np.array(case["ids"]), distance_metric="euclidean")


def _reference_interface():
    """What the reference's benchmark package defines and computes, recorded by oracle/make_golden_cuvs_bench.py."""
    return json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cuvs_bench_interface.json")))


def test_c0_harness_recall_against_the_reference_cpu_ground_truth():
    ds = _c0_dataset_with_the_reference_ground_truth()
    recs = bb.run_config({"name": "cpu_exact", "groups": {"base": {"build": {}, "search": {}}}}, ds, k=10, batch_size=50,
                         mode="throughput", backend=OracleExactBackend({"name": "cpu_exact"}))
    assert recs[1]["Recall"] >= 0.999 and recs[1]["n_queries"] == 100


def test_c0_plumbing_10k_x_128_k10_on_cpu():
    ds = _dataset()
    cfg = {"name": "cpu_exact", "groups": {"base": {"build": {}, "search": {}}}}
    for mode in ("throughput", "latency"):
        recs = bb.run_config(cfg, ds, k=10, batch_size=200, mode=mode, backend=OracleExactBackend({"name": "cpu_exact"}))
        json.dumps(recs)  # records are plain JSON
        build, search = recs[0], recs[1]
        assert build["name"] == "cpu_exact/build" and build["time_unit"] == "s" and build["success"]
        assert search["name"] == "cpu_exact/search" and search["time_unit"] == "ms"
        assert search["Recall"] >= 0.999 and search["items_per_second"] > 0 and search["n_queries"] == 500
        assert ("p99" in search) == (mode == "latency")


def test_search_space_expansion_follows_the_reference_yaml_layout():
    group = _reference_interface()["cuvs_ivf_pq_test_group"]  # the `test` group of the reference's cuvs_ivf_pq.yaml
    seen = []

    class Recorder(OracleExactBackend):
        def _build_one(self, algo, metric, vectors, build_param):
            seen.append(("build", build_param))
            return super()._build_one(algo, metric, vectors, build_param)

        def _search_batch(self, handle, algo, queries, k, search_param, dataset):
            seen.append(("search", tuple(sorted(search_param.items()))))
            return super()._search_batch(handle, algo, queries, k, search_param, dataset)

    recs = bb.run_config({"name": "cuvs_ivf_pq", "groups": {"test": group}}, _dataset(n=2000, nq=40), k=10, batch_size=40,
                         backend=Recorder({"name": "x"}))
    builds = [s for s in seen if s[0] == "build"]
    assert builds == [("build", {"nlist": 1024, "pq_dim": 16, "pq_bits": 6, "ratio": 1, "niter": 20})]
    assert {dict(s[1])["nprobe"] for s in seen if s[0] == "search"} == {1, 5}
    assert [r["name"] for r in recs] == ["cuvs_ivf_pq/build", "cuvs_ivf_pq/search", "cuvs_ivf_pq/search"]
    assert recs[1]["search_params"][0]["smemLutDtype"] == "half"


def test_recall_definition():
    found = np.array([[1, 2, 3], [4, 5, 6]])
    truth = np.array([[3, 2, 9, 1], [7, 8, 4, 5]])
    assert bb.recall_at_k(found, truth, 3) == pytest.approx(3 / 6)


def test_plugin_is_a_backend_of_the_reference_package():
    """The plugin implements every abstract method of the reference's BenchmarkBackend (python/cuvs_bench/cuvs_bench/backends/
    base.py) with the reference's parameters, and its result records are the reference's BuildResult / SearchResult JSON
    records on the same values."""
    gold = _reference_interface()
    assert not getattr(bb.CuvsB200Backend, "__abstractmethods__", frozenset())
    for name, params in gold["abstract_methods"].items():
        attr = inspect.getattr_static(bb.CuvsB200Backend, name)
        assert not getattr(attr, "__isabstractmethod__", False), name
        if params is None:
            assert isinstance(attr, property), name
        else:
            assert list(inspect.signature(attr).parameters) == params, name
    assert bb.BuildResult(**BUILD_RESULT).to_json() == gold["build_result_json"]
    assert bb.SearchResult(**SEARCH_RESULT).to_json() == gold["search_result_json"]


def test_c0_through_the_reference_orchestrator(tmp_path):
    """BASELINE configs[0] end to end through the REFERENCE's own benchmark code: cuvs_bench's BenchmarkOrchestrator
    (orchestrator/orchestrator.py:27-290) loads a dataset YAML + an algorithm YAML, expands the parameter grid with its own
    ConfigLoader base class, reads the .fbin / .ibin files with its own loader and drives a backend registered through its
    registry — here the plugin's harness with the test-only CPU searcher, on 10k x 128 f32, k = 10, with the ground truth the
    reference's CPU path computed.  Skipped where the reference checkout is absent."""
    if not os.path.isdir(REF_PKG):
        pytest.skip("no reference checkout on this box")
    yaml = pytest.importorskip("yaml")
    case = [c for c in json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                                                   "cuvs_bench_cpu_groundtruth.json")))["cases"] if c["name"] == "c0_10k_x_128_l2"][0]
    rng = np.random.default_rng(case["seed"])
    base = rng.standard_normal((case["n"], case["d"]), dtype=np.float32)
    queries = rng.standard_normal((case["nq"], case["d"]), dtype=np.float32)

    def write_bin(path, a):  # cuvs-bench binary format, legacy header (cuvs_bench/_bin_format.py): uint32 rows, uint32 cols, data
        with open(path, "wb") as f:
            np.array(a.shape, dtype=np.uint32).tofile(f)
            np.ascontiguousarray(a).tofile(f)

    ddir = tmp_path / "c0"
    ddir.mkdir()
    write_bin(ddir / "base.fbin", base)
    write_bin(ddir / "query.fbin", queries)
    write_bin(ddir / "groundtruth.neighbors.ibin", np.array(case["ids"], dtype=np.int32))
    ds_yaml = tmp_path / "datasets.yaml"
    ds_yaml.write_text(yaml.safe_dump([{"name": "c0", "base_file": "c0/base.fbin", "query_file": "c0/query.fbin",
                                        "groundtruth_neighbors_file": "c0/groundtruth.neighbors.ibin", "dims": case["d"],
                                        "distance": "euclidean"}]))
    adir = tmp_path / "algos"
    adir.mkdir()
    (adir / "cpu_exact.yaml").write_text(yaml.safe_dump({"name": "cpu_exact", "groups": {"base": {"build": {"dummy": [1]}, "search": {"ef": [10, 20]}}}}))

    sys.path.insert(0, REF_PKG)
    try:
        try:
            importlib.import_module("cuvs_bench.orchestrator")
        except Exception as e:  # noqa: BLE001
            pytest.skip(f"reference cuvs_bench.orchestrator not importable here: {e}")
        mod = importlib.reload(bb)
        try:
            if not mod.HAVE_CUVS_BENCH:
                pytest.skip("reference cuvs_bench.backends not importable here")
            from cuvs_bench.backends.registry import get_registry, register_config_loader
            from cuvs_bench.orchestrator import BenchmarkOrchestrator

            class CpuExact(mod.HarnessMixin, mod.BenchmarkBackend):
                def _build_one(self, algo, metric, vectors, build_param):
                    return (np.ascontiguousarray(vectors, dtype=np.float32), metric)

                def _search_batch(self, handle, algo, q, k, search_param, dataset):
                    return oracle.knn(handle[0], np.ascontiguousarray(q, dtype=np.float32), k, handle[1])

            try:
                get_registry().register("cpu_exact_test", CpuExact)
            except ValueError:
                pass
            register_config_loader("cpu_exact_test", mod.make_config_loader("cpu_exact", "cpu_exact_test"))
            results = BenchmarkOrchestrator(backend_type="cpu_exact_test").run_benchmark(
                mode="sweep", dataset="c0", dataset_path=str(tmp_path), dataset_configuration=str(ds_yaml),
                algorithm_configuration=str(adir), algorithms="cpu_exact", count=10, batch_size=50, search_mode="throughput")
            assert len(results) == 2 and results[0].success and results[1].success
            build, search = results
            assert build.to_json()["name"] == "cpu_exact/build"
            assert search.recall >= 0.999 and search.neighbors.shape == (case["nq"], 10)
            assert len(search.metadata["all_results"]) == 2  # two search-parameter combinations of the YAML grid
            assert search.to_json()["items_per_second"] > 0
        finally:
            for name in [m for m in sys.modules if m == "cuvs_bench" or m.startswith("cuvs_bench.")]:
                del sys.modules[name]
            sys.path.remove(REF_PKG)
            importlib.reload(bb)
    finally:
        if REF_PKG in sys.path:
            sys.path.remove(REF_PKG)


def test_recall_and_grid_expansion_agree_with_the_reference_helpers():
    """bb.recall_at_k vs cuvs_bench.backends._utils.compute_recall, and run_config's Cartesian expansion vs expand_param_grid
    (python/cuvs_bench/cuvs_bench/backends/_utils.py:125-215), on seeded inputs — the reference's answers recorded."""
    gold = _reference_interface()
    for (found, truth, k), want in zip(recall_inputs(), gold["recall"], strict=True):  # set recall over the first k ids
        assert bb.recall_at_k(found, truth, k) == pytest.approx(want)
    grid = gold["param_grid"]
    mine = [dict(zip(sorted(grid), vals)) for vals in itertools.product(*[grid[x] for x in sorted(grid)])]
    theirs = gold["param_grid_expanded"]
    assert sorted(map(lambda d: sorted(d.items()), mine)) == sorted(map(lambda d: sorted(d.items()), theirs))
