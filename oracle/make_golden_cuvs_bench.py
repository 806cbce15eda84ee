#!/usr/bin/env python
"""Golden vectors from the REFERENCE ITSELF, executed in the build container (test infrastructure).

The reference ships one CPU implementation of the hot path's semantics: the exact k-nearest-neighbour search its benchmark
package uses to generate ground truth when no GPU is present,
    python/cuvs_bench/cuvs_bench/generate_groundtruth/__main__.py:104-171   cpu_search(dataset, queries, k, metric)
    python/cuvs_bench/cuvs_bench/generate_groundtruth/__main__.py:174-214   calc_truth (row batches + k-way merge)
(pure numpy; `metric` is spelled 'squeclidean' there).  This script imports that module from a reference checkout, runs it on
small seeded inputs and writes its OUTPUTS to tests/golden/cuvs_bench_cpu_groundtruth.json.  The inputs are not stored: tests
regenerate them from the seeds below with the same numpy Generator calls (`inputs()`), so the fixture stays small.

It also records, in tests/golden/cuvs_bench_interface.json, what tests/test_bench_backend_cpu.py checks the plugin
(cuvs_b200/bench_backend.py) against: the abstract methods of the package's BenchmarkBackend and their parameters, the JSON
records of its BuildResult / SearchResult, its recall and parameter-grid helpers on seeded inputs, and the `test` group of
its cuvs_ivf_pq.yaml.  The tests need only the fixtures, not the checkout.

    python oracle/make_golden_cuvs_bench.py <reference checkout>      # rewrites both fixtures
"""
import importlib
import inspect
import json
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "cuvs_bench_cpu_groundtruth.json")
OUT_INTERFACE = os.path.join(ROOT, "tests", "golden", "cuvs_bench_interface.json")

CASES = [
    # BASELINE configs[0]'s shape: 10k x 128 f32, k = 10
    dict(name="c0_10k_x_128_l2", n=10_000, d=128, nq=100, k=10, metric="squeclidean", seed=123, via="calc_truth"),
    dict(name="small_ip", n=3_000, d=33, nq=50, k=7, metric="inner_product", seed=5, via="cpu_search"),
    dict(name="small_l2_k1", n=777, d=8, nq=40, k=1, metric="squeclidean", seed=9, via="cpu_search"),
]


def inputs(case):
    """Seeded inputs of a case — the SAME calls are made by the tests (tests/test_oracle_golden.py)."""
    rng = np.random.default_rng(case["seed"])
    ds = rng.standard_normal((case["n"], case["d"]), dtype=np.float32)
    qs = rng.standard_normal((case["nq"], case["d"]), dtype=np.float32)
    return ds, qs


def recall_inputs():
    """Seeded (found, truth, k) triples for the recall helper (tests/test_bench_backend_cpu.py feeds the same ones to ours)."""
    rng = np.random.default_rng(3)
    for k, gtk in [(8, 16), (10, 10), (1, 5), (12, 12)]:
        found = np.stack([rng.permutation(40)[:k] for _ in range(25)])
        truth = np.stack([rng.permutation(40)[:gtk] for _ in range(25)])
        yield found, truth, k


PARAM_GRID = {"nlist": [1024, 2048], "pq_dim": [64, 32], "ratio": [10]}
BUILD_RESULT = dict(index_path="", build_time_seconds=1.0, index_size_bytes=2, algorithm="a", build_params={"nlist": 4})
SEARCH_RESULT = dict(neighbors=None, distances=None, search_time_ms=3.5, queries_per_second=1000.0, recall=0.9, algorithm="a",
                     search_params=[{"nprobe": 5}], latency_percentiles={"p50": 1.0, "p99": 2.0}, gpu_time_seconds=0.25,
                     cpu_time_seconds=0.5, metadata={"batch_size": 10})


def interface(ref_pkg):
    import yaml
    base = importlib.import_module("cuvs_bench.backends.base")
    utils = importlib.import_module("cuvs_bench.backends._utils")
    methods = {}
    for name in sorted(base.BenchmarkBackend.__abstractmethods__):
        attr = inspect.getattr_static(base.BenchmarkBackend, name)
        methods[name] = None if isinstance(attr, property) else list(inspect.signature(attr).parameters)
    algos = os.path.join(ref_pkg, "cuvs_bench", "config", "algos", "cuvs_ivf_pq.yaml")
    out = {"source": "rapidsai/cuvs python/cuvs_bench/cuvs_bench (backends/base.py, backends/_utils.py, config/algos/cuvs_ivf_pq.yaml), "
                     "recorded by oracle/make_golden_cuvs_bench.py",
           "abstract_methods": methods,
           "build_result_json": base.BuildResult(**BUILD_RESULT).to_json(),
           "search_result_json": base.SearchResult(**SEARCH_RESULT).to_json(),
           "recall": [utils.compute_recall(found, truth, k) for found, truth, k in recall_inputs()],
           "param_grid": PARAM_GRID, "param_grid_expanded": utils.expand_param_grid(PARAM_GRID),
           "cuvs_ivf_pq_test_group": yaml.safe_load(open(algos))["groups"]["test"]}
    with open(OUT_INTERFACE, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", OUT_INTERFACE, os.path.getsize(OUT_INTERFACE), "bytes")


def main(ref_pkg):
    sys.path.insert(0, ref_pkg)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = importlib.import_module("cuvs_bench.generate_groundtruth.__main__")
    assert not ref.gpu_system and ref.xp.__name__ == "numpy", "expected the reference's numpy fallback path"
    out = {"source": "rapidsai/cuvs python/cuvs_bench/cuvs_bench/generate_groundtruth/__main__.py (cpu_search / calc_truth), "
                     "executed by oracle/make_golden_cuvs_bench.py in the build container",
           "numpy": np.__version__, "cases": []}
    for c in CASES:
        ds, qs = inputs(c)
        if c["via"] == "calc_truth":
            d, i = ref.calc_truth(ds, qs, c["k"], metric=c["metric"])
        else:
            d, i = ref.cpu_search(ds, qs, c["k"], metric=c["metric"])
        out["cases"].append(dict(c, ids=np.asarray(i).astype(int).tolist(),
                                 distances=[[float(np.float32(v)) for v in row] for row in np.asarray(d)]))
    with open(OUT, "w") as f:
        json.dump(out, f)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")
    interface(ref_pkg)


if __name__ == "__main__":
    main(os.path.join(sys.argv[1], "python", "cuvs_bench"))
