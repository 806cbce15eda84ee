#!/usr/bin/env python
"""bench.py — one JSON line per run (driver contract, "tier" reading).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A step = one search() of the whole 10k-query batch through the library's C ABI.
  value   QPS with queries resident in HBM (device-timed, CUDA events, L2 flushed between steps)
  e2e     QPS through the public Python binding with HOST (pinned) queries: H2D of the batch and D2H
          of neighbors+distances are inside the timed region
  roofline  dominant kernel, timed live with CUDA events on the launching stream (cuvsB200Timing*)
  cpu_baseline  the oracle (C port, OpenMP) on a bounded sample of the same workload, rank 0, N=1
--impl reference: the reference has no CPU implementation of these searches and its CUDA build
cannot be produced offline (DESIGN.md), so the reference arm times the oracle port on the host cores.

Workloads (--workload): ivf_pq (DEFAULT = the metric's configuration: 100M x 128 f32 on one GPU, n_lists 16384, pq_dim 64 (64-byte
codes), n_probes 48, exact refine of 2k candidates, batch 10k, k 10; 51 GB of vectors generated on the device; --lut-dtype
f16|u8|f32; N > 1 = index sharded by IVF list, one all-gather of partial top-k), ivf_pq_c2 (BASELINE configs[2]: 10M x 128, n_lists
1024, n_probes 64), brute_force (configs[1], 1M x 128, bit-exact vs the oracle), cagra (configs[3], 10M x 96, degree 64, itopk 64;
--walk-bits 32|16), ivf_flat (configs[4] scaled to 10M, list-sharded for N > 1).  --no-cpu skips the CPU baseline, --no-aux the
secondary harder-data point.  --dump-outputs DIR writes what the last timed step returned (distances.npy, neighbors.npy) so
that two builds can be compared output for output: the inputs are generated from fixed seeds, and index builds sum and order
in input order, not in atomic order (tests/test_build_determinism_gpu.py asserts equal indexes and equal search answers for
two builds of one input).  Recall denominators come from
our exact brute force, itself checked against the oracle on a slice of the same tensors (config.ground_truth_check); a failed
check or recall < 0.95 adds PARITY_FAILED to the line.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm=j["hbm_gbs"], tf_burst=j["bf16_tflops"], tf_sust=j.get("bf16_tflops_sustained", j["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, gpu_index=0):
        self.rows, self.stop, self.idx = [], threading.Event(), gpu_index
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows else None,
                "samples": len(self.rows), "reasons": sorted(reasons),
                "note": "sampled over a ~1.5 s pre-load of the same search plus the timed steps"}


# ----------------------------------------------------------------------------------------- workloads
def gen_clustered(n, d, seed, centers, sigma=0.25, device="cuda", chunk=1 << 20):
    """SURVEY §8d synthetic data: points = centre + sigma * N(0, I), generated on the device."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n, d), dtype=torch.float32, device=device)
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        lab = torch.randint(0, centers.shape[0], (e - s,), generator=g, device=device)
        out[s:e] = centers[lab] + sigma * torch.randn((e - s, d), generator=g, device=device)
    return out


def gen_manifold(n, d, seed, rank=16, noise=0.05, device="cuda", chunk=1 << 20):
    """Embedding-like data: x = z A + noise * N(0, I_d), z ~ N(0, I_rank), A fixed (seed 99) — intrinsic dimension `rank`,
    so nearest neighbours are meaningful (SIFT/DEEP-like), unlike iid or well-separated-cluster data in >= 96 dimensions."""
    ga = torch.Generator(device=device)
    ga.manual_seed(99)
    A = torch.randn((rank, d), generator=ga, device=device) / rank ** 0.5
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n, d), dtype=torch.float32, device=device)
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        z = torch.randn((e - s, rank), generator=g, device=device)
        out[s:e] = z @ A + noise * torch.randn((e - s, d), generator=g, device=device)
    return out


class BruteForceWorkload:
    """configs[1]: brute_force::search 1M x 128 f32 L2, batch 10k, k=10."""
    name = "brute_force 1M x 128 f32 L2 (sqeuclidean), batch 10k, k=10"
    dtype = "bf16x3->f32"  # split-bf16 tensor-core products, fp32 accumulate, fp32 exact re-scoring
    timing_section = "tc_scan"

    def __init__(self, n=1_000_000, d=128, nq=10_000, k=10, seed=1234):
        self.n, self.d, self.nq, self.k = n, d, nq, k
        from cuvs_b200.neighbors import brute_force
        self.bf = brute_force
        g = torch.Generator(device="cuda")
        g.manual_seed(99)
        centers = torch.randn((max(1, n // 1000), d), generator=g, device="cuda")
        self.dataset = gen_clustered(n, d, seed, centers)
        self.queries = gen_clustered(nq, d, seed + 3087, centers)
        self.index = brute_force.build(self.dataset)
        self.h_queries = self.queries.cpu().pin_memory()
        self.neighbors = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        self.distances = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        self.h_neighbors = torch.empty((nq, k), dtype=torch.int64).pin_memory()
        self.h_distances = torch.empty((nq, k), dtype=torch.float32).pin_memory()

    def config(self):
        return {"workload": self.name, "n": self.n, "dim": self.d, "batch": self.nq, "k": self.k, "metric": "sqeuclidean",
                "data": "clustered gaussians (SURVEY 8d), seed 1234/4321", "l2_flush": "256 MiB write between timed steps",
                "recall_at_10": 1.0, "parallelism": "single GPU"}

    def step(self, res):
        self.bf.search(self.index, self.queries, self.k, neighbors=self.neighbors, distances=self.distances, resources=res)

    def e2e_step(self, res):
        q = self.h_queries.to("cuda", non_blocking=True)
        self.bf.search(self.index, q, self.k, neighbors=self.neighbors, distances=self.distances, resources=res)
        self.h_neighbors.copy_(self.neighbors, non_blocking=True)
        self.h_distances.copy_(self.distances, non_blocking=True)

    def e2e_bytes(self):
        return self.nq * self.d * 4, self.nq * self.k * 12

    def units(self):
        return self.nq

    def roofline(self, kernel_ms, pk):
        flops = 2.0 * self.nq * self.n * self.d  # algorithmic (useful) FLOPs; the 3-term split executes 3x this
        ach = flops / (kernel_ms * 1e-3) / 1e12
        return {"bound": "tensor", "kernel": "tc_scan_kernel (tcgen05, split-bf16 x3 + fused top-k')", "achieved": ach,
                "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": ach / pk["tf_burst"],
                "frac_executed_flops": 3 * ach / pk["tf_burst"], "peak_source": pk["src"] + " bf16 burst (kernel timed alone)",
                "traffic": None, "kernel_ms": kernel_ms}

    def cpu_baseline(self, budget_s=20.0):
        return cpu_baseline_on_slice(self.dataset, self.queries, self.k, budget_s, "the same search, answered on the host")

    def outputs(self):
        return {"distances": self.distances, "neighbors": self.neighbors}

    def check(self):
        import oracle
        qs = self.queries[:32].cpu().numpy()
        rd, ri = oracle.knn(self.dataset.cpu().numpy(), qs, self.k)
        ok = (self.neighbors[:32].cpu().numpy() == ri).all()
        return bool(ok)


def cpu_exact_knn_rate(ds_rows, qs, k, budget_s, what, n_total=None, repeats=3):
    """CPU baseline: exact fp32 kNN with the oracle port on ALL host threads, in a separate process with pinned OpenMP
    threads (oracle/cpu_baseline.py), `repeats` timed repeats after a warm-up, median reported.  `ds_rows` may be a ROW SLICE of the
    workload's dataset (host RAM / time bound): the rate is then scaled by rows(slice) / n_total — exact kNN cost is linear
    in the rows scanned — and the sample says so."""
    import tempfile
    threads = os.cpu_count() or 1
    n_slice = ds_rows.shape[0]
    n_total = n_total or n_slice
    tag = f"cuvs_b200_cpu_{os.getpid()}"
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    f_ds, f_q = os.path.join(shm, tag + "_ds.npy"), os.path.join(shm, tag + "_q.npy")
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), OMP_PROC_BIND="spread", OMP_PLACES="threads", MKL_NUM_THREADS=str(threads))
    script = os.path.join(ROOT, "oracle", "cpu_baseline.py")
    try:
        np.save(f_ds, ds_rows)
        # size the query sample from a short probe run so that warm-up + repeats take ~budget_s
        np.save(f_q, np.ascontiguousarray(qs[:16]))
        r = subprocess.run([sys.executable, script, f_ds, f_q, str(k), "1"], env=env, capture_output=True, text=True, timeout=600)
        probe = json.loads(r.stdout.strip().splitlines()[-1])
        rate = max(probe["probe_rates_qps"].values())
        # at least one full 256-query block: the workload is a 10k-query BATCH, and a skinny GEMM (a few dozen queries per pass
        # over the rows) would measure the host's memory bandwidth, not what a tuned CPU brute force does with the batch
        m = int(min(len(qs), max(256, budget_s / (repeats + 1.0) * rate)))
        np.save(f_q, np.ascontiguousarray(qs[:m]))
        r = subprocess.run([sys.executable, script, f_ds, f_q, str(k), str(repeats), probe["formulation"]], env=env, capture_output=True,
                           text=True, timeout=900)
        out = json.loads(r.stdout.strip().splitlines()[-1])
    finally:
        for f in (f_ds, f_q):
            if os.path.exists(f):
                os.remove(f)
    ts = sorted(out["times_s"])
    scale = n_slice / float(n_total)
    qps = [m / t * scale for t in ts]
    form = "blocked SGEMM + top-k (oracle.knn_blocked)" if out["formulation"] == "blocked" else "sequential-fmaf scan (oracle.knn, OpenMP)"
    sample = (f"{m} queries, exact fp32 kNN over {n_slice} rows"
              + (f" (a row slice of the {n_total}-row dataset; rate scaled by {scale:.4g}: cost is linear in rows)" if n_slice != n_total else "")
              + f" ({what}); {form}; separate process, OMP_PROC_BIND=spread OMP_PLACES=threads; {repeats} repeats after warm-up: "
              f"median {qps[len(qps) // 2]:.3g}, min {qps[-1]:.3g}, max {qps[0]:.3g} q/s")
    return {"value": qps[len(qps) // 2], "unit": "queries/s", "cores": threads, "kind": "port", "sample": sample,
            "repeats_qps": qps}


CPU_SLICE_ROWS = 4_000_000   # rows of the dataset the CPU arms scan (host RAM / time bound); rates are scaled to the full size
GT_CHECK_ROWS = 1_000_000    # rows over which the ground-truth machinery is checked against the oracle
GT_CHECK_QUERIES = 256


def cpu_baseline_on_slice(dataset, queries, k, budget_s, what):
    n = dataset.shape[0]
    m = min(n, CPU_SLICE_ROWS)
    return cpu_exact_knn_rate(dataset[:m].cpu().numpy(), queries[:1024].cpu().numpy(), k, budget_s, what, n_total=n)


def oracle_gt_check(dataset, queries, k):
    """The recall denominators of the IVF / graph workloads come from our own exact brute force (the only thing that can
    answer 10k queries over 1e8 rows here).  This pins that machinery to the ORACLE on the same tensors: exact kNN of the
    first 256 queries over the first 1M rows by `oracle.knn` (CPU, pinned fp32 arithmetic) vs `exact_ground_truth` on the
    same slice — ids must agree (bit-exact brute force; a handful of exact-tie swaps are tolerated)."""
    import oracle
    oracle.set_threads(os.cpu_count() or 1)
    rows = min(dataset.shape[0], GT_CHECK_ROWS)
    nq = min(queries.shape[0], GT_CHECK_QUERIES)
    ds, qs = dataset[:rows], queries[:nq]
    t0 = time.time()
    _, ri = oracle.knn(ds.cpu().numpy(), qs.cpu().numpy(), k)
    ours = exact_ground_truth(ds, qs.contiguous(), k).cpu().numpy()
    same = float((ours == ri).mean())
    sets = float(np.mean([len(np.intersect1d(a, b)) / float(k) for a, b in zip(ours, ri)]))
    return {"queries": int(nq), "rows": int(rows), "ids_identical": same, "id_sets_identical": sets, "ok": bool(sets >= 0.999),
            "checker": "oracle.knn (CPU)", "seconds": round(time.time() - t0, 1)}


def exact_ground_truth(dataset, queries, k, chunk=10_000_000):
    """Exact kNN ids by our brute force, the dataset taken in chunks (bounds the temporary bf16 planes at 100M rows)."""
    from cuvs_b200.neighbors import brute_force
    best_d, best_i = None, None
    for c0 in range(0, dataset.shape[0], chunk):
        bf = brute_force.build(dataset[c0:c0 + chunk])
        d, i = brute_force.search(bf, queries, k)
        i = i.to(torch.int64) + c0
        del bf
        if best_d is None:
            best_d, best_i = d, i
        else:
            dd, ii = torch.cat([best_d, d], 1), torch.cat([best_i, i], 1)
            sel = dd.topk(k, dim=1, largest=False).indices
            best_d, best_i = dd.gather(1, sel), ii.gather(1, sel)
    return best_i


class IvfPqWorkload:
    """The metric's configuration: ivf_pq::search 100M x 128 f32 on one B200, batch 10k, k=10 (n_lists 16384, pq_dim 64 ->
    64-byte codes, the smallest n_probes with recall@10 >= 0.95 after an exact refine of 2k candidates).  BASELINE configs[2]
    (10M x 128, n_lists 1024, n_probes 64) is `--workload ivf_pq_c2`."""
    dtype = "bf16 (PQ codes decoded to bf16 on the SM, tcgen05 bf16 MMA, fp32 accumulate); fp32 exact refine"
    timing_section = "pq_scan"

    def __init__(self, n=100_000_000, d=128, nq=10_000, k=10, n_lists=16384, pq_dim=64, n_probes=48, refine_ratio=2, seed=1234,
                 rank=0, world=1, lut_dtype="f16", data_rank=16, resources=None, shard_rows=False):
        from cuvs_b200.neighbors import brute_force, ivf_pq, refine
        self.n, self.d, self.nq, self.k = n, d, nq, k
        self.rank, self.world = rank, world
        self._res = resources
        self.shard_rows = bool(shard_rows) and world > 1   # N > 1: keep only this rank's fp32 rows for the exact refine
        self.local_rows = self.local_gid = None
        self.n_lists, self.pq_dim, self.n_probes, self.refine_ratio = n_lists, pq_dim, n_probes, refine_ratio
        self.data_rank = data_rank
        self.name = (f"ivf_pq {n // 1_000_000}M x {d} f32, n_lists={n_lists} pq_dim={pq_dim} pq_bits=8 n_probes={n_probes}, "
                     f"batch {nq}, k={k}, refine_ratio={refine_ratio}")
        self.pq, self.refine = ivf_pq, refine
        self.dataset = gen_manifold(n, d, seed, rank=data_rank)
        self.queries = gen_manifold(nq, d, seed + 3087, rank=data_rank)
        t0 = time.time()
        self.train_fraction = min(0.5, max(4_000_000, 256 * n_lists) / n)
        params = ivf_pq.IndexParams(n_lists=n_lists, pq_dim=pq_dim, pq_bits=8, kmeans_n_iters=10,
                                    kmeans_trainset_fraction=self.train_fraction)
        if world == 1:
            self.index = ivf_pq.build(params, self.dataset)
            self.sharded = None
        else:
            self.index, self.sharded = self._build_shard(params)
        torch.cuda.synchronize()
        self.build_s = time.time() - t0
        import numpy as _np
        self.lut_dtype = lut_dtype
        lut = {"f32": _np.float32, "f16": _np.float16, "u8": _np.uint8}[lut_dtype]
        self.sp = ivf_pq.SearchParams(n_probes=n_probes, lut_dtype=lut)
        self.kc = k * refine_ratio
        self.cand = torch.empty((nq, self.kc), dtype=torch.int64, device="cuda")
        self.cand_d = torch.empty((nq, self.kc), dtype=torch.float32, device="cuda")
        self.h_queries = self.queries.cpu().pin_memory()
        self.neighbors = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        self.distances = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        self.h_neighbors = torch.empty((nq, k), dtype=torch.int64).pin_memory()
        self.h_distances = torch.empty((nq, k), dtype=torch.float32).pin_memory()
        # ground truth (exact, our brute force — itself pinned to the oracle on a slice of these tensors) for recall
        self.gt = exact_ground_truth(self.dataset, self.queries, k)
        self.gt_check = oracle_gt_check(self.dataset, self.queries, k) if rank == 0 else None
        self.recall = None
        if self.shard_rows:
            self.dataset = None  # from here on the rank holds its shard only: index + its own rows + the id map
            torch.cuda.empty_cache()

    def _build_shard(self, params):
        """List-sharded index: quantizers trained on rank 0 and broadcast (bit-identical on every rank), every rank keeps the
        rows whose IVF list it owns (list % world == rank).  No inter-rank movement of vectors (cuvs_b200/distributed.py)."""
        import torch.distributed as dist
        from cuvs_b200.cluster import kmeans
        from cuvs_b200.distributed import Comm, ShardedIvfFlat, owner_of_list
        pq = self.pq
        p0 = pq.IndexParams(n_lists=self.n_lists, pq_dim=self.pq_dim, pq_bits=8, kmeans_n_iters=10, add_data_on_build=False,
                            kmeans_trainset_fraction=self.train_fraction)  # same training subsample as the 1-GPU build
        proto = pq.build(p0, self.dataset)
        quant = [proto.pq_centers.clone(), proto.centers.clone(), proto.centers_rot.clone(), proto.rotation_matrix.clone()]
        for t in quant:
            dist.broadcast(t, src=0)
        index = pq.build_precomputed(p0, self.d, *quant)
        kp = kmeans.KMeansParams(n_clusters=self.n_lists)
        ids = torch.arange(self.n, dtype=torch.int64, device="cuda")
        step = 1 << 20
        own_rows, own_gid, n_local = [], [], 0
        for s in range(0, self.n, step):
            rows = self.dataset[s:s + step]
            labels, _ = kmeans.predict(kp, rows, quant[1])
            mine = owner_of_list(labels.to(torch.int64), self.world) == self.rank
            r, g = rows[mine].contiguous(), ids[s:s + step][mine].contiguous()
            if self.shard_rows:
                # sharded memory plan: the index stores LOCAL row numbers, the rank keeps only the fp32 rows of its own lists
                # (for the exact refine) and the local -> global id map; the full dataset is dropped after the ground truth
                own_rows.append(r)
                own_gid.append(g)
                g = torch.arange(n_local, n_local + r.shape[0], dtype=torch.int64, device="cuda")
                n_local += r.shape[0]
            pq.extend(index, r, g)
        if self.shard_rows:
            self.local_rows, self.local_gid = torch.cat(own_rows), torch.cat(own_gid)
            del own_rows, own_gid

        def local_search(local, sp, q, k):
            res = self._res
            rows = self.local_rows if self.shard_rows else self.dataset
            if self.refine_ratio > 1:
                pq.search(sp, local, q, self.kc, neighbors=self.cand, distances=self.cand_d, resources=res)
                self.refine(rows, q, self.cand, indices=self.neighbors, distances=self.distances, resources=res)
            else:
                pq.search(sp, local, q, k, neighbors=self.neighbors, distances=self.distances, resources=res)
            if self.shard_rows:  # local row numbers -> global ids (pad entries, < 0 or out of range, pass through)
                # (torch ops on the current stream = the resource's stream: bench creates Resources() on it)
                loc = self.neighbors
                ok = (loc >= 0) & (loc < self.local_gid.shape[0])
                self.neighbors_g = torch.where(ok, self.local_gid[loc.clamp(0, self.local_gid.shape[0] - 1)], loc)
                return self.distances, self.neighbors_g
            return self.distances, self.neighbors  # (no host sync: the exchange step is enqueued on the same stream)

        comm = Comm(self._res) if self._res is not None else None
        return index, ShardedIvfFlat(index, local_search=local_search, comm=comm)

    def _search(self, q, res):
        if self.sharded is not None:
            self._res = res
            d, i = self.sharded.search(self.sp, q, self.k, resources=res)
            self.final_d, self.final_i = d, i
            return
        if self.refine_ratio > 1:
            self.pq.search(self.sp, self.index, q, self.kc, neighbors=self.cand, distances=self.cand_d, resources=res)
            self.refine(self.dataset, q, self.cand, indices=self.neighbors, distances=self.distances, resources=res)
        else:
            self.pq.search(self.sp, self.index, q, self.k, neighbors=self.neighbors, distances=self.distances, resources=res)

    def step(self, res):
        self._search(self.queries, res)

    def e2e_step(self, res):
        q = self.h_queries.to("cuda", non_blocking=True)
        self._search(q, res)
        self.h_neighbors.copy_(self.final_i if self.sharded is not None else self.neighbors, non_blocking=True)
        self.h_distances.copy_(self.final_d if self.sharded is not None else self.distances, non_blocking=True)

    def e2e_bytes(self):
        return self.nq * self.d * 4, self.nq * self.k * 12

    def units(self):
        return self.nq

    def outputs(self):
        if self.sharded is not None:
            return {"distances": self.final_d, "neighbors": self.final_i}
        return {"distances": self.distances, "neighbors": self.neighbors}

    def check(self):
        nb = self.final_i if self.sharded is not None else self.neighbors
        hit = (nb.unsqueeze(2) == self.gt.unsqueeze(1)).any(dim=2).float().mean().item()
        self.recall = hit
        return hit >= 0.95 and (self.gt_check is None or self.gt_check["ok"])

    def config(self):
        sizes = self.index.list_sizes.float()
        return {"workload": self.name, "n": self.n, "dim": self.d, "batch": self.nq, "k": self.k, "metric": "sqeuclidean",
                "n_lists": self.n_lists, "pq_dim": self.pq_dim, "pq_bits": 8, "n_probes": self.n_probes,
                "refine_ratio": self.refine_ratio, "lut_dtype": self.lut_dtype,
                "scan": ("2-pass split-bf16 residual x bf16-exact decoded rows = the fp32 LUT sums to fp32 rounding" if self.lut_dtype == "f32"
                         else "1-pass bf16 residual x decoded rows (reduced-precision LUT requested)"),
                "scan_kernel": self.scan_kernel_name(),
                "recall_at_10": self.recall, "ground_truth_check": self.gt_check, "index_build_s": round(self.build_s, 2),
                "list_size_max_over_mean": round((sizes.max() / sizes.mean()).item(), 2),
                "index_device_bytes": self.index.device_bytes, "index_streamed": self.index.streamed,
                "data": f"rank-{self.data_rank} gaussian manifold in {self.d}-d + 0.05 noise (embedding-like), seeds 1234/4321; "
                        "SURVEY 8d's clustered gaussians (sigma 0.25: 1000 near-equidistant neighbours per point) make recall@10 a coin "
                        "toss for any PQ/graph method and are used for brute_force only; `harder_data` below = the same run on rank-32 data",
                "l2_flush": "256 MiB write between timed steps",
                "parallelism": "single GPU" if self.world == 1 else
                f"index sharded by IVF list over {self.world} GPUs (list % {self.world}), per-shard search + exact refine, one NCCL "
                "all-gather of partial top-k + k-way merge on every rank; "
                + ("every rank keeps only the fp32 rows of its own lists (local ids + id map)" if self.shard_rows
                   else "every rank keeps the full fp32 dataset for the refine")}

    def dense(self):
        """The library's own rule (ivf_pq.cu: dense_probing): a small index also caches decoded rows, and a batch that sends
        >= 128 queries to the average list is served from them instead of re-decoding each list per 64-query group."""
        return bool(getattr(self.index, "has_decoded_rows", False)) and self.kc <= 32 and self.nq * self.n_probes >= 128 * self.n_lists

    def scan_kernel_name(self):
        if not getattr(self.index, "streamed", True) or self.dense():
            return "tc_scan_kernel over the index's decoded bf16 rows (small index + densely probing batch: scan_tc.cu)"
        return "pq_stream_scan_kernel: 64-byte codes streamed from HBM, decoded on the SM (scan_pq.cu)"

    def scan_volume(self):
        """(sum over (query, probe) pairs of the probed list's length, padded rows of the DISTINCT probed lists) — from the
        probe sets the library itself would compute (lists owned by other ranks have size 0 here)."""
        c = self.index.centers
        sizes = self.index.list_sizes.to(torch.int64)
        touched = torch.zeros(self.n_lists, dtype=torch.bool, device="cuda")
        tot = 0
        for s in range(0, self.nq, 2048):
            q = self.queries[s:s + 2048]
            dist = (c * c).sum(1)[None, :] - 2.0 * q @ c.t()
            pr = dist.topk(self.n_probes, dim=1, largest=False).indices
            tot += int(sizes[pr].sum().item())
            touched[pr.reshape(-1)] = True
        padded = ((sizes + 127) // 128 * 128)[touched & (sizes > 0)]
        return tot, int(padded.sum().item())

    def roofline(self, kernel_ms, pk):
        """Dominant kernel = the fine scan.  Two ceilings, both from ALGORITHMIC work (DESIGN.md §5):
        hbm    every probed list's code stream read once: (pq_dim + 4) bytes per (padded) row of the distinct probed lists
               — the compulsory traffic of a batch (at 100M rows every list is probed by some query of a 10k batch);
        tensor one multiply-add per (query-probe pair, list row, component): 2 * scanned_rows * dim FLOP.
        `bound` names the ceiling the launch sits closer to; `frac` is against it."""
        rows, touched_rows = self.scan_volume()
        flops = 2.0 * rows * self.d
        streamed = getattr(self.index, "streamed", True) and not self.dense()
        hbm_bytes = touched_rows * ((self.pq_dim + 4.0) if streamed else (2.0 * self.d + 32.0))  # decoded rows: bf16 row + half-norm planes
        t = kernel_ms * 1e-3
        tf, gbs = flops / t / 1e12, hbm_bytes / t / 1e9
        f_t, f_h = tf / pk["tf_burst"], gbs / pk["hbm"]
        kern = ("pq_stream_scan_kernel (PQ codes streamed by cp.async.bulk, decoded on the SM, tcgen05 bf16 MMA, threshold "
                "filter epilogue)" if streamed else "tc_scan_kernel over decoded PQ rows (TMA tiles, tcgen05 bf16 MMA, fused top-k')")
        out = {"kernel": kern, "kernel_ms": kernel_ms, "scanned_rows": rows, "touched_list_rows": touched_rows,
               "algorithmic_hbm_bytes": hbm_bytes, "algorithmic_flops": flops, "traffic": None,
               "hbm": {"achieved_GBps": gbs, "peak_GBps": pk["hbm"], "frac": f_h},
               "tensor": {"achieved_TFLOPs": tf, "peak_TFLOPs": pk["tf_burst"], "frac": f_t},
               "peak_source": pk["src"] + " (HBM copy bandwidth; bf16 burst: the kernel is timed alone)",
               "reference_formulation": {"algorithmic_code_bytes": rows * self.pq_dim,
                                         "note": "the reference streams list_len * pq_dim code bytes per (query, probe) pair; this kernel "
                                                 "streams each probed list once per group of <= 64 probing queries"}}
        if f_h >= f_t:
            out.update({"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": f_h})
        else:
            out.update({"bound": "tensor", "achieved": tf, "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": f_t})
        return out

    def cpu_baseline(self, budget_s=20.0):
        return cpu_baseline_on_slice(self.dataset, self.queries, self.k, budget_s,
                                     "the reference has no CPU IVF / graph search; exact kNN is its CPU answer")


class CagraWorkload:
    """configs[3]: cagra::search 10M x 96 f32, graph_degree=64 itopk=64, batch 10k."""
    dtype = "f32"
    timing_section = "cagra_search"

    def __init__(self, n=10_000_000, d=96, nq=10_000, k=10, degree=64, itopk=64, seed=1234, rank=0, world=1, walk_bits=32):
        from cuvs_b200.neighbors import brute_force, cagra
        self.n, self.d, self.nq, self.k, self.degree, self.itopk = n, d, nq, k, degree, itopk
        self.name = f"cagra {n // 1_000_000}M x {d} f32, graph_degree={degree} itopk={itopk} search_width=1, batch {nq}, k={k}"
        self.cagra = cagra
        self.dataset = gen_manifold(n, d, seed)
        self.queries = gen_manifold(nq, d, seed + 3087)
        t0 = time.time()
        self.index = cagra.build(cagra.IndexParams(graph_degree=degree, intermediate_graph_degree=2 * degree), self.dataset)
        torch.cuda.synchronize()
        self.build_s = time.time() - t0
        self.walk_bits = walk_bits
        if walk_bits == 16:
            self.index.set_walk_precision(16)
        self.sp = cagra.SearchParams(itopk_size=itopk)
        self.h_queries = self.queries.cpu().pin_memory()
        self.neighbors = torch.empty((nq, k), dtype=torch.uint32, device="cuda")
        self.distances = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        self.h_neighbors = torch.empty((nq, k), dtype=torch.uint32).pin_memory()
        self.h_distances = torch.empty((nq, k), dtype=torch.float32).pin_memory()
        self.gt = exact_ground_truth(self.dataset, self.queries, k)
        self.gt_check = oracle_gt_check(self.dataset, self.queries, k)
        self.recall = None

    def step(self, res):
        self.cagra.search(self.sp, self.index, self.queries, self.k, neighbors=self.neighbors, distances=self.distances, resources=res)

    def e2e_step(self, res):
        q = self.h_queries.to("cuda", non_blocking=True)
        self.cagra.search(self.sp, self.index, q, self.k, neighbors=self.neighbors, distances=self.distances, resources=res)
        self.h_neighbors.copy_(self.neighbors, non_blocking=True)
        self.h_distances.copy_(self.distances, non_blocking=True)

    def e2e_bytes(self):
        return self.nq * self.d * 4, self.nq * self.k * 8

    def units(self):
        return self.nq

    def outputs(self):
        return {"distances": self.distances, "neighbors": self.neighbors}

    def check(self):
        nb = self.neighbors.to(torch.int64)
        self.recall = (nb.unsqueeze(2) == self.gt.unsqueeze(1)).any(dim=2).float().mean().item()
        return self.recall >= 0.95 and self.gt_check["ok"]

    def config(self):
        return {"workload": self.name, "n": self.n, "dim": self.d, "batch": self.nq, "k": self.k, "metric": "sqeuclidean",
                "graph_degree": self.degree, "itopk": self.itopk,
                "walk": "fp16 copy of the rows for the walk + fp32 re-rank of the final 32" if self.walk_bits == 16 else "fp32 rows",
                "recall_at_10": self.recall, "ground_truth_check": self.gt_check, "index_build_s": round(self.build_s, 2),
                "data": "rank-16 gaussian manifold in 96-d + 0.05 noise (embedding-like), seeds 1234/4321",
                "l2_flush": "256 MiB write between timed steps", "parallelism": "single GPU"}

    def roofline(self, kernel_ms, pk):
        """HBM-bound random gathers.  `achieved` = the walk's ALGORITHMIC bytes / live kernel time, where the algorithmic bytes
        are the dram bytes ncu measured for this exact configuration (profiles/traffic.json: every byte the walk reads is a
        first-touch row or adjacency gather — L2 hit rate 6 % — so measured dram traffic IS the algorithmic traffic); without
        a capture for this size the SURVEY 8d upper bound (every child row fetched, no hash dedup) is used and says so."""
        iters = self.itopk + 5
        row_b = self.d * (2 if self.walk_bits == 16 else 4)  # bytes of one vector row as the walk reads it
        bytes_ub = self.nq * ((self.itopk + self.degree + iters * self.degree) * row_b + iters * self.degree * 4)
        measured = ncu_traffic("cagra", self) if self.walk_bits == 32 else None
        used = measured if measured else bytes_ub
        ach = used / (kernel_ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "cagra_search_kernel (one warp per query, register bitonic top-k, smem hash)", "achieved": ach,
                "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "peak_source": pk["src"] + " HBM copy",
                "traffic": None, "kernel_ms": kernel_ms, "bytes_basis": "measured dram bytes per launch (ncu, profiles/traffic.json)" if measured
                else "UPPER BOUND of gathered bytes (every child row fetched); hash-deduplicated children are not fetched, so true traffic is lower",
                "upper_bound_bytes": bytes_ub}

    def cpu_baseline(self, budget_s=20.0):
        return cpu_baseline_on_slice(self.dataset, self.queries, self.k, budget_s,
                                     "the reference has no CPU IVF / graph search; exact kNN is its CPU answer")


class IvfFlatWorkload:
    """configs[4] scaled to what builds in-bench: ivf_flat::search n x 128 f32 (default 10M), sharded by IVF list over the
    ranks (list % world) with one NCCL all-gather of the partial top-k (cuvs_b200/distributed.py)."""
    dtype = "bf16 tensor-core list scan (1 pass), fp32 accumulate; exact fp32 re-score of the candidates"
    timing_section = "ivf_flat_scan"

    def __init__(self, n=10_000_000, d=128, nq=10_000, k=10, n_lists=4096, n_probes=64, seed=1234, rank=0, world=1, resources=None):
        from cuvs_b200.neighbors import ivf_flat
        from cuvs_b200.distributed import ShardedIvfFlat, build_sharded_ivf_flat
        self.n, self.d, self.nq, self.k, self.n_lists, self.n_probes = n, d, nq, k, n_lists, n_probes
        self.rank, self.world = rank, world
        self.name = f"ivf_flat {n // 1_000_000}M x {d} f32, n_lists={n_lists} n_probes={n_probes}, batch {nq}, k={k}"
        self.flat = ivf_flat
        self.dataset = gen_manifold(n, d, seed)
        self.queries = gen_manifold(nq, d, seed + 3087)
        t0 = time.time()
        params = ivf_flat.IndexParams(n_lists=n_lists, kmeans_n_iters=10, kmeans_trainset_fraction=min(0.5, max(2_000_000, 128 * n_lists) / n))
        if world == 1:
            self.index = ivf_flat.build(params, self.dataset)
            self.sharded = None
        else:
            step = 1 << 21
            ids = torch.arange(n, dtype=torch.int64, device="cuda")
            chunks = ((self.dataset[s:s + step], ids[s:s + step]) for s in range(0, n, step))
            n_train = int(max(2_000_000, 128 * n_lists))
            self.sharded = build_sharded_ivf_flat(params, self.dataset[:: max(1, n // n_train)].contiguous(), chunks, resources=resources)
            self.index = self.sharded.local
        torch.cuda.synchronize()
        self.build_s = time.time() - t0
        self.sp = ivf_flat.SearchParams(n_probes=n_probes)
        self.h_queries = self.queries.cpu().pin_memory()
        self.neighbors = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        self.distances = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        self.h_neighbors = torch.empty((nq, k), dtype=torch.int64).pin_memory()
        self.h_distances = torch.empty((nq, k), dtype=torch.float32).pin_memory()
        self.gt = exact_ground_truth(self.dataset, self.queries, k)
        self.gt_check = oracle_gt_check(self.dataset, self.queries, k) if rank == 0 else None
        self.recall = None

    def _search(self, q, res):
        if self.sharded is not None:
            self.final_d, self.final_i = self.sharded.search(self.sp, q, self.k, resources=res)
        else:
            self.flat.search(self.sp, self.index, q, self.k, neighbors=self.neighbors, distances=self.distances, resources=res)
            self.final_d, self.final_i = self.distances, self.neighbors

    def step(self, res):
        self._search(self.queries, res)

    def e2e_step(self, res):
        q = self.h_queries.to("cuda", non_blocking=True)
        self._search(q, res)
        self.h_neighbors.copy_(self.final_i, non_blocking=True)
        self.h_distances.copy_(self.final_d, non_blocking=True)

    def e2e_bytes(self):
        return self.nq * self.d * 4, self.nq * self.k * 12

    def units(self):
        return self.nq

    def outputs(self):
        return {"distances": self.final_d, "neighbors": self.final_i}

    def check(self):
        self.recall = (self.final_i.unsqueeze(2) == self.gt.unsqueeze(1)).any(dim=2).float().mean().item()
        return self.recall >= 0.95 and (self.gt_check is None or self.gt_check["ok"])

    def config(self):
        return {"workload": self.name, "n": self.n, "dim": self.d, "batch": self.nq, "k": self.k, "metric": "sqeuclidean",
                "n_lists": self.n_lists, "n_probes": self.n_probes, "recall_at_10": self.recall, "ground_truth_check": self.gt_check,
                "index_build_s": round(self.build_s, 2),
                "data": "rank-16 gaussian manifold in 128-d + 0.05 noise (embedding-like), seeds 1234/4321",
                "l2_flush": "256 MiB write between timed steps",
                "parallelism": "single GPU" if self.world == 1 else
                f"index sharded by IVF list over {self.world} GPUs (list % {self.world}), per-shard scan + exact re-score, one NCCL "
                "all-gather of partial top-k + k-way merge on every rank"}

    def roofline(self, kernel_ms, pk):
        # scanned (query, row) pairs of THIS rank (lists it owns), from the probe lists the library itself would compute
        c = self.flat_centers()
        sizes = self.index.list_sizes.to(torch.int64)
        rows = 0
        for s in range(0, self.nq, 2048):
            q = self.queries[s:s + 2048]
            dist = (c * c).sum(1)[None, :] - 2.0 * q @ c.t()
            rows += int(sizes[dist.topk(self.n_probes, dim=1, largest=False).indices].sum().item())
        flops = 2.0 * rows * self.d
        ach = flops / (kernel_ms * 1e-3) / 1e12
        return {"bound": "tensor", "kernel": "tc_scan_kernel over IVF-Flat lists (tcgen05 bf16 1-pass, fused top-k')", "achieved": ach,
                "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": ach / pk["tf_burst"],
                "peak_source": pk["src"] + " bf16 burst (kernel timed alone)", "traffic": None, "kernel_ms": kernel_ms,
                "scanned_rows": rows,
                "reference_formulation": {"algorithmic_bytes": rows * self.d * 4,
                                          "note": "the reference re-reads list_len*dim*4 bytes per (query, probe) pair (SURVEY a8)"}}

    def flat_centers(self):
        return self.index.centers

    def cpu_baseline(self, budget_s=20.0):
        return IvfPqWorkload.cpu_baseline(self, budget_s)


class IvfPqC2Workload(IvfPqWorkload):
    """BASELINE configs[2]: ivf_pq::search 10M x 128 f32, nlist=1024 pq_dim=64 nprobe=64, batch 10k."""

    def __init__(self, n=10_000_000, n_lists=1024, n_probes=64, **kw):
        super().__init__(n=n, n_lists=n_lists, n_probes=n_probes, **kw)


WORKLOADS = {"brute_force": BruteForceWorkload, "ivf_pq": IvfPqWorkload, "ivf_pq_c2": IvfPqC2Workload, "cagra": CagraWorkload,
             "ivf_flat": IvfFlatWorkload}


METRIC_NAME = "QPS @ recall@10>=0.95 (queries/s of one batched 10k-query search() call; recall@10 in config)"


def ncu_traffic(workload, wl):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
    capture (profiles/traffic.json, written by scripts/ncu_summary.py); only valid for the configuration it was captured on."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")
    try:
        ent = json.load(open(path)).get(workload)
    except (OSError, ValueError):
        return None
    if not ent or ent.get("n") != getattr(wl, "n", None) or ent.get("world", 1) != getattr(wl, "world", 1):
        return None
    return ent.get("dram_bytes_per_launch")


DUMP_LIMIT_BYTES = 60 << 20   # array bytes of --dump-outputs: under 64 MB in all with the .npy headers


def dump_outputs(outputs, out_dir):
    """Writes each output of the timed search as out_dir/<name>.npy: floating-point values as float32, ids as float64 (exact
    below 2**53).  Above DUMP_LIMIT_BYTES in all, every array keeps the same fixed, seeded sample of query rows, whose row
    numbers go to rows.npy."""
    arrays = {}
    for name, t in outputs.items():
        a = t.detach().cpu().numpy()
        arrays[name] = a.astype(np.float32 if a.dtype.kind == "f" and a.itemsize <= 4 else np.float64)
    n = next(iter(arrays.values())).shape[0]
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        keep = int(DUMP_LIMIT_BYTES // (total / n + 8))
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def launches():
    from cuvs_b200._capi import lib
    lib.cuvsB200KernelLaunches.restype = C.c_longlong
    return int(lib.cuvsB200KernelLaunches())


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from cuvs_b200._capi import lib
    from cuvs_b200.common import Resources
    lib.cuvsB200TimingTotalMs.restype = C.c_double

    kw = {}
    if args.n:
        kw["n"] = args.n
    if args.nq:
        kw["nq"] = args.nq
    if args.workload in ("ivf_pq", "ivf_pq_c2"):
        kw["lut_dtype"] = args.lut_dtype
        if args.data_rank:
            kw["data_rank"] = args.data_rank
        for name in ("n_lists", "n_probes", "refine_ratio", "pq_dim"):
            if getattr(args, name):
                kw[name] = getattr(args, name)
        kw["rank"], kw["world"] = rank, world
        kw["shard_rows"] = args.shard_rows
    if args.workload == "ivf_flat":
        for name in ("n_lists", "n_probes"):
            if getattr(args, name):
                kw[name] = getattr(args, name)
        kw["rank"], kw["world"] = rank, world
    if args.workload == "cagra":
        if args.itopk:
            kw["itopk"] = args.itopk
        if args.degree:
            kw["degree"] = args.degree
        kw["walk_bits"] = args.walk_bits
    res = Resources()
    if args.workload in ("ivf_pq", "ivf_pq_c2", "ivf_flat"):
        kw["resources"] = res
    wl = WORKLOADS[args.workload](**kw)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        total = 0.0
        for _ in range(steps):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn(res)
            res.sync()
            e.record()
            e.synchronize()
            total += s.elapsed_time(e)
        return total

    for _ in range(max(args.warmup, 3)):
        wl.step(res)
    res.sync()
    barrier()
    prof = os.environ.get("CUVS_B200_PROFILE") == "1"      # ncu --profile-from-start off: only the timed steps
    with ClockSampler(local) as clk:
        # the timed region is only tens of milliseconds: keep the GPU under the same load for ~1.5 s first so that the
        # nvidia-smi sampler (one query per ~0.25 s) sees clocks and throttle reasons UNDER LOAD, then time (still sampling)
        t_load = time.time()
        wl.step(res)
        res.sync()
        one = torch.tensor([time.time() - t_load], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(one, op=dist.ReduceOp.MAX)  # same iteration count on every rank (the step has a collective)
        n_load = 0 if prof else int(min(400, max(10, 1.5 / max(float(one[0]), 1e-4))))
        for _ in range(n_load):
            wl.step(res)
            res.sync()
        barrier()
        lib.cuvsB200TimingReset()   # kernel sections and launch counts cover the timed steps only
        lib.cuvsB200TimingEnable(1)
        l0 = launches()
        if prof:
            torch.cuda.profiler.start()
        ms = timed(wl.step, args.steps)
        if prof:
            torch.cuda.profiler.stop()
        n_launch = launches() - l0
        lib.cuvsB200TimingEnable(0)
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(wl.outputs(), args.dump_outputs)
    cnt = C.c_int(0)
    kernel_ms_total = lib.cuvsB200TimingTotalMs(wl.timing_section.encode(), C.byref(cnt))
    kernel_ms = kernel_ms_total / max(cnt.value, 1)
    ok = wl.check()

    # end-to-end: host queries in, host results out
    for _ in range(2):
        wl.e2e_step(res)
    res.sync()
    barrier()
    e2e_ms = timed(wl.e2e_step, args.steps)
    barrier()

    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])
    pk = peaks()
    if rank == 0:
        units = wl.units() * args.steps
        hb, db = wl.e2e_bytes()
        line = {
            "metric": METRIC_NAME, "value": units / (ms * 1e-3),
            "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": wl.dtype, "data": "synthetic", "config": wl.config(), "clocks": clk.summary(),
            "e2e": {"value": units / (e2e_ms * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": hb, "d2h_bytes_per_step": db,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": n_launch, "parity_spot_check": ok,
            "roofline": wl.roofline(kernel_ms, pk),
        }
        line["roofline"]["traffic"] = ncu_traffic(args.workload, wl)
        if not ok:
            line["PARITY_FAILED"] = ("recall@10 below 0.95 or ground-truth machinery disagrees with the oracle — this line is NOT "
                                     "a valid measurement of the metric")
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = wl.cpu_baseline()
        if world == 1 and args.workload == "ivf_pq" and not args.no_aux:
            del wl
            torch.cuda.empty_cache()
            line["config"]["harder_data"] = harder_data_point(args, res, timed)
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def harder_data_point(args, res, timed):
    """The same search on a HARDER distribution (rank-32 manifold: twice the intrinsic dimension, PQ with 2 dims per code has
    less to exploit), at 10M rows so that it fits beside the main run: QPS + recall, reported inside the main line's config."""
    wl = IvfPqWorkload(n=10_000_000, n_lists=4096, n_probes=192, refine_ratio=4, data_rank=32, lut_dtype=args.lut_dtype)
    for _ in range(3):
        wl.step(res)
    res.sync()
    ms = timed(wl.step, args.steps)
    ok = wl.check()
    return {"workload": wl.name, "data": "rank-32 gaussian manifold + 0.05 noise", "qps": wl.units() * args.steps / (ms * 1e-3),
            "recall_at_10": wl.recall, "ok": bool(ok)}


def run_reference(args):
    """Reference arm.  cuVS has no CPU implementation of these searches (only refine_host and hnswlib) and its CUDA build
    cannot be produced offline (DESIGN.md §2), so this times the oracle port — exact fp32 kNN, all host threads, in the
    pinned-thread subprocess of oracle/cpu_baseline.py — on the SAME tensors as our arm (same torch generator and seeds; on
    the device when there is one, then copied to the host): a row slice of the dataset (host RAM / time bound), the rate
    scaled to the full row count.  Each "step" is one timed repeat of the bounded query sample.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    d, nq, k = (96 if wl == "cagra" else 128), args.nq or 10_000, 10
    n = args.n or {"brute_force": 1_000_000, "ivf_pq": 100_000_000}.get(wl, 10_000_000)
    rows = min(n, CPU_SLICE_ROWS)
    if wl == "brute_force":
        g = torch.Generator(device=dev)
        g.manual_seed(99)
        centers = torch.randn((max(1, n // 1000), d), generator=g, device=dev)
        ds = gen_clustered(rows, d, 1234, centers, device=dev)
        qs = gen_clustered(1024, d, 1234 + 3087, centers, device=dev)
        name = BruteForceWorkload.name
    else:
        rk = args.data_rank or 16
        ds = gen_manifold(rows, d, 1234, rank=rk, device=dev)   # == the first `rows` rows of the GPU arm's dataset
        qs = gen_manifold(1024, d, 1234 + 3087, rank=rk, device=dev)
        name = f"{wl} {n // 1_000_000}M x {d} f32 workload, answered by exact CPU kNN (the reference has no CPU {wl} search)"
    budget = max(8.0, 12.0 * args.steps / 3.0)
    cb = cpu_exact_knn_rate(ds.cpu().numpy(), qs.cpu().numpy(), k, budget, "same tensors as the GPU arm", n_total=n,
                            repeats=args.steps)
    v = cb["value"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC_NAME, "value": v, "unit": "queries/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": args.steps, "warmup": 1, "ms_per_step": None, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": name, "n": n, "dim": d, "batch": nq, "k": k, "metric": "sqeuclidean", "recall_at_10": 1.0,
                   "note": "steps/warmup: the CPU arm runs 1 warm-up + --steps timed repeats of a bounded query sample (median reported)"},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ivf_pq", choices=sorted(WORKLOADS))
    ap.add_argument("--n", "--rows", dest="n", type=int, default=0,
                    help="dataset rows (under torchrun use --rows: torchrun's own parser rejects --n as an ambiguous abbreviation)")
    ap.add_argument("--nq", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--n-lists", dest="n_lists", type=int, default=0)
    ap.add_argument("--n-probes", dest="n_probes", type=int, default=0)
    ap.add_argument("--refine-ratio", dest="refine_ratio", type=int, default=0)
    ap.add_argument("--pq-dim", dest="pq_dim", type=int, default=0)
    ap.add_argument("--lut-dtype", dest="lut_dtype", default="f16", choices=["f32", "f16", "u8"],
                    help="ivf_pq search lut_dtype: f16/u8 (reduced-precision LUT, the usual throughput setting) -> 1-pass bf16 scan; f32 (API default) -> 2-pass scan")
    ap.add_argument("--walk-bits", dest="walk_bits", type=int, default=32, choices=[16, 32],
                    help="cagra: precision of the rows the graph walk reads (16 = fp16 copy + fp32 re-rank, 32 = fp32)")
    ap.add_argument("--data-rank", dest="data_rank", type=int, default=0, help="intrinsic dimension of the synthetic manifold data (default 16)")
    ap.add_argument("--no-shard-rows", dest="shard_rows", action="store_false",
                    help="ivf_pq, N > 1: keep the full fp32 dataset on every rank for the refine (default: every rank keeps only the rows "
                         "of the lists it owns — local ids + an id map — and drops the dataset after the ground truth is computed)")
    ap.add_argument("--shard-rows", dest="shard_rows", action="store_true", help="(default) see --no-shard-rows")
    ap.set_defaults(shard_rows=True)
    ap.add_argument("--no-aux", action="store_true", help="skip the secondary harder-data (rank-32, 10M) measurement of the ivf_pq line")
    ap.add_argument("--itopk", type=int, default=0)
    ap.add_argument("--degree", type=int, default=0)
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm only times the CPU search)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
