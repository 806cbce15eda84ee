#!/bin/bash
# One parametrised GPU runner (replaces the per-experiment scripts of round 1):  scripts/gpu_stage.sh STAGE...
# Every stage writes its log under gpurun_out/ (merged back by gpurun); stages never abort the following ones.
mkdir -p gpurun_out
for stage in "$@"; do
  case "$stage" in
    pq_tests)   timeout 900 python -m pytest tests/test_ivf_pq_gpu.py -q > gpurun_out/pq_tests.log 2>&1; echo "pq_tests rc=$?" ;;
    all_tests)  timeout 1700 python -m pytest tests -m gpu -q > gpurun_out/all_tests.log 2>&1; echo "all_tests rc=$?" ;;
    c2)         timeout 600 python bench.py --workload ivf_pq_c2 --steps 10 --no-cpu --no-aux > gpurun_out/bench_c2.log 2>&1; echo "c2 rc=$?" ;;
    sweep100m)  timeout 900 python scripts/sweep_probes.py 100000000 16384 "32,40,48,56,64" > gpurun_out/sweep100m.log 2>&1; echo "sweep rc=$?" ;;
    bench)      timeout 1500 python bench.py > gpurun_out/bench_default.log 2>&1; echo "bench rc=$?" ;;
    onec2)      timeout 600 python scripts/sweep_probes.py 10000000 1024 "64" > gpurun_out/onec2.log 2>&1; echo "onec2 rc=$?" ;;
    one100m)    timeout 900 python scripts/sweep_probes.py 100000000 16384 "48" > gpurun_out/one100m.log 2>&1; echo "one100m rc=$?" ;;
    prof100m)   CUVS_B200_PROFILE=1 timeout 1200 ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:pq_stream_scan -c 1 -f -o gpurun_out/r02_pq100m python scripts/sweep_probes.py 100000000 16384 "48" > gpurun_out/prof100m.log 2>&1; echo "prof100m rc=$?" ;;
    launches100m) CUVS_B200_PROFILE=1 timeout 1200 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/r02_launches100m.csv python scripts/sweep_probes.py 100000000 16384 "48" > gpurun_out/launches100m.log 2>&1; echo "launches100m rc=$?" ;;
    profc2)     CUVS_B200_PROFILE=1 timeout 900 ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:pq_stream_scan -c 1 -f -o gpurun_out/r02_pqc2 python scripts/sweep_probes.py 10000000 1024 "64" > gpurun_out/profc2.log 2>&1; echo "profc2 rc=$?" ;;
    bf)         timeout 600 python bench.py --workload brute_force --steps 10 > gpurun_out/bench_bf.log 2>&1; echo "bf rc=$?" ;;
    c2cpu)      timeout 600 python bench.py --workload ivf_pq_c2 --steps 10 --no-aux > gpurun_out/bench_c2.log 2>&1; echo "c2cpu rc=$?" ;;
    cagra)      timeout 900 python bench.py --workload cagra --steps 10 --no-cpu > gpurun_out/bench_cagra.log 2>&1; echo "cagra rc=$?" ;;
    flat)       timeout 900 python bench.py --workload ivf_flat --steps 10 --no-cpu > gpurun_out/bench_flat.log 2>&1; echo "flat rc=$?" ;;
    profcagra)  CUVS_B200_PROFILE=1 timeout 900 ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:cagra_search -c 1 -f -o gpurun_out/r02_cagra python bench.py --workload cagra --steps 1 --no-cpu > gpurun_out/profcagra.log 2>&1; echo "profcagra rc=$?" ;;
    profc2tc)   CUVS_B200_PROFILE=1 timeout 900 ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:tc_scan_kernel -c 2 -f -o gpurun_out/r02_c2 python bench.py --workload ivf_pq_c2 --steps 1 --no-cpu --no-aux > gpurun_out/profc2tc.log 2>&1; echo "profc2tc rc=$?" ;;
    launchesc2) CUVS_B200_PROFILE=1 timeout 900 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/r02_launchesc2.csv python bench.py --workload ivf_pq_c2 --steps 1 --no-cpu --no-aux > gpurun_out/launchesc2.log 2>&1; echo "launchesc2 rc=$?" ;;
    cagra_tests) timeout 600 python -m pytest tests/test_cagra_gpu.py -q > gpurun_out/cagra_tests.log 2>&1; echo "cagra_tests rc=$?" ;;
    profselect) CUVS_B200_PROFILE=1 timeout 900 ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:select_k_reg -c 1 -f -o gpurun_out/r02_selectk python scripts/sweep_probes.py 100000000 16384 "48" > gpurun_out/profselect.log 2>&1; echo "profselect rc=$?" ;;
    benchq)     timeout 900 python bench.py --no-cpu --no-aux > gpurun_out/bench_quick.log 2>&1; echo "benchq rc=$?" ;;
    mgtests)    timeout 600 python -m pytest tests/test_mg_gpu.py tests/test_distributed_nccl.py -q > gpurun_out/mg_tests.log 2>&1; echo "mgtests rc=$?" ;;
    bench2)     timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus 2 --steps 5 --warmup 3 --rows 20000000 --n-lists 4096 --no-aux > gpurun_out/bench_n2.log 2>&1; echo "bench2 rc=$?" ;;
    fusedtest)  timeout 600 python -m pytest tests/test_ivf_flat_gpu.py -q -k "fused or matches_oracle" > gpurun_out/fused_tests.log 2>&1; echo "fusedtest rc=$?" ;;
    smoke)      timeout 600 python __graft_entry__.py smoke > gpurun_out/smoke.log 2>&1; echo "smoke rc=$?" ;;
    *)          echo "unknown stage $stage" ;;
  esac
done
tail -n 5 gpurun_out/*.log
