#!/bin/bash
# One parametrised GPU-box runner (use through gpurun):  scripts/gpu_run.sh <tag> <task> [args...]
#   tests [pytest args]     GPU test suite (default: everything marked gpu)
#   bench [bench args]      one bench.py run, JSON line -> gpurun_out/<tag>_bench.json
#   ops   [bench args]      per-op device-time table of one step program -> gpurun_out/<tag>_per_op_us.txt
#   launches [bench args]   ncu launch list (time + DRAM bytes) of a short bench -> gpurun_out/<tag>_launches.csv
#   probe                   isolated GEMM timings + numeric checks (tests/gpu_trace_gemm.py)
#   py <script> [args]      any python script
#   full <kernel-regex> [skip] [count]   one `ncu --set full` capture -> gpurun_out/<tag>_<...>.ncu-rep
# Several tasks can be chained with "--":  gpu_run.sh r2 tests -- bench --steps 2
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
TAG=$1; shift
run_task() {
  local task=$1; shift
  case "$task" in
    tests)
      if [ $# -eq 0 ]; then set -- tests/; fi
      timeout 1500 python -m pytest "$@" -q -m gpu --timeout 300 -p no:cacheprovider -rA > gpurun_out/${TAG}_tests.log 2>&1
      grep -E "^(PASSED|FAILED|ERROR)|passed|failed|error" gpurun_out/${TAG}_tests.log | grep -v "^PASSED" | tail -40 ;;
    bench)
      timeout 900 python bench.py "$@" > gpurun_out/${TAG}_bench.json 2> gpurun_out/${TAG}_bench.err
      tail -c 1500 gpurun_out/${TAG}_bench.err; cat gpurun_out/${TAG}_bench.json ;;
    benchn)           # benchn <name> [bench args]: like bench, output in gpurun_out/<tag>_bench_<name>.json
      local nm=$1; shift
      timeout 900 python bench.py "$@" > gpurun_out/${TAG}_bench_${nm}.json 2> gpurun_out/${TAG}_bench_${nm}.err
      tail -c 600 gpurun_out/${TAG}_bench_${nm}.err; cut -c1-420 gpurun_out/${TAG}_bench_${nm}.json ;;
    ops)
      timeout 600 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --profile-ops "$@" 2> gpurun_out/${TAG}_per_op_us.txt | cut -c1-300
      tail -n +1 gpurun_out/${TAG}_per_op_us.txt | head -150 ;;
    launches)
      timeout 900 ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none \
        -c 2000 --csv --log-file gpurun_out/${TAG}_launches.csv python bench.py --steps 1 --warmup 1 --timesteps 3 \
        --no-cpu-baseline --no-e2e "$@" > gpurun_out/${TAG}_launches.log 2>&1
      tail -3 gpurun_out/${TAG}_launches.log | cut -c1-300; wc -l gpurun_out/${TAG}_launches.csv ;;
    full)
      local k=$1; local skip=${2:-60}; local cnt=${3:-3}
      timeout 900 ncu --set full --clock-control none --import-source on -k regex:$k -s $skip -c $cnt \
        -o gpurun_out/${TAG}_$(echo $k | tr -c 'a-zA-Z0-9\n' _)_full -f python bench.py --steps 1 --warmup 1 --timesteps 2 \
        --no-cpu-baseline --no-e2e > gpurun_out/${TAG}_full.log 2>&1
      tail -2 gpurun_out/${TAG}_full.log | cut -c1-300; ls -la gpurun_out/${TAG}_*.ncu-rep ;;
    probe)
      GNT_ONLY=1 timeout 600 python tests/gpu_trace_gemm.py 2>&1 | tee gpurun_out/${TAG}_gemm_probe.txt | grep -v "^   prod_wait" | tail -60 ;;
    train-launches)   # per-kernel device time of one training iteration (ncu launch list)
      timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 6000 --csv --log-file gpurun_out/${TAG}_train_launches.csv \
        python bench.py --config train --steps 1 --warmup 1 "$@" > gpurun_out/${TAG}_train_launches.log 2>&1
      python scripts/summarize_launches.py gpurun_out/${TAG}_train_launches.csv | tee gpurun_out/${TAG}_train_kernels.txt ;;
    dp2)              # needs gpurun --gpus 2: data-parallel training check + 2-GPU bench lines
      timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tests/gpu_dp_train_check.py 2>&1 | tail -8 | tee gpurun_out/${TAG}_dp2_check.log
      timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \
        bench.py --gpus 2 --config train --steps 5 --warmup 3 2>gpurun_out/${TAG}_dp2_train.err | tail -1 | tee gpurun_out/${TAG}_dp2_train.json
      timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 \
        bench.py --gpus 2 --steps 2 --warmup 2 --no-cpu-baseline "$@" 2>gpurun_out/${TAG}_dp2_sample.err | tail -1 | tee gpurun_out/${TAG}_dp2_sample.json ;;
    py)
      timeout 900 python "$@" 2>&1 | tail -40 | tee gpurun_out/${TAG}_py.log ;;
    *) echo "unknown task $task"; return 2 ;;
  esac
}
args=()
for a in "$@"; do
  if [ "$a" == "--" ]; then run_task "${args[@]}"; args=(); else args+=("$a"); fi
done
[ ${#args[@]} -gt 0 ] && run_task "${args[@]}"
echo "gpu_run done"
