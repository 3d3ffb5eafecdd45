#!/bin/bash
# Round-2 GPU visit: parity tests, parity report, driver-shaped bench (both arms), ncu launch list and full captures.
#   gpurun --timeout 2400 -- 'bash scripts/gpu_round2.sh <tag> "test report bench list ncu"'
# (compute-sanitizer is closed on this pool: profiles/r2_compute_sanitizer_closed.txt; scripts/sanitize_small.py is its driver)
tag=${1:-r2}
parts=${2:-"test report bench"}
has() { [[ " $parts " == *" $1 "* ]]; }
out=gpurun_out
mkdir -p $out
if has test; then
  timeout 900 python -m pytest tests -m gpu -q > $out/${tag}_pytest.log 2>&1; echo "pytest rc=$?" | tee -a $out/${tag}_pytest.log
  tail -4 $out/${tag}_pytest.log
fi
if has report; then
  timeout 600 python scripts/parity_report.py > $out/${tag}_parity_report.txt 2> $out/${tag}_parity_report.err; echo "report rc=$?"
  tail -2 $out/${tag}_parity_report.txt
fi
if has bench; then
  nvidia-smi --query-gpu=index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active --format=csv -lms 500 > $out/${tag}_clocks.csv &
  smi=$!
  timeout 900 python bench.py --steps 20 --warmup 5 > $out/${tag}_bench.json 2> $out/${tag}_bench.err; echo "bench rc=$?"
  tail -3 $out/${tag}_bench.err
  timeout 600 python bench.py --impl reference --steps 20 --warmup 5 > $out/${tag}_bench_ref.json 2> $out/${tag}_bench_ref.err; echo "ref rc=$?"
  timeout 900 python bench.py --steps 4000 --warmup 100 --skip-configs --skip-cpu --skip-hbm > $out/${tag}_bench_1000.json 2> $out/${tag}_bench_1000.err; echo "bench1000 rc=$?"
  kill $smi
fi
if has list; then   # launch list of the bench command's TIMED REGION (cudaProfilerStart/Stop around it; same command line otherwise)
  timeout 300 python bench.py --steps 20 --warmup 5 --skip-cpu --skip-hbm --skip-configs > $out/${tag}_plain.log 2>&1 &&
  timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off -c 400 --csv --log-file $out/${tag}_launches.csv \
      python bench.py --steps 20 --warmup 5 --skip-cpu --skip-hbm --skip-configs --profile-region > $out/${tag}_ncu_list.log 2>&1
  echo "launch list rc=$?"
fi
if has ncu; then
  timeout 300 python scripts/profile_kernels.py --mode replay --launches 2 --replay-steps 20 > $out/${tag}_prof_plain.log 2>&1 &&
  timeout 600 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k 'regex:replay_tma_kernel<double' -s 1 -c 1 -f -o $out/${tag}_replay20 \
      python scripts/profile_kernels.py --mode replay --launches 2 --replay-steps 20 > $out/${tag}_ncu_replay.log 2>&1
  echo "ncu replay rc=$?"
  timeout 300 python scripts/profile_rollout.py --scenario bus-stop --envs 131072 --launches 3 > $out/${tag}_roll_plain.log 2>&1 &&
  timeout 600 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k 'regex:rollout_kernel<double' -s 2 -c 1 -f -o $out/${tag}_busstop \
      python scripts/profile_rollout.py --scenario bus-stop --envs 131072 --launches 3 > $out/${tag}_ncu_roll.log 2>&1
  echo "ncu rollout rc=$?"
  timeout 300 python scripts/bench_dense.py --envs 20000 --steps 3 --chunk 10 --warm 40 > $out/${tag}_dense_plain.log 2>&1 &&
  timeout 600 ncu --set full --clock-control none --import-source on --kernel-name-base demangled -k 'regex:dense_kernel<double' -s 6 -c 1 -f -o $out/${tag}_dense \
      python scripts/bench_dense.py --envs 20000 --steps 3 --chunk 10 --warm 40 > $out/${tag}_ncu_dense.log 2>&1
  echo "ncu dense rc=$?"
fi
exit 0
