#!/bin/bash
# round-2 evidence run (one GPU): GPU tests, bench lines of every BASELINE config, ncu launch list, full captures
# usage (under gpurun): bash tools/r2_profile.sh [tag]      (SKIP_TESTS=1 / SKIP_CONFIGS=1 / SKIP_NCU=1 to shorten)
TAG=${1:-r2}
O=gpurun_out
mkdir -p $O
if [ -z "$SKIP_TESTS" ]; then
timeout 900 python -m pytest tests -m gpu -x -q > $O/${TAG}_tests.log 2>&1; echo "tests rc=$?"
tail -3 $O/${TAG}_tests.log
fi
timeout 600 python bench.py --steps 20 --warmup 3 > $O/${TAG}_bench.json 2> $O/${TAG}_bench.err; echo "bench rc=$?"
if [ -z "$SKIP_CONFIGS" ]; then
timeout 300 python bench.py --steps 10 --warmup 3 --mode injected --cpu-batch 0 --no-e2e > $O/${TAG}_bench_injected.json 2> $O/${TAG}_bench_injected.err; echo "injected rc=$?"
timeout 300 python bench.py --config hs_gae --steps 10 --warmup 3 > $O/${TAG}_bench_hs_gae.json 2> $O/${TAG}_bench_hs_gae.err; echo "hs_gae rc=$?"
timeout 400 python bench.py --config ant1m --steps 5 --warmup 2 > $O/${TAG}_bench_ant1m.json 2> $O/${TAG}_bench_ant1m.err; echo "ant1m rc=$?"
timeout 900 python bench.py --config sweep --steps 3 --warmup 1 > $O/${TAG}_bench_sweep.json 2> $O/${TAG}_bench_sweep.err; echo "sweep rc=$?"
fi
if [ -z "$SKIP_NCU" ]; then
NB="python bench.py --steps 2 --warmup 1 --cpu-batch 0 --no-e2e"
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $O/${TAG}_launches.csv $NB > $O/${TAG}_ncu_launch.log 2>&1; echo "launch list rc=$?"
# ens_mlp3_tc_kernel instances alternate: policy (merged actor+V+VC), dynamics (K1) -> two consecutive launches
timeout 900 ncu --set full --clock-control none --import-source on -k ens_mlp3_tc_kernel --launch-skip 40 -c 2 -o $O/${TAG}_tc -f $NB > $O/${TAG}_ncu_tc.log 2>&1; echo "ncu tc rc=$?"
for spec in "row:rollout_step_kernel:20" "polrows:policy_rows_kernel:20" "gae:gae_paths_strict_kernel:1"; do
  name=${spec%%:*}; rest=${spec#*:}; kern=${rest%%:*}; skip=${rest##*:}
  timeout 600 ncu --set full --clock-control none --import-source on -k $kern --launch-skip $skip -c 1 -o $O/${TAG}_${name} -f $NB > $O/${TAG}_ncu_${name}.log 2>&1; echo "ncu $name rc=$?"
done
fi
