# Round-end evidence (run under gpurun, one GPU).  Only CSV summaries are kept (gpurun_out is capped at 64 MiB).
#   $1 = tag; FULL=1 also captures `--set full` for every kernel of one pipelined step (several minutes).
TAG=${1:-r01d}
ncu --metrics gpu__time_duration.sum --clock-control none -c 1200 --csv --log-file gpurun_out/${TAG}_launches.csv python bench.py --steps 4 --warmup 3 > gpurun_out/${TAG}_launches_bench.log 2>&1
python tools/launch_summary.py gpurun_out/${TAG}_launches.csv 88 4 > gpurun_out/${TAG}_launches_summary.txt 2>&1
if [ "$FULL" = "1" ]; then
  ncu --set full --clock-control none -s 720 -c 100 -f -o /tmp/${TAG}_full python bench.py --steps 4 --warmup 3 > gpurun_out/${TAG}_full_bench.log 2>&1
  python tools/ncu_summary.py /tmp/${TAG}_full.ncu-rep gpurun_out/${TAG}_ncu_full_one_step.csv
fi
