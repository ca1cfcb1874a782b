#!/bin/bash
# A/B of the WORLD analysis kernels and of bench.py between two builds of libryk kept side by side in csrc/:
#   tools/gpu_d4c_ab.sh OUT_DIR BASE_LIB NEW_LIB [NEW_TIMELINE_LIB] [BASE_TIMELINE_LIB]
# (a *_TIMELINE_LIB is built with RYK_NVCC_EXTRA=-DRYK_D4C_TIMELINE).  Writes everything under OUT_DIR (relative to the repository root).
set -u
cd "$(dirname "$0")/.."
C=realtime_yukarin_b200/csrc
O=$1; shift; mkdir -p $O
BASE=$C/$1; NEW=$C/$2
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/gpu.txt
for tag in base new; do
  lib=$BASE; [ $tag = new ] && lib=$NEW
  RYK_LIB=$lib timeout 600 python tools/gpu_bench_analysis.py --reps 300 --json $O/standalone_$tag.json --dump $O/outputs_$tag.npz 2>$O/standalone_$tag.err | tail -1
done
python tools/gpu_bench_analysis.py --compare $O/outputs_base.npz $O/outputs_new.npz | tee $O/outputs_compare.json
for i in 3 4; do
  if [ $# -ge $i ]; then
    f=$O/timeline_$i.txt; rm -f $f
    RYK_LIB=$C/${!i} RYK_D4C_TIMELINE_FILE=$f timeout 600 python tools/gpu_bench_analysis.py --timeline-runs 20 2>$O/timeline_$i.err
    echo "== timeline ${!i}"; python tools/gpu_bench_analysis.py --timeline-summary $f | tee $O/timeline_${!i}.summary.txt
  fi
done
for r in 1 2 3; do
  for tag in base new; do
    lib=$BASE; [ $tag = new ] && lib=$NEW
    RYK_LIB=$lib timeout 600 python bench.py --gpus 1 --steps 100 --no-extra --dump-outputs $O/wave_$tag 2>$O/bench_${tag}_$r.err | tail -1 > $O/bench_${tag}_$r.json
    python -c "import json,sys; d=json.load(open('$O/bench_${tag}_$r.json')); print('$tag run $r', round(d['value'],1), 'sustained', d.get('sustained',{}).get('value'), 'in-kernel ms', d['roofline']['ms_per_step_in_kernel'])"
  done
done
python -c "
import numpy as np, glob
for f in sorted(glob.glob('$O/wave_base/*.npy')):
    a = np.load(f); b = np.load(f.replace('wave_base', 'wave_new'))
    print(f.split('/')[-1], 'max |diff| / peak', float(np.max(np.abs(a - b)) / max(np.max(np.abs(a)), 1e-30)))
" | tee $O/wave_compare.txt
