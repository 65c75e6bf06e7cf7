#!/bin/bash
# ncu evidence: launch list of one profiled run + full-set captures of selected kernels ($1 = regex, default all hot ones)
python -c "from opticalflowclustering_b200 import _build; _build.build()"
mkdir -p gpurun_out
rm -f gpurun_out/prof_*.ncu-rep
KREG='regex:prefilter|polyexp|flow_iter|flow_upsample|bgr2gray|flow_encode|grid_cells|minmax'
python tools/profile_step.py > gpurun_out/profile_plain.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -k "$KREG" -c 200 --csv --log-file gpurun_out/launches.csv python tools/profile_step.py > gpurun_out/ncu_list.log 2>&1
echo "list rc=$?"
for k in ${1:-flow_iter_tmem polyexp_strip prefilter_direct}; do
  # capture the launches of this kernel in the third (last) step of the script: skip 2/3 of them
  n=$(grep -c "$k" gpurun_out/launches.csv); s=$((n * 2 / 3)); c=$((n - s)); [ $c -gt 4 ] && c=4
  ncu --set full --clock-control none --import-source on -k regex:$k -s $s -c $c -o gpurun_out/prof_$k -f python tools/profile_step.py > gpurun_out/ncu_$k.log 2>&1; echo "$k rc=$? (skip $s, capture $c)"
done
ls -la gpurun_out | tail -8
