#!/bin/bash
# A/B of kernel switches on one B200: each line "NAME VAR=VAL ..." runs the short bench in a fresh process and prints
# pairs/s plus the per-kernel times.  Usage: bash tools/ab_flow.sh <tag> "base" "noshare OFC_TMEM_SHARE=0" ...
TAG=$1; shift
export PYTHONPATH=.
mkdir -p gpurun_out
for spec in "$@"; do
  name=${spec%% *}; envs=""
  # "name@expN ..." runs with build_variants/libofc_expN.so swapped in (the box's copy of the tree is scratch)
  if [[ "$name" == *@* ]]; then
    var=${name#*@}; name=${name%@*}
    [ -f opticalflowclustering_b200/libofc.so.orig ] || cp opticalflowclustering_b200/libofc.so opticalflowclustering_b200/libofc.so.orig
    cp build_variants/libofc_$var.so opticalflowclustering_b200/libofc.so
  elif [ -f opticalflowclustering_b200/libofc.so.orig ]; then
    cp opticalflowclustering_b200/libofc.so.orig opticalflowclustering_b200/libofc.so
  fi
  [[ "$spec" == *" "* ]] && envs=${spec#* }
  env $envs python bench.py --steps 10 --warmup 3 --no-extras --no-cpu-baseline ${OFC_AB_ARGS} > gpurun_out/${TAG}_ab_${name}.json 2> gpurun_out/${TAG}_ab_${name}.err
  python - "$name" gpurun_out/${TAG}_ab_${name}.json <<'PY'
import json, sys
try:
    d = json.loads(open(sys.argv[2]).read().strip().splitlines()[-1])
    k = d["kernels"]
    print(f"{sys.argv[1]:14s} {d['value']:8.1f} pairs/s  e2e {d['e2e']['value']:8.1f}  step {d['ms_per_step']:.3f} ms | " + "  ".join(f"{n.replace('flow_','')} {v['ms_per_step']:.3f}" for n, v in k.items()))
except Exception as e:
    print(sys.argv[1], "FAILED", e)
PY
done
