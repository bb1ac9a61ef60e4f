#!/bin/bash
# On the GPU box: bench each variants/libse_NAME.so in turn (same box, same clocks) and print the GEMM kernel times.
# NAME "cur" = the library already in the package directory.
cd "$(dirname "$0")/.."
for v in "$@"; do
  if [ "$v" != cur ]; then cp variants/libse_$v.so speech_enhancement_mi_b200/libse_b200.so; fi
  timeout 200 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-extras --no-e2e > gpurun_out/vb_$v.json 2> gpurun_out/vb_$v.err
  python - "$v" <<'PY'
import json, sys
v = sys.argv[1]
try:
    d = json.loads(open(f"gpurun_out/vb_{v}.json").read().strip().splitlines()[-1])
    k = {x["name"]: round(x["ms"] * 1000, 1) for x in d["kernels"]}
    names = ["convlist.2.conv+elu+gate", "convlist.3.conv+elu", "convlist.3.gate1x1", "gru.l0.input_proj", "gru.l1.input_proj", "gru.fc+elu",
             "deconvlist.0.deconv+elu", "deconvlist.0.skip+gln+blend", "deconvlist.1.deconv+elu", "deconvlist.1.skip+gln+blend"]
    print(v, round(d["ms_per_step"], 3), [k.get(n) for n in names])
except Exception as e:
    print(v, "failed", e)
PY
done
