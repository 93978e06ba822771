#!/bin/bash
# development sweep (on a B200): cross-attention CTA cap under two lanes
# usage: tools/sweep_lanes.sh <tag> "<xa_ctas> ..."
tag=${1:-sweep}; shift
out=/tmp/sweep_lanes_$tag
mkdir -p $out
for xa in ${@:-"96 148 128 112"}; do
  SW_XA_CTAS=$xa python bench.py --steps 2 --warmup 2 --no-cpu-baseline > $out/${tag}_x${xa}.json 2> $out/${tag}_x${xa}.err
  python - <<PY
import json
try:
    d = json.load(open("$out/${tag}_x${xa}.json"))
    print("xa_ctas $xa: value %.1f ms/step %.1f decode_ms %.1f enc_ms %.1f xattn_frac %.3f dec_frac %.3f parity %d/%d" % (
        d["value"], d["ms_per_step"], d["stages"]["device_ms_per_step"]["decode"], d["stages"]["device_ms_per_step"]["encode"],
        d["roofline"]["frac"], d["stages"]["decode_frac_of_hbm"], d["parity_check"]["token_identical_to_expected"], d["parity_check"]["windows"]))
except Exception as e:
    print("xa_ctas $xa failed", e)
PY
done
