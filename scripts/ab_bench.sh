# same-box A/B of an environment knob: bash scripts/ab_bench.sh VAR "v1 v2 ..." [bench args]
mkdir -p gpurun_out
USAGE='usage: bash scripts/ab_bench.sh VAR "v1 v2 ..." [bench args]'
VAR=${1:?$USAGE}; VALS=${2:?$USAGE}; shift 2
for rep in 1 2; do
for v in $VALS; do
  env $VAR=$v timeout 100 python bench.py --no-cpu-baseline --steps 100 --warmup 5 "$@" 2>/dev/null | tail -1 > gpurun_out/ab_$v.json
  python - <<PY
import json
d=json.loads(open("gpurun_out/ab_$v.json").read())
print("$VAR=$v", round(d["value"]), round(d["ms_per_step"]*1000,1), "e2e", round(d["e2e"]["value"]), d["clocks"]["sm_mhz"], {k["kernel"][:6]:round(k["ms"]*1000,1) for k in d["kernels"]})
PY
done
done
