#!/bin/bash
# Round-2 acceptance run on one B200 (under gpurun): the whole -m gpu suite, the default bench
# line (with CPU arms), and one bench line per BASELINE config -> gpurun_out/<tag>_*.json
mkdir -p gpurun_out
tag=${1:-r2cfg}
log=gpurun_out/${tag}.log
: > $log
step() { echo "== $1" >> $log; shift; timeout "$@" >> $log 2>&1; rc=$?; if [ $rc -ne 0 ]; then echo "STEP FAILED rc=$rc" >> $log; tail -60 $log; exit 1; fi; }
if [ -z "$SKIP_TESTS" ]; then step "pytest -m gpu" 900 python -m pytest tests -x -q -m gpu; fi
if [ -z "$SKIP_DEFAULT" ]; then
echo "== bench default (C2)" >> $log
timeout 400 python bench.py > gpurun_out/${tag}_C2.json 2> gpurun_out/${tag}_C2.err || { echo FAILED >> $log; tail -5 gpurun_out/${tag}_C2.err >> $log; }
fi
for c in ${CFGS:-C1 C3 C4 C5}; do
  echo "== bench $c" >> $log
  timeout 500 python bench.py --config $c --steps 5 --warmup 3 ${CFG_ARGS:---cpu-seconds 4} > gpurun_out/${tag}_$c.json 2> gpurun_out/${tag}_$c.err || { echo FAILED >> $log; tail -5 gpurun_out/${tag}_$c.err >> $log; }
done
python - >> $log <<'PY'
import json, glob, os
tag = os.environ.get("TAG", "")
for f in sorted(glob.glob("gpurun_out/*_C?.json")):
    try:
        d = json.loads([l for l in open(f) if l.startswith("{")][-1])
    except Exception as e:
        print(f, "no line", e); continue
    cb = d.get("cpu_baseline") or {}
    print(os.path.basename(f), "| value", round(d["value"]), "| e2e", round(d["e2e"]["value"]), "| kernel_ms", round(d["roofline"]["kernel_ms"], 3),
          "| frac", round(d["roofline"]["frac"], 4), "| d2h", d["e2e"]["d2h_bytes_per_step"], "| cpu", round(cb.get("value", 0), 1),
          "eff", cb.get("cores_effective"), "heap", round((cb.get("optimised") or {}).get("value", 0), 1), "|", d["roofline"]["kernel"])
PY
tail -40 $log
