#!/bin/bash
# Round-2 acceptance on one B200: whole -m gpu suite, smoke(), the
# default bench line, the ncu launch list of the same command and one `ncu --set full` capture.
mkdir -p gpurun_out
tag=${1:-r2final}
log=gpurun_out/${tag}.log
: > $log
step() { echo "== $1" >> $log; shift; timeout "$@" >> $log 2>&1; rc=$?; if [ $rc -ne 0 ]; then echo "STEP FAILED rc=$rc" >> $log; fi; }
step "pytest -m gpu" 600 python -m pytest tests -q -m gpu
step "smoke" 120 python __graft_entry__.py smoke
echo "== default bench" >> $log
timeout 400 python bench.py > gpurun_out/${tag}_bench.json 2> gpurun_out/${tag}_bench.err; tail -c 400 gpurun_out/${tag}_bench.json >> $log
echo "== reference arm" >> $log
timeout 200 python bench.py --impl reference --steps 3 --warmup 1 > gpurun_out/${tag}_reference.json 2>> $log
step "ncu launch list" 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/${tag}_launches.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-e2e-variants
step "ncu full" 400 ncu --set full --clock-control none --import-source on -k regex:spf_quad_kernel -s 3 -c 1 -f -o gpurun_out/${tag}_full \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-e2e-variants
grep -v "^==PROF\|^==WARN\|^{" $log | tail -40
