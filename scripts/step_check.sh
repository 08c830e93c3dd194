#!/bin/bash
# Staged hardware validation of the coupling-step kernel; every stage in its own process under `timeout`.
mkdir -p gpurun_out
LOG=gpurun_out/step_check.log
: > $LOG
run() { echo "--- $*" >> $LOG; timeout 120 "$@" >> $LOG 2>&1; echo "rc=$?" >> $LOG; }
for s in t0 t1 t2 t3 t4 c0 c1 c2 c3 c4 c5 c6 c7 c8; do run python scripts/step_check.py $s; done
echo "=== pytest gpu" >> $LOG
timeout 900 python -m pytest tests -m gpu -q -x 2>&1 | tail -15 >> $LOG
echo "=== ncu step kernel" >> $LOG
timeout 600 ncu --set full --clock-control none --import-source on -k regex:rq_coupling_step -s 4 -c 1 -o gpurun_out/ncu_step_r2b -f python bench.py --steps 1 --warmup 1 --rows 262144 --no-cpu-baseline --no-spline-roofline --no-extras --no-parity-check 2>&1 | tail -2 >> $LOG
cat $LOG
