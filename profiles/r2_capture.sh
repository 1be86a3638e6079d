#!/bin/bash
# round-2 evidence run: GPU tests, the bench line timed as in round 2 (500 steps in 25 windows of 20: 1024 settle +
# 5 warm-up + 500 timed launches, which the skip/count values below assume), then (each only after its command ran
# clean without ncu) the launch list of the bench and one full capture of a steady single-step launch
cd "$(dirname "$0")/.."
OUT="${OUT:-profiles/_capture}"   # where the evidence files go
mkdir -p "$OUT"
python -m pytest tests -m gpu -q 2>&1 | tail -4
python bench.py --steps 500 --windows 25 --warmup 5 > $OUT/r2c_bench.json 2> $OUT/r2c_bench.err || { tail -5 $OUT/r2c_bench.err; exit 1; }
python bench.py --no-legs --steps 500 --windows 25 --warmup 5 --e2e-steps 0 > /dev/null 2>&1 || exit 1
ncu --metrics gpu__time_duration.sum --clock-control none --launch-skip 1024 -c 560 --csv --log-file $OUT/r2c_ncu_launches.csv \
    python bench.py --no-legs --steps 500 --windows 25 --warmup 5 --e2e-steps 0 > $OUT/r2c_ncu.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:macm_step_kernel --launch-skip 1100 -c 1 -f -o $OUT/r2c_steady \
    python bench.py --no-legs --steps 500 --windows 25 --warmup 5 --e2e-steps 0 >> $OUT/r2c_ncu.log 2>&1
ls -la "$OUT" | tail -5
