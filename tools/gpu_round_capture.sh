# Final capture of a round (one GPU job): GPU tests, bench line, reference arm, ncu launch list of the bench, full ncu
# captures of the forward kernels, compute-sanitizer.  Tag = $1 (default r02), output directory = $2 (default build/capture,
# git-ignored).  Run from the repo root of the snapshot.
set -x
T=${1:-r02}
OUT=${2:-build/capture}
cd $GRAFT_REPO_ROOT
export DSAC_SKIP_BUILD=1
mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.max.sm,clocks.sm --format=csv,noheader; nproc
timeout 1500 python -m pytest tests -m gpu -q -s --timeout=900 -rf > $OUT/${T}_pytest.log 2>&1; tail -3 $OUT/${T}_pytest.log
timeout 900 python bench.py --steps 10 --warmup 3 > $OUT/${T}_bench_line.json 2> $OUT/${T}_bench.err; tail -c 600 $OUT/${T}_bench_line.json; tail -3 $OUT/${T}_bench.err
timeout 300 python bench.py --impl reference --steps 3 --warmup 1 > $OUT/${T}_bench_reference.json 2>> $OUT/${T}_bench.err; tail -c 300 $OUT/${T}_bench_reference.json
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $OUT/launches_${T}.csv python bench.py --steps 2 --warmup 3 > $OUT/${T}_ncu_bench.log 2>&1
# full captures: the steady-state pass is the second one; the number of launches of each kernel in one pass (it depends on
# the round / portion schedule) is counted from a one-pass launch list, and -s skips exactly the first pass
REPS=1 timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/${T}_onepass.csv python tools/prof_driver.py > /dev/null 2>&1
for k in k1_filter k1_slot k1_solve k_score k_refine; do
  skip=$(grep -c "[ :\"]$k[<(]" $OUT/${T}_onepass.csv); echo "$k: $skip launches per pass"
  REPS=2 timeout 400 ncu --set full --clock-control none --import-source on -k regex:$k -c 1 -s $skip -f -o $OUT/${k}_${T} python tools/prof_driver.py > $OUT/ncu_$k.log 2>&1; tail -1 $OUT/ncu_$k.log
done
timeout 300 ncu --set full --clock-control none --import-source on -k regex:k_gather -c 1 -s 2 -f -o $OUT/k_gather_${T} python tools/gather_probe.py > $OUT/ncu_k_gather.log 2>&1; tail -1 $OUT/ncu_k_gather.log
timeout 200 python tools/gather_probe.py 2>&1 | tail -2 > $OUT/${T}_gather_probe.txt; cat $OUT/${T}_gather_probe.txt
timeout 300 python tools/sampler_breakdown.py 2>&1 | grep "^n=" > $OUT/${T}_sampler_breakdown.txt; cat $OUT/${T}_sampler_breakdown.txt
NB=1 timeout 100 python tools/slot_phases.py 2>&1 | grep "slot thread-0" > $OUT/${T}_slot_phases.txt; NB=1024 timeout 100 python tools/slot_phases.py 2>&1 | grep "slot thread-0" >> $OUT/${T}_slot_phases.txt; cat $OUT/${T}_slot_phases.txt
for tool in memcheck racecheck initcheck; do NB=5 REPS=1 timeout 400 compute-sanitizer --tool $tool python tools/prof_driver.py 2>&1 | grep -E "ERROR SUMMARY|RACECHECK SUMMARY" | sed "s/^/$tool fwd (5 frames): /"; done > $OUT/sanitizer_${T}.txt 2>&1
timeout 300 compute-sanitizer --tool memcheck python -m pytest tests/test_gpu_upstream.py -m gpu -q 2>&1 | grep -E "ERROR SUMMARY|passed|failed" | sed "s/^/memcheck upstream (k_gather_patches TMA store, k_coords_from_prediction): /" >> $OUT/sanitizer_${T}.txt
timeout 400 compute-sanitizer --tool memcheck python -m pytest tests/test_gpu_backward.py -m gpu -q -k "test_backward_matches_oracle or (dsac_variant_backward_matches_oracle and 16)" 2>&1 | grep -E "ERROR SUMMARY|passed|failed" | sed "s/^/memcheck backward + backward_dsac: /" >> $OUT/sanitizer_${T}.txt
cat $OUT/sanitizer_${T}.txt
ls -la $OUT | tail -15
