#!/bin/bash
# Development: the 1-GPU evidence run of a round in one gpurun call -- GPU tests, both bench arms, the ncu launch list of the
# bench command, one `ncu --set full` capture of the backward and the forward, the config table, the map-shape table, the
# sanitizer passes.  Results under gpurun_out/r2/ with the suffix TAG.  (A number printed under ncu is never a bench value.)
cd "$(dirname "$0")/.."
O=gpurun_out/r2; mkdir -p $O; TAG=${TAG:-_final2}
STEPS=${STEPS:-"pytest bench launches ncu tables sanitize"}
for s in $STEPS; do
  case $s in
    pytest) timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -3 | tee $O/pytest$TAG.log ;;
    bench)  timeout 600 python bench.py 2>$O/bench$TAG.err | tail -1 | tee $O/bench$TAG.json | cut -c1-600
            timeout 600 python bench.py --impl reference --steps 20 --warmup 5 2>>$O/bench$TAG.err | tail -1 | tee $O/bench_reference$TAG.json | cut -c1-300 ;;
    launches) timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/launches_bench$TAG.csv \
                python bench.py --steps 2 --warmup 3 --no-cpu-baseline > $O/bench_under_ncu$TAG.log 2>&1 ;;
    ncu)    PROF_N=16 timeout 600 ncu --set full --clock-control none --import-source on -k regex:bwd_tma -c 1 -f -o $O/prof_bwd$TAG python tools/prof_driver.py 2>&1 | tail -1
            PROF_N=16 timeout 600 ncu --set full --clock-control none --import-source on -k regex:fwd_tma -c 1 -f -o $O/prof_fwd$TAG python tools/prof_driver.py 2>&1 | tail -1 ;;
    tables) timeout 600 python tools/config_table.py 2>&1 | tee $O/config_table$TAG.log | tail -30
            timeout 200 python tools/map_bench.py 2>&1 | tee $O/map_bench$TAG.log ;;
    sanitize)
            for tool in memcheck synccheck; do echo "== $tool"; timeout 900 compute-sanitizer --tool $tool python tools/sanitize_case.py 2>&1 | grep -E "ERROR SUMMARY|COMPUTE-SANITIZER|Error|hazard" | head -5; done | tee $O/sanitizer$TAG.log
            if ls pwstablenet_b200/var/libpwswarp_atomic.so.xz >/dev/null 2>&1; then
              mkdir -p /tmp/pwsvar; xz -d -k -c pwstablenet_b200/var/libpwswarp_atomic.so.xz > /tmp/pwsvar/libpwswarp_atomic.so
              echo "== racecheck (atomic progress build)" | tee -a $O/sanitizer$TAG.log
              PWS_LIB_PATH=/tmp/pwsvar/libpwswarp_atomic.so timeout 1200 compute-sanitizer --tool racecheck python tools/sanitize_case.py 2>&1 | grep -E "RACECHECK SUMMARY|Error|hazard" | head -5 | tee -a $O/sanitizer$TAG.log
            fi ;;
  esac
done
