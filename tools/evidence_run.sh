#!/bin/bash
# One GPU box, final code of the round: GPU test log, bench line, ncu launch lists (bench + fit), ncu --set full captures of
# the hot kernels, sanitizer logs.  Everything lands in gpurun_out/ev_*; the summaries are copied into profiles/ by hand.
#   gpurun --timeout 1500 -- 'bash tools/evidence_run.sh'
set -u
O=gpurun_out
python -m pytest tests -m gpu -x -q > $O/ev_gpu_tests.log 2>&1; tail -2 $O/ev_gpu_tests.log
python bench.py > $O/ev_bench.json 2> $O/ev_bench.err; tail -c 200 $O/ev_bench.json; echo
B="python bench.py --steps 2 --warmup 3 --no-fit --no-cpu-baseline"
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/ev_launches.csv $B > $O/ev_launches.log 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/ev_fit_launches.csv python tools/fit_bench.py 1000000 0 1 > $O/ev_fit_launches.log 2>&1
ncu --set full --clock-control none --import-source on -k 'regex:k_p2l_grid|k_p2p_sym|k_m2l_stream|k_p2m_t|k_l2p_t' -s 10 -c 5 -f -o $O/ev_full \
    python bench.py --steps 1 --warmup 3 --no-fit --no-cpu-baseline > $O/ev_full.log 2>&1
ncu --set full --clock-control none --import-source on -k 'regex:k_dom_solve|k_cholesky|k_tri_gemv' -s 6 -c 8 -f -o $O/ev_solver \
    python tools/fit_bench.py 1000000 0 1 > $O/ev_solver.log 2>&1
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 9 python tools/sanitize_smoke.py > $O/ev_memcheck.log 2>&1; echo "memcheck rc=$?" >> $O/ev_memcheck.log
timeout 900 compute-sanitizer --tool racecheck --racecheck-report all --error-exitcode 9 python tools/sanitize_smoke.py > $O/ev_racecheck.log 2>&1; echo "racecheck rc=$?" >> $O/ev_racecheck.log
tail -3 $O/ev_memcheck.log $O/ev_racecheck.log
ls -la $O/ev_*
