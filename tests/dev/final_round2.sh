#!/bin/bash
# Final verification of the round on one B200 box: full GPU test suite, smoke, the bench line and the reference arm,
# the bench launch list, and `ncu --set full` captures of the kernels that changed (axis column passes, MDFT).
cd "$(dirname "$0")/../.."
mkdir -p gpurun_out
O=gpurun_out
( timeout 1500 python -m pytest tests -m gpu -x -q > $O/final_pytest.log 2>&1; echo "pytest rc=$?" >> $O/final_pytest.log )
( timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/final_smoke.log 2>&1; echo "smoke rc=$?" >> $O/final_smoke.log )
( timeout 600 python bench.py --steps 20 --warmup 3 > $O/final_bench_1gpu.json 2> $O/final_bench_1gpu.err; echo "bench rc=$?" >> $O/final_bench_1gpu.err )
( timeout 400 python bench.py --impl reference --steps 3 --warmup 1 > $O/final_bench_reference.json 2> $O/final_bench_reference.err )
( timeout 400 ncu --metrics gpu__time_duration.sum --clock-control none -c 600 --csv --log-file $O/final_bench_launches.csv python bench.py --steps 1 --warmup 3 --calls-per-step 1 > $O/final_bench_under_ncu.log 2>&1 )
( REPS=1 timeout 500 ncu --set full --clock-control none --import-source on -k regex:axis_reg -c 12 -f -o $O/final_axis python tools/profile_axis.py > $O/final_axis_ncu.log 2>&1 )
( timeout 400 ncu --set full --clock-control none --import-source on -k regex:tc_gemm -s 8 -c 2 -f -o $O/final_mdft python tools/bench_mdft.py > $O/final_mdft_ncu.log 2>&1 )
( timeout 200 python tools/bench_paths.py > $O/final_paths.log 2>&1 )
( timeout 200 python tools/bench_mdft.py > $O/final_mdft.log 2>&1; timeout 200 python tools/micro/tf32_peak.py >> $O/final_mdft.log 2>&1; timeout 200 python tools/bench_coronagraph.py 2>&1 | grep p32 >> $O/final_mdft.log )
tail -3 $O/final_pytest.log; tail -2 $O/final_smoke.log; cat $O/final_bench_1gpu.json | cut -c1-600; tail -2 $O/final_bench_1gpu.err; cat $O/final_paths.log $O/final_mdft.log
