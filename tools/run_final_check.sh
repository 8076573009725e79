set -u
O=gpurun_out
timeout 1500 python -m pytest tests -q -m gpu 2>&1 | tail -25 > $O/final_tests.log
timeout 300 python __graft_entry__.py --smoke > $O/final_smoke.log 2>&1; echo "smoke rc=$?" >> $O/final_tests.log
timeout 300 ./oracle/_ref/shim/shim_harness > $O/final_shim.log 2>&1; echo "shim rc=$?" >> $O/final_tests.log
timeout 900 python bench.py > $O/final_bench.json 2> $O/final_bench.err; echo "bench rc=$?" >> $O/final_tests.log
cat $O/final_tests.log; tail -2 $O/final_smoke.log; grep -E "FAIL|hits" $O/final_shim.log | tail -3; head -c 400 $O/final_bench.json
