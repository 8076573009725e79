set -u
O=gpurun_out
timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -8 > $O/r02_t9.log
timeout 300 ./oracle/_ref/shim/shim_harness > $O/r02_shim_harness.log 2>&1; echo "shim rc=$?" >> $O/r02_t9.log
timeout 300 python tools/devbench.py lab 8192 > $O/r02_dev_lab.log 2>&1
timeout 300 python tools/devbench.py stencils 4096 > $O/r02_dev_stencils.log 2>&1
cat $O/r02_t9.log; tail -3 $O/r02_shim_harness.log; cat $O/r02_dev_lab.log $O/r02_dev_stencils.log
