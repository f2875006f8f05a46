#!/bin/bash
# r02k: one-sweep sort parity and timing
O=gpurun_out; mkdir -p $O
timeout 900 python -m pytest tests/test_gpu_parity.py -m gpu -q -k "sort or weighted" > $O/r02k_gputest.log 2>&1; echo "pytest rc=$?" >> $O/r02k_gputest.log
tail -4 $O/r02k_gputest.log
timeout 300 python profiles/sort_probe.py 2e8 3 > $O/r02k_sort.txt 2>&1
cat $O/r02k_sort.txt
