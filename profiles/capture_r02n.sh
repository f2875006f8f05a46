#!/bin/bash
# r02n: sort after the full-tile fast path: parity
O=gpurun_out; mkdir -p $O; rm -f $O/r02n_sort_variants.txt
timeout 900 python -m pytest tests/test_gpu_parity.py -m gpu -q -k "sort or weighted" > $O/r02n_gputest.log 2>&1; echo "pytest rc=$?" >> $O/r02n_gputest.log
tail -4 $O/r02n_gputest.log
