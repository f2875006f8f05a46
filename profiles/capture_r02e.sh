#!/bin/bash
# r02e: W-S fast-path changes (parity), then the fused chain kernel with its source page
O=gpurun_out; mkdir -p $O
timeout 900 python -m pytest tests -m gpu -q -x -k "ws or config2 or golden or crmath" > $O/r02e_gputest.log 2>&1; echo "pytest rc=$?" >> $O/r02e_gputest.log
tail -3 $O/r02e_gputest.log
SMALL="python bench.py --rays 2e7 --steps 2 --warmup 3 --no-e2e --no-cpu-baseline --no-configs"
$SMALL > $O/r02e_bench_small.json 2> $O/r02e_bench_small.err &&
ncu --set full --clock-control none --import-source on -k regex:k_chain -s 3 -c 1 -o $O/r02e_k_chain -f $SMALL > $O/r02e_ncu_k_chain.log 2>&1
if [ -f $O/r02e_k_chain.ncu-rep ]; then
  python profiles/summarize.py kernel $O/r02e_k_chain.ncu-rep > $O/r02e_k_chain.txt 2>&1
  ncu -i $O/r02e_k_chain.ncu-rep --page source --csv 2>/dev/null | gzip -9 > $O/r02e_k_chain_source.csv.gz
  rm -f $O/r02e_k_chain.ncu-rep
fi
