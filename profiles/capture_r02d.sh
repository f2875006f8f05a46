#!/bin/bash
# r02d: parity of the rewritten LL / Zernike / W-S clamp paths, then the captures
O=gpurun_out; mkdir -p $O
timeout 900 python -m pytest tests -m gpu -q -x -k "legendre or zern or ws or golden or fused or surfaces or config" > $O/r02d_gputest.log 2>&1; echo "pytest rc=$?" >> $O/r02d_gputest.log
tail -3 $O/r02d_gputest.log
bash profiles/capture_routines.sh r02d
