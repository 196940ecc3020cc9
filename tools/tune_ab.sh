#!/bin/bash
# A/B of CSVB200_TUNE values in ONE run on the same box: bash tools/tune_ab.sh "0 1024" [rounds]
for r in $(seq 1 ${2:-2}); do for t in $1; do CSVB200_TUNE=$t bash tools/kbench.sh t$t 2>/dev/null | sed "s/^/round $r /"; done; done
