#!/bin/bash
# usage: tools/prof_report.sh <ncu-rep> <cubin-basename e.g. lrds_tc_f16x3> <kernel-substring> [top]
set -e
rep=$1; unit=$2; kname=$3; top=${4:-40}
tmp=$(mktemp -d)
ncu -i $rep --page raw --csv > $tmp/raw.csv 2>/dev/null
ncu -i $rep --page source --csv > $tmp/src.csv 2>/dev/null
python tools/ncu_summary.py $tmp/raw.csv "$(basename $rep)"
lib=$(cd "$(dirname "$0")/.." && pwd)/sde_sampler_lrds_b200/csrc/liblrds_b200.so
(cd $tmp && cuobjdump -xelf all "$lib" >/dev/null 2>&1)
echo
echo '```'
python tools/ncu_by_line.py $tmp/src.csv $tmp/$unit.sm_100a.cubin "$kname" $top
echo '```'
rm -rf $tmp
