#!/bin/bash
# Evidence bundle of round 2 (tag r02): launch list, ncu full-set captures of EVERY conv kernel variant, single-pass
# DRAM traffic.  Raw CSV pages are condensed with scripts/ncu_summary.py on the build box.
# Usage: scripts/gpu_evidence_r02.sh [OUT]  (output directory; default build/evidence_r02, which git ignores)
OUT=${1:-build/evidence_r02}
mkdir -p $OUT
T=r02
NCU="ncu --set full --clock-control none --import-source on"
B2="python bench.py --workload cfg2 --steps 1 --warmup 1 --no-cpu"
# launch list of the headline command (short clip so that the list stays small): BSVD clip + RRDBNet frames
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv --log-file $OUT/${T}_launches_cfg3.csv python bench.py --steps 1 --warmup 1 --clip 2 --no-cpu > $OUT/ncu_list.log 2>&1
tail -1 $OUT/ncu_list.log | cut -c1-200
# <32>: one residual dense block of the trunk (five consecutive launches of the second frame); <64> + <16>: the tail
timeout 900 $NCU -k regex:conv3x3_stream -s 390 -c 5 -f -o $OUT/${T}_trunk_full $B2 > $OUT/ncu_a.log 2>&1
timeout 900 $NCU -k regex:conv3x3_stream -s 700 -c 5 -f -o $OUT/${T}_tail_full $B2 > $OUT/ncu_b.log 2>&1
# <64> body + <48> last conv of SRVGGNetCompact-32 x4 at 720p
timeout 900 $NCU -k regex:conv3x3_stream -s 64 -c 5 -f -o $OUT/${T}_srvgg_full python scripts/ncu_srvgg.py > $OUT/ncu_c.log 2>&1
# BSVD-32 clip (fp16, 8 frames): first DenBlock incl. the two stride-2 convs on the streaming kernel, scatter / PixelShuffle stores
timeout 900 $NCU -k regex:conv3x3_stream -s 97 -c 16 -f -o $OUT/${T}_bsvd_full python scripts/profile_bsvd.py 8 > $OUT/ncu_d.log 2>&1
for r in trunk tail srvgg bsvd; do
  ncu -i $OUT/${T}_${r}_full.ncu-rep --page raw --csv > $OUT/${T}_${r}_full_raw.csv 2>/dev/null
  wc -l $OUT/${T}_${r}_full_raw.csv
done
rm -f $OUT/*.ncu-rep
# DRAM traffic of one RRDBNet frame, one pass, warm caches
timeout 900 ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum --cache-control none --clock-control none \
  -k regex:'conv3x3|prep_kernel' -c 800 --csv --log-file $OUT/${T}_dram_launches_b1.csv $B2 > $OUT/ncu_f.log 2>&1
ls -la $OUT | tail -20
