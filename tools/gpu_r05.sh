#!/bin/bash
# One run on one B200 (a few minutes): the packed-fp32 candidate round against the parent commit's build.
#   mcpar_b200/variants/libmcgpu_old.so = libmcgpu.so built at the parent commit (copied there before the change);
#   the tree's own libmcgpu.so is the new build.
# Writes OUTDIR/r05_*: the card's name and power limit, bench.py --dump-outputs of both builds (outputs compared
# byte for byte), and three alternating timed runs of each build for three configurations.
#   usage: bash tools/gpu_r05.sh OUTDIR
OUT=${1:?usage: bash tools/gpu_r05.sh OUTDIR}
mkdir -p "$OUT"
OLD=$PWD/mcpar_b200/variants/libmcgpu_old.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/r05_smi.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/r05_build.log 2>&1 || echo "build rc=$?" >> $OUT/r05_build.log

# results: the default bench line with its outputs dumped, old and new build
MCGPU_LIB=$OLD timeout 600 python bench.py --no-cpu --no-e2e --no-modes --dump-outputs $OUT/r05_dump_old > $OUT/r05_dump_old.json 2> $OUT/r05_dump.err
timeout 600 python bench.py --no-cpu --no-e2e --no-modes --dump-outputs $OUT/r05_dump_new > $OUT/r05_dump_new.json 2>> $OUT/r05_dump.err
diff -rq $OUT/r05_dump_old $OUT/r05_dump_new > $OUT/r05_dump_cmp.txt 2>&1 \
  && echo "dumps identical: $(ls $OUT/r05_dump_new | wc -l) files" >> $OUT/r05_dump_cmp.txt \
  || echo "dumps DIFFER" >> $OUT/r05_dump_cmp.txt
rm -rf $OUT/r05_dump_old $OUT/r05_dump_new     # 60 MB each: only the comparison is kept

# timing: old and new alternately, three runs each
B="python bench.py --no-cpu --no-e2e --no-modes --steps 300"
for cfg in "default:" "summix:--remote-mode summix" "rosen2d:--workload rosen2d"; do
  tag=${cfg%%:*}; args=${cfg#*:}
  for i in 1 2 3; do
    MCGPU_LIB=$OLD timeout 300 $B $args > $OUT/r05_${tag}_old_$i.json 2>> $OUT/r05_bench.err
    timeout 300 $B $args > $OUT/r05_${tag}_new_$i.json 2>> $OUT/r05_bench.err
  done
done

cat $OUT/r05_smi.txt $OUT/r05_dump_cmp.txt
