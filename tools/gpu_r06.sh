#!/bin/bash
# One run on one B200: the d = 2 table of acceptance-ratio bounds against the parent commit's build.
#   mcpar_b200/variants/libmcgpu_old.so  = libmcgpu.so built at the parent commit (copied there before the change);
#   mcpar_b200/variants/libmcgpu_cnt<G>.so = counting builds (tools/build_variant.py cnt<G> -DMCGPU_CELL_COUNT -DMCGPU_CELL_G=<G>);
#   the tree's own libmcgpu.so is the new build.
# Writes OUTDIR/r06_*: the card's name and power limit, the GPU tests and smoke(), bench.py --dump-outputs of both
# builds (compared byte for byte), three alternating timed runs of each build for five configurations, and the
# table's hit rates at G = 32 / 64 / 128.
#   usage: bash tools/gpu_r06.sh OUTDIR
OUT=${1:?usage: bash tools/gpu_r06.sh OUTDIR}
mkdir -p "$OUT"
V=$PWD/mcpar_b200/variants
OLD=$V/libmcgpu_old.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/r06_smi.txt 2>&1
python -c "import __graft_entry__ as g; g.build()" > $OUT/r06_build.log 2>&1 || echo "build rc=$?" >> $OUT/r06_build.log
timeout 1500 python -m pytest -q -m gpu tests > $OUT/r06_pytest_gpu.txt 2>&1; echo "pytest -m gpu rc=$?" >> $OUT/r06_pytest_gpu.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r06_smoke.txt 2>&1; echo "smoke rc=$?" >> $OUT/r06_smoke.txt

# results: the default bench line with its outputs dumped, old and new build
MCGPU_LIB=$OLD timeout 600 python bench.py --no-cpu --no-e2e --no-modes --dump-outputs $OUT/r06_dump_old > $OUT/r06_dump_old.json 2> $OUT/r06_dump.err
timeout 600 python bench.py --no-cpu --no-e2e --no-modes --dump-outputs $OUT/r06_dump_new > $OUT/r06_dump_new.json 2>> $OUT/r06_dump.err
diff -rq $OUT/r06_dump_old $OUT/r06_dump_new > $OUT/r06_dump_cmp.txt 2>&1 \
  && echo "dumps identical: $(ls $OUT/r06_dump_new | wc -l) files" >> $OUT/r06_dump_cmp.txt \
  || echo "dumps DIFFER" >> $OUT/r06_dump_cmp.txt
rm -rf $OUT/r06_dump_old $OUT/r06_dump_new     # 60 MB each: only the comparison is kept

# timing: old and new alternately, three runs each
B="python bench.py --no-cpu --no-e2e --no-modes --steps 300"
for cfg in "default:" "rosen2d:--workload rosen2d" "summix:--remote-mode summix" "pool64:--pool 64" "pool256:--pool 256"; do
  tag=${cfg%%:*}; args=${cfg#*:}
  for i in 1 2 3; do
    MCGPU_LIB=$OLD timeout 300 $B $args > $OUT/r06_${tag}_old_$i.json 2>> $OUT/r06_bench.err
    timeout 300 $B $args > $OUT/r06_${tag}_new_$i.json 2>> $OUT/r06_bench.err
  done
done

# hit rates of the table, default line, from the counting builds
for g in 32 64 128; do
  timeout 300 python tools/cell_hits.py $V/libmcgpu_cnt$g.so --no-cpu --no-e2e --no-modes --steps 300 2>> $OUT/r06_hits.err | tail -1 > $OUT/r06_hits_g$g.json
done

cat $OUT/r06_smi.txt $OUT/r06_dump_cmp.txt; tail -3 $OUT/r06_pytest_gpu.txt; tail -1 $OUT/r06_smoke.txt; cat $OUT/r06_hits_g*.json
