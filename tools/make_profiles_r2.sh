#!/bin/bash
# Run on the GPU box (gpurun): round-2 evidence.  bench line, launch list of the same command, ncu --set full captures of every
# extraction kernel (each preceded by the same command without ncu; numbers printed under ncu are never used), latency tables.
set -u
TAG=${1:-r02a}
OUT=gpurun_out
mkdir -p $OUT
python bench.py --steps 10 --warmup 3 > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err
LARGS="--steps 2 --warmup 1 --no-knn2 --no-cpu --no-other --no-cfg4"
python bench.py $LARGS > $OUT/plain.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -c 120 --csv --log-file $OUT/${TAG}_launches_b512.csv python bench.py $LARGS > $OUT/ncu_l.log 2>&1
python tools/launch_shares.py $OUT/${TAG}_launches_b512.csv $OUT/${TAG}_bench.json 512 > $OUT/${TAG}_launch_shares_b512.txt 2>&1
ARGS="--steps 1 --warmup 1 --batch 64 --no-knn2 --no-cpu --no-other --no-cfg4"
python bench.py $ARGS > $OUT/plain.log 2>&1 || { tail -5 $OUT/plain.log; exit 1; }
for K in fast_cells_warp:3 octree_kernel:1 orient_describe:1 pyr_resize_pipe:7 blur_mma:1; do
  NAME=${K%%:*}; SKIP=${K##*:}
  ncu --set full --clock-control none --import-source on -k regex:$NAME -s $SKIP -c 1 -f -o $OUT/${TAG}_$NAME python bench.py $ARGS > $OUT/ncu_$NAME.log 2>&1
  tail -n 1 $OUT/ncu_$NAME.log
done
KARGS="--steps 1 --warmup 1 --batch 32 --no-cpu --no-other --no-cfg4 --knn-ndb 1000000 --knn-reps 1"
python bench.py $KARGS > $OUT/plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:knn2_kernel -s 1 -c 1 -f -o $OUT/${TAG}_knn2 python bench.py $KARGS > $OUT/ncu_k.log 2>&1
python tools/latency.py > $OUT/${TAG}_single_frame_latency.txt 2>&1
tail -n 3 $OUT/${TAG}_launch_shares_b512.txt
