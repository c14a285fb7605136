#!/bin/bash
# Run on the GPU box (gpurun): final bench + ncu evidence, copied into profiles/ under the tag given as $1 (e.g. r01b).
# Every ncu command is preceded by the same command without ncu (B200_PROFILING.md); numbers printed under ncu are never used.
set -u
TAG=${1:-r01b}
OUT=gpurun_out
mkdir -p $OUT profiles
python bench.py --steps 10 --warmup 3 > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err
# launch list of the bench's own batch (512 frames per launch)
LARGS="--steps 2 --warmup 1 --no-knn2 --no-cpu --no-other"
python bench.py $LARGS > $OUT/plain.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -c 120 --csv --log-file $OUT/${TAG}_launches_b512.csv python bench.py $LARGS > $OUT/ncu_l.log 2>&1
python tools/launch_shares.py $OUT/${TAG}_launches_b512.csv $OUT/${TAG}_bench.json 512 > $OUT/${TAG}_launch_shares_b512.txt 2>&1
# full captures of the dominant extraction kernel and of the matcher (small batch: ncu replays each kernel ~40 times)
ARGS="--steps 1 --warmup 1 --batch 64 --no-knn2 --no-cpu --no-other"
python bench.py $ARGS > $OUT/plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:fast_cells_warp -s 3 -c 1 -f -o $OUT/${TAG}_fast_cells_warp python bench.py $ARGS > $OUT/ncu_f.log 2>&1
KARGS="--steps 1 --warmup 1 --batch 32 --no-cpu --no-other --knn-ndb 1000000 --knn-reps 1"   # --no-other: the KITTI pair of the other configs launches knn2_kernel first (4 CTAs)
python bench.py $KARGS > $OUT/plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:knn2_kernel -s 1 -c 1 -f -o $OUT/${TAG}_knn2 python bench.py $KARGS > $OUT/ncu_k.log 2>&1
python bench.py $ARGS > $OUT/plain.log 2>&1 && \
ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -k regex:fast_cells_warp -s 3 -c 3 --csv --log-file $OUT/${TAG}_fast_dram.csv python bench.py $ARGS > $OUT/ncu_d.log 2>&1
python bench.py $ARGS > $OUT/plain.log 2>&1 && \
ncu --set full --clock-control none --import-source on -k regex:blur_mma -s 1 -c 1 -f -o $OUT/${TAG}_blur_mma python bench.py $ARGS > $OUT/ncu_b.log 2>&1
python tools/latency.py > $OUT/${TAG}_single_frame_latency.txt 2>&1
# rectification / resize kernels and the projection-guided searches (SURVEY.md §8(f)2-3)
python tools/prep_bench.py > $OUT/${TAG}_prep_bench.json 2> $OUT/prep_bench.err && \
ncu --set full --clock-control none --import-source on -k regex:remap_tiled_kernel -s 3 -c 1 -f -o $OUT/${TAG}_remap_tiled python tools/prep_bench.py > $OUT/ncu_r.log 2>&1
python tools/prep_bench.py > $OUT/plain.log 2>&1 && \
ncu --metrics gpu__time_duration.sum --clock-control none -k regex:"proj_|frame_grid" -c 40 --csv --log-file $OUT/${TAG}_proj_launches.csv python tools/prep_bench.py > $OUT/ncu_p.log 2>&1
tail -n 2 $OUT/ncu_f.log; tail -n 2 $OUT/ncu_k.log; tail -n 3 $OUT/${TAG}_launch_shares_b512.txt
