#!/bin/bash
# SASS evidence for profiles/ (run on the CPU box: cuobjdump reads the built liborbx.so): one listing per production kernel
# (instruction text only, encodings stripped) + a summary with the opcode histogram and the Blackwell-specific mnemonics
# (UTMALDG = cp.async.bulk.tensor / TMA, LDGSTS = cp.async, VIMNMX(3) = packed integer min/max, LOP3/POPC = the matcher).
TAG=${1:-r02}
SO=wut_cuda_orb_slam3_b200/liborbx.so
OUT=profiles
mkdir -p $OUT
SUM=$OUT/${TAG}_sass_summary.txt
echo "cuobjdump -sass of $SO ($(date -u +%Y-%m-%dT%H:%MZ)); arch: $(cuobjdump -lelf $SO | grep -o 'sm_[0-9a-z]*' | sort | uniq -c | tr '\n' ' ')" > $SUM
cuobjdump -sass $SO 2>/dev/null | awk '
  /Function :/ { fn=$3 }
  /^[ \t]+\/\*[0-9a-f]+\*\/[ \t]+[A-Z@]/ { line=$0; sub(/^[ \t]+\/\*[0-9a-f]+\*\/[ \t]+/, "", line); sub(/[ \t]*\/\*.*$/, "", line); print fn "\t" line }' > /tmp/all_sass.tsv
for pat in pyr_resize_pipe_kernel pyr_resize_tiled_kernelILi32 pyr_level0_tiled blur_pipe_kernel fast_cells_warp_kernelILi48 fast_cells_kernel octree_kernelILi256 octree_kernelILi1024 orient_describe_kernelILb1 orient_describe_kernelILb0 pack_kernelILi256 knn2_imma_kernel knn2_kernelILi6 knn2_merge stereo_match_kernel remap_tiled resize_tiled distinctive_kernel; do
  fn=$(cut -f1 /tmp/all_sass.tsv | grep "$pat" | sort -u | head -1)
  [ -z "$fn" ] && { echo "missing $pat" >> $SUM; continue; }
  short=$(echo $pat | sed 's/ILi/_/')
  grep -F "$fn" /tmp/all_sass.tsv | cut -f2 > $OUT/${TAG}_sass_${short}.txt
  n=$(wc -l < $OUT/${TAG}_sass_${short}.txt)
  echo "" >> $SUM
  echo "== $short ($fn): $n instructions" >> $SUM
  echo "   Blackwell / async mnemonics: $(grep -oE '^(@!?U?P[0-9] +)?(UTMALDG[.A-Z0-9]*|UTMASTG[.A-Z0-9]*|UBLKCP[.A-Z0-9]*|LDGSTS[.A-Z0-9]*|SYNCS[.A-Z0-9]*|UTC[A-Z]*MMA|HMMA|LDTM|STTM)' $OUT/${TAG}_sass_${short}.txt | sed 's/^@!\?U\?P[0-9] \+//' | sort | uniq -c | tr '\n' ';')" >> $SUM
  echo "   top opcodes: $(sed 's/^@!\?U\?P[0-9] \+//' $OUT/${TAG}_sass_${short}.txt | awk '{print $1}' | sed 's/\..*//' | sort | uniq -c | sort -rn | head -12 | awk '{printf "%s %s, ", $2, $1}')" >> $SUM
done
cat $SUM | head -60
