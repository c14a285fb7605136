#!/bin/sh
# build_ref.sh — compiles the REFERENCE's own functions of the hot path into oracle/_ref/libref.so (test infrastructure).
#
# The reference as a whole cannot be built here (OpenCV / OpenCL / boost / Eigen / Sophus headers and its cmake build are not in
# this image), but the functions that carry the reference-owned logic of the path are plain C++ over a handful of OpenCV
# containers.  This recipe slices them — by line range, from the sources WHERE THEY LIE in the kpmrozowski/wut-cuda-orb-slam3
# checkout named by ORB_REFERENCE_ROOT, at build time —
# into oracle/_ref/gen/*.inc (git-ignored, never committed) and compiles them against oracle/ref_shim/ (container types only;
# the one OpenCV algorithm a slice calls, cv::FAST, is forwarded to the cv2-pinned oracle).  tests/test_ref_pin.py then checks
# the oracle against this library and tests/golden/make_ref_golden.py freezes its answers as fixtures (tests/golden/ref_golden.json)
# that tests/test_golden.py checks without the reference.
#
# Without ORB_REFERENCE_ROOT the script builds nothing (and says so); tests/test_ref_pin.py, tests/test_gpu_ref.py and the
# reference check of tests/test_gpu_round2.py then compare with the reference's stored answers (tests/golden/ref_pin_golden.json)
# instead of the live library, and the Frame call-site test skips.
set -e
HERE=$(cd "$(dirname "$0")" && pwd)
REF=${ORB_REFERENCE_ROOT:-}
OUT="$HERE/_ref"
if [ -z "$REF" ] || [ ! -d "$REF/src" ]; then
    echo "build_ref: set ORB_REFERENCE_ROOT to a kpmrozowski/wut-cuda-orb-slam3 checkout to build oracle/_ref/libref.so;" \
         "without it the reference tests use the stored answers in tests/golden/ref_pin_golden.json"
    exit 0
fi
mkdir -p "$OUT/gen"
slice() { sed -n "$2,$3p" "$REF/$1" > "$OUT/gen/$4"; }
# --- extractor ---------------------------------------------------------------------------------------------------------
slice include/ORBextractor.h   39 120 ORBextractor_classes.inc       # class ExtractorNode, class ORBextractor
slice src/ORBextractor.cc      99 149 orb_constants_descriptor.inc   # PATCH_SIZE..factorPI, computeOrbDescriptor
slice src/ORBextractor.cc     151 408 orb_bit_pattern.inc            # bit_pattern_31_
slice src/ORBextractor.cc     410 468 orb_ctor.inc                   # ORBextractor::ORBextractor (tables, umax)
slice src/ORBextractor.cc     515 582 orb_divide_compare.inc         # ExtractorNode::DivideNode, compareNodes
slice src/ORBextractor.cc     584 774 orb_distribute_octree.inc      # ORBextractor::DistributeOctTree
slice src/ORBextractor.cc     867 950 orb_tile_calc_keypoints.inc    # tileCalcKeypoints (the CPU cell loop)
slice src/ORBextractor.cc    1283 1303 orb_pack_loop.inc             # operator(): scale + lapping-area placement loop
# --- matcher / frame grid ----------------------------------------------------------------------------------------------
slice src/ORBmatcher3.cc      592 653 matcher_maxima_distance.inc    # ComputeThreeMaxima, DescriptorDistance
slice src/ORBmatcher1.cc       45 223 matcher_projection_map.inc     # SearchByProjection(Frame, MapPoints), RadiusByViewingCos
slice src/ORBmatcher3.cc      256 590 matcher_projection_frames.inc  # SearchByProjection(Current, Last) and (Current, KeyFrame)
slice src/ORBmatcher1.cc      225 427 matcher_bow_kf_frame.inc       # SearchByBoW(KeyFrame*, Frame&, ...)
slice src/ORBmatcher2.cc       36 177 matcher_bow_kf_kf.inc          # SearchByBoW(KeyFrame*, KeyFrame*, ...)
slice src/ORBmatcher2.cc      179 418 matcher_triangulation.inc      # SearchForTriangulation
slice src/CameraModels/Pinhole.cpp 114 128 pinhole_epipolar_tail.inc # Pinhole::epipolarConstrain after F12 (line test)
slice src/MapPoint.cc         368 397 mappoint_distinctive_core.inc  # ComputeDistinctiveDescriptors: distance matrix, least median
slice src/Frame.cc            841 1011 frame_stereo_matches.inc      # Frame::ComputeStereoMatches
slice src/Frame.cc            387 418 frame_assign_grid.inc          # Frame::AssignFeaturesToGrid
slice src/Frame.cc            687 766 frame_area_posingrid.inc       # Frame::GetFeaturesInArea, Frame::PosInGrid
slice src/Frame.cc            111 127 frame_ctor_scale_extract.inc   # stereo Frame ctor: accessor block + the two ExtractORB threads
slice src/Frame.cc            420 455 frame_extract_orb.inc          # extractorParenthesis, Frame::ExtractORB
# --- DBoW2 (vendored under Thirdparty/DBoW2) -----------------------------------------------------------------------------
D=Thirdparty/DBoW2/DBoW2
slice $D/BowVector.cpp         34 84 dbow2_bowvector.inc             # addWeight, addIfNotExist, normalize
slice $D/FeatureVector.cpp     31 45 dbow2_featurevector.inc         # addFeature
slice $D/FORB.cpp              81 101 dbow2_forb_distance.inc        # FORB::distance
slice $D/FORB.cpp             120 135 dbow2_forb_fromstring.inc      # FORB::fromString
slice $D/ScoringObject.cpp     23 68 dbow2_l1_score.inc              # L1Scoring::score
slice $D/TemplatedVocabulary.h 1126 1196 dbow2_transform_all.inc     # transform(features, BowVector, FeatureVector, levelsup)
slice $D/TemplatedVocabulary.h 1217 1259 dbow2_transform_one.inc     # transform(feature, word_id, weight, nid, levelsup)
slice $D/TemplatedVocabulary.h 1337 1424 dbow2_load_text.inc         # loadFromTextFile
# the system compiler links libstdc++ dynamically; a toolchain that links it statically breaks iostreams in a dlopen()ed library
if [ -x /usr/bin/g++ ]; then CXX=/usr/bin/g++; else CXX=${CXX:-g++}; fi
# plain -O3 as the reference builds (CMakeLists.txt:105-107), no FMA contraction
$CXX -O3 -std=c++17 -fPIC -ffp-contract=off -w -I"$HERE/ref_shim" -I"$OUT/gen" -shared -o "$OUT/libref.so" \
    "$HERE/ref_shim/ref_wrapper.cpp" "$HERE/ref_shim/ref_dbow2_wrapper.cpp" -L"$HERE/_build" -lorb_oracle -Wl,-rpath,'$ORIGIN/../_build'
echo "build_ref: built $OUT/libref.so from $REF"
# The reference's call site of the extractor (Frame ctor accessor block + Frame::ExtractORB) compiled UNCHANGED against the
# drop-in adapter header; linked against the product library, run on the GPU by tests/test_gpu_round2.py.
ROOT=$(cd "$HERE/.." && pwd)
if [ -f "$ROOT/wut_cuda_orb_slam3_b200/liborbx.so" ]; then
    $CXX -O2 -std=c++17 -w -pthread -I"$ROOT/tests/cpp/cv_stub" -I"$ROOT/include" -I"$ROOT/wut_cuda_orb_slam3_b200/csrc/adapter" -I"$OUT/gen" \
        -o "$OUT/frame_callsite_test" "$HERE/ref_shim/frame_callsite_main.cpp" -L"$ROOT/wut_cuda_orb_slam3_b200" -lorbx \
        -Wl,-rpath,'$ORIGIN/../../wut_cuda_orb_slam3_b200'
    echo "build_ref: built $OUT/frame_callsite_test (reference src/Frame.cc:111-127, 420-455 against csrc/adapter/ORBextractor.h)"
fi
