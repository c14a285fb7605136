"""B200-native ORB front end (pyramid -> FAST -> octree -> orientation -> blur -> rBRIEF -> Hamming matching).

Host-side mirror of the reference's interface for this path (ORB_SLAM3::ORBextractor / ORBmatcher) over the C-ABI
library liborbx.so (include/orbx.h).  The compute path is hand-written sm_100a CUDA; importing this package without
the built library raises (no CPU fallback).
"""
from . import capi, synth  # noqa: F401
from .capi import KP_DTYPE, OrbxError, lib  # noqa: F401
from .bow import (FeatureVector, ORBVocabulary, search_by_bow, search_for_triangulation,  # noqa: F401
                  search_for_triangulation_batch)
from .extractor import ORBextractor, compute_tables, distribute_octree  # noqa: F401
from .prep import Rectifier, undistort_keypoints  # noqa: F401
from .projection import (FrameView, KeyFrameView, fuse, fuse_sim3, projection_rounds, search_by_projection_kf,  # noqa: F401
                         search_by_projection_last, search_by_projection_map, search_by_projection_sim3, search_for_initialization)
from . import io  # noqa: F401
from .matcher import (ORBmatcher, ShardedMatcher, compute_stereo_matches, distinctive_descriptor, distinctive_descriptors, extract_stereo,  # noqa: F401
                      knn2_device, knn2_merge_device, measure_popc_peak, rotation_consistency)

lib()  # fail loudly at import time if the CUDA extension is missing
