// loop_oracle.cpp — CPU ORACLE (TEST INFRASTRUCTURE ONLY, never shipped, never on the product path).
//
// Line-by-line restatement of the two loop-closing searches of ORBmatcher (upstream ORB-SLAM3 v1.0, NLeft == -1):
//   SearchByProjection(KeyFrame* pKF, Sophus::Sim3f& Scw, vpPoints, [vpPointsKFs,] vpMatched, [vpMatchedKF,] th, ratioHamming)
//                                                                                          src/ORBmatcher1.cc:429-648
//   Fuse(KeyFrame* pKF, Sophus::Sim3f& Scw, vpPoints, th, vpReplacePoint)                 src/ORBmatcher2.cc:612-729
// KeyFrame::IsInImage and KeyFrame::GetFeaturesInArea are the ones of tests/cpp/fuse_oracle.cpp, whose grid is the projection
// oracle's own Frame::AssignFeaturesToGrid; both files are included, not copied.  The map-point side of each loop (isBad, the
// spAlreadyFound snapshot, the Sophus / Eigen projection, p3Dc(2) < 0, the distance window, the viewing angle, PredictScale) is
// folded into (valid, u, v, level) by the caller.  SearchByProjection runs the sequential loop with vpMatched updated in place;
// for Fuse the bookkeeping after a match (vpReplacePoint / AddMapPoint) is left out: per pair this returns bestIdx when
// bestDist <= TH_LOW, else -1.  Built on demand by tests/loop_oracle.py into build/.
#include <climits>

#include "fuse_oracle.cpp"

extern "C" {

// SearchByProjection(pKF, Scw, vpPoints, vpMatched, th, ratioHamming).  The key frame: kp / desc [n], bounds_grid[6],
// scale[nlev] (mvScaleFactors).  matched[n] = vpMatched as point ids (-1 = NULL), in / out: entries assigned by this call become
// the point index.  Point i: valid[i], (u[i], v[i]) = pKF->mpCamera->project(p3Dc), level[i] = PredictScale, descriptor row i of
// pdesc.  Returns nmatches, or -1 where the reference would write vpMatched[-1] (no candidate and TH_LOW * ratioHamming >= 256).
int orbo_search_by_projection_sim3(const KeyPoint* kp, const uint8_t* desc, int n, const float* bounds_grid, const float* scale,
                                   int32_t* matched, int n_points, const uint8_t* valid, const float* u, const float* v,
                                   const int32_t* level, const uint8_t* pdesc, int th, float ratioHamming)
{
    KeyFrame K;
    fill_frame(K, kp, desc, nullptr, n, bounds_grid, scale);
    KeyFrame* pKF = &K;
    int32_t* vpMatched = matched;
    int nmatches = 0;
    // For each Candidate MapPoint Project and Match
    for (int iMP = 0, iendMP = n_points; iMP < iendMP; iMP++) {
        // Discard Bad MapPoints and already found; depth, distance window, viewing angle (the caller)
        if (!valid[iMP]) continue;
        const float uv0 = u[iMP], uv1 = v[iMP];
        // Point must be inside the image
        if (!pKF->IsInImage(uv0, uv1)) continue;
        int nPredictedLevel = level[iMP];
        // Search in a radius
        const float radius = th * pKF->mvScaleFactors[nPredictedLevel];
        const std::vector<size_t> vIndices = pKF->GetFeaturesInArea(uv0, uv1, radius);
        if (vIndices.empty()) continue;
        // Match to the most similar keypoint in the radius
        const uint8_t* dMP = pdesc + (size_t)iMP * 32;
        int bestDist = 256;
        int bestIdx = -1;
        for (std::vector<size_t>::const_iterator vit = vIndices.begin(), vend = vIndices.end(); vit != vend; vit++) {
            const size_t idx = *vit;
            if (vpMatched[idx] != -1) continue;
            const int& kpLevel = pKF->mvKeysUn[idx].octave;
            if (kpLevel < nPredictedLevel - 1 || kpLevel > nPredictedLevel) continue;
            const uint8_t* dKF = pKF->mDescriptors + idx * 32;
            const int dist = DescriptorDistance(dMP, dKF);
            if (dist < bestDist) {
                bestDist = dist;
                bestIdx = (int)idx;
            }
        }
        if (bestDist <= TH_LOW * ratioHamming) {
            if (bestIdx < 0) return -1;
            vpMatched[bestIdx] = iMP;
            nmatches++;
        }
    }
    return nmatches;
}

// The search part of Fuse(pKF, Scw, vpPoints, th, vpReplacePoint) for n_kf key frames, in the layout of orbo_fuse
// (tests/cpp/fuse_oracle.cpp) without mvuRight, mvInvLevelSigma2, mbf and invz: the Sim3 Fuse has no reprojection gate.
void orbo_fuse_sim3(int n_kf, const int32_t* feat_off, const KeyPoint* kp, const uint8_t* desc, const float* bounds_grid, int nlev,
                    const float* scale, const int32_t* kf_off, const uint8_t* point_desc, const int32_t* point, const uint8_t* valid,
                    const float* u, const float* v, const int32_t* level, float th, int32_t* match, int32_t* n_fused)
{
    for (int k = 0; k < n_kf; ++k) {
        KeyFrame K;
        const int f0 = feat_off[k];
        fill_frame(K, kp + f0, desc + (size_t)f0 * 32, nullptr, feat_off[k + 1] - f0, bounds_grid + 6 * k, scale + (size_t)nlev * k);
        KeyFrame* pKF = &K;
        int nFused = 0;
        // For each candidate MapPoint project and match
        for (int iMP = kf_off[k]; iMP < kf_off[k + 1]; iMP++) {
            match[iMP] = -1;
            // Discard Bad MapPoints and already found; depth (the caller)
            if (!valid[iMP]) continue;
            const float uv0 = u[iMP], uv1 = v[iMP];
            // Point must be inside the image
            if (!pKF->IsInImage(uv0, uv1)) continue;
            // Compute predicted scale level (distance window and viewing angle: the caller)
            const int nPredictedLevel = level[iMP];
            // Search in a radius
            const float radius = th * pKF->mvScaleFactors[nPredictedLevel];
            const std::vector<size_t> vIndices = pKF->GetFeaturesInArea(uv0, uv1, radius);
            if (vIndices.empty()) continue;
            // Match to the most similar keypoint in the radius
            const uint8_t* dMP = point_desc + (size_t)point[iMP] * 32;
            int bestDist = INT_MAX;
            int bestIdx = -1;
            for (std::vector<size_t>::const_iterator vit = vIndices.begin(); vit != vIndices.end(); vit++) {
                const size_t idx = *vit;
                const int& kpLevel = pKF->mvKeysUn[idx].octave;
                if (kpLevel < nPredictedLevel - 1 || kpLevel > nPredictedLevel) continue;
                const uint8_t* dKF = pKF->mDescriptors + idx * 32;
                int dist = DescriptorDistance(dMP, dKF);
                if (dist < bestDist) {
                    bestDist = dist;
                    bestIdx = (int)idx;
                }
            }
            // If there is already a MapPoint replace otherwise add new measurement: the caller's bookkeeping
            if (bestDist <= TH_LOW) {
                match[iMP] = bestIdx;
                nFused++;
            }
        }
        n_fused[k] = nFused;
    }
}

}  // extern "C"
