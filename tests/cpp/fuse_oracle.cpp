// fuse_oracle.cpp — CPU ORACLE (TEST INFRASTRUCTURE ONLY, never shipped, never on the product path).
//
// Line-by-line restatement of the search part of ORBmatcher::Fuse(KeyFrame* pKF, const vector<MapPoint*>& vpMapPoints, th,
// bRight) (src/ORBmatcher2.cc:420-610, NLeft == -1, bRight == false), as LocalMapping::SearchInNeighbors calls it
// (src/LocalMapping.cc:766-803), with KeyFrame::IsInImage and KeyFrame::GetFeaturesInArea (the KeyFrame version: no level
// arguments).  The key frame's grid is the projection oracle's own Frame::AssignFeaturesToGrid, which this file compiles in
// unchanged (oracle/projection_oracle.cpp is included, not copied).  The map-point side of the loop (isBad, IsInKeyFrame, the
// Sophus / Eigen projection, the distance window, the viewing angle, PredictScale) is folded into (valid, u, v, invz, level) by
// the caller, and the bookkeeping after a match (AddMapPoint / Replace) is left out: per pair this returns bestIdx when
// bestDist <= TH_LOW, else -1.  Built on demand by tests/fuse_oracle.py into build/.
#include "../../oracle/projection_oracle.cpp"

namespace {
constexpr int TH_LOW = 50;            // src/ORBmatcher1.cc:37

// The slice of ORB_SLAM3::KeyFrame that Fuse reads.  The grid (mGrid) is the frame's, copied by the KeyFrame constructor.
struct KeyFrame : Frame {
    float mbf = 0;
    const float* mvInvLevelSigma2 = nullptr;
    int NLeft = -1;

    // KeyFrame::IsInImage
    bool IsInImage(const float& x, const float& y) const { return (x >= mnMinX && x < mnMaxX && y >= mnMinY && y < mnMaxY); }

    // KeyFrame::GetFeaturesInArea(x, y, r, bRight = false)
    std::vector<size_t> GetFeaturesInArea(const float& x, const float& y, const float& r) const
    {
        std::vector<size_t> vIndices;
        vIndices.reserve(N);
        float factorX = r;
        float factorY = r;
        const int nMinCellX = std::max(0, (int)floor((x - mnMinX - factorX) * mfGridElementWidthInv));
        if (nMinCellX >= FRAME_GRID_COLS) return vIndices;
        const int nMaxCellX = std::min((int)FRAME_GRID_COLS - 1, (int)ceil((x - mnMinX + factorX) * mfGridElementWidthInv));
        if (nMaxCellX < 0) return vIndices;
        const int nMinCellY = std::max(0, (int)floor((y - mnMinY - factorY) * mfGridElementHeightInv));
        if (nMinCellY >= FRAME_GRID_ROWS) return vIndices;
        const int nMaxCellY = std::min((int)FRAME_GRID_ROWS - 1, (int)ceil((y - mnMinY + factorY) * mfGridElementHeightInv));
        if (nMaxCellY < 0) return vIndices;
        for (int ix = nMinCellX; ix <= nMaxCellX; ix++) {
            for (int iy = nMinCellY; iy <= nMaxCellY; iy++) {
                const std::vector<size_t> vCell = mGrid[ix][iy];
                for (size_t j = 0, jend = vCell.size(); j < jend; j++) {
                    const KeyPoint& kpUn = mvKeysUn[vCell[j]];
                    const float distx = kpUn.x - x;
                    const float disty = kpUn.y - y;
                    if (fabs(distx) < r && fabs(disty) < r) vIndices.push_back(vCell[j]);
                }
            }
        }
        return vIndices;
    }
};
}  // namespace

extern "C" {

// KeyFrame::GetFeaturesInArea on one key frame; returns the count, indices in the reference's order.
int orbo_kf_get_features_in_area(const KeyPoint* kp, int n, const float* bounds_grid, float x, float y, float r, int32_t* out)
{
    KeyFrame K;
    fill_frame(K, kp, nullptr, nullptr, n, bounds_grid, nullptr);
    const std::vector<size_t> v = K.GetFeaturesInArea(x, y, r);
    for (size_t i = 0; i < v.size(); ++i) out[i] = (int32_t)v[i];
    return (int)v.size();
}

// n_kf key frames with their features concatenated: key frame k owns rows [feat_off[k], feat_off[k + 1]) of kp / desc / uright
// (mvuRight: -1 for monocular), bounds_grid[k][6], scale[k][nlev] (mvScaleFactors), inv_sigma2[k][nlev] (mvInvLevelSigma2),
// bf[k] (mbf).  Pairs [kf_off[k], kf_off[k + 1]) belong to key frame k: map point point[q] (descriptor row of point_desc),
// valid[q] (the map-point side of the skip tests), u / v = pCamera->project(p3Dc), invz = 1 / p3Dc(2), level = PredictScale.
// Writes match[nq] and n_fused[n_kf] (what Fuse returns when no point changes state during the call).
void orbo_fuse(int n_kf, const int32_t* feat_off, const KeyPoint* kp, const uint8_t* desc, const float* uright, const float* bounds_grid,
               int nlev, const float* scale, const float* inv_sigma2, const float* bf, const int32_t* kf_off, const uint8_t* point_desc,
               const int32_t* point, const uint8_t* valid, const float* u, const float* v, const float* invz_in, const int32_t* level,
               float th, int32_t* match, int32_t* n_fused)
{
    for (int k = 0; k < n_kf; ++k) {
        KeyFrame K;
        const int f0 = feat_off[k];
        fill_frame(K, kp + f0, desc + (size_t)f0 * 32, uright + f0, feat_off[k + 1] - f0, bounds_grid + 6 * k, scale + (size_t)nlev * k);
        K.mbf = bf[k];
        K.mvInvLevelSigma2 = inv_sigma2 + (size_t)nlev * k;
        KeyFrame* pKF = &K;
        const float& bfk = pKF->mbf;
        int nFused = 0;
        for (int i = kf_off[k]; i < kf_off[k + 1]; i++) {
            match[i] = -1;
            if (!valid[i]) continue;
            const float invz = invz_in[i];
            const float uv0 = u[i], uv1 = v[i];
            // Point must be inside the image
            if (!pKF->IsInImage(uv0, uv1)) continue;
            const float ur = uv0 - bfk * invz;
            const int nPredictedLevel = level[i];
            // Search in a radius
            const float radius = th * pKF->mvScaleFactors[nPredictedLevel];
            const std::vector<size_t> vIndices = pKF->GetFeaturesInArea(uv0, uv1, radius);
            if (vIndices.empty()) continue;
            // Match to the most similar keypoint in the radius
            const uint8_t* dMP = point_desc + (size_t)point[i] * 32;
            int bestDist = 256;
            int bestIdx = -1;
            for (std::vector<size_t>::const_iterator vit = vIndices.begin(), vend = vIndices.end(); vit != vend; vit++) {
                size_t idx = *vit;
                const KeyPoint& kp = pKF->mvKeysUn[idx];
                const int& kpLevel = kp.octave;
                if (kpLevel < nPredictedLevel - 1 || kpLevel > nPredictedLevel) continue;
                if (pKF->mvuRight[idx] >= 0) {
                    // Check reprojection error in stereo
                    const float& kpx = kp.x;
                    const float& kpy = kp.y;
                    const float& kpr = pKF->mvuRight[idx];
                    const float ex = uv0 - kpx;
                    const float ey = uv1 - kpy;
                    const float er = ur - kpr;
                    const float e2 = ex * ex + ey * ey + er * er;
                    if (e2 * pKF->mvInvLevelSigma2[kpLevel] > 7.8) continue;
                } else {
                    const float& kpx = kp.x;
                    const float& kpy = kp.y;
                    const float ex = uv0 - kpx;
                    const float ey = uv1 - kpy;
                    const float e2 = ex * ex + ey * ey;
                    if (e2 * pKF->mvInvLevelSigma2[kpLevel] > 5.99) continue;
                }
                const uint8_t* dKF = pKF->mDescriptors + idx * 32;
                const int dist = DescriptorDistance(dMP, dKF);
                if (dist < bestDist) {
                    bestDist = dist;
                    bestIdx = (int)idx;
                }
            }
            // If there is already a MapPoint replace otherwise add new measurement: the caller's bookkeeping
            if (bestDist <= TH_LOW) {
                match[i] = bestIdx;
                nFused++;
            }
        }
        n_fused[k] = nFused;
    }
}

}  // extern "C"
