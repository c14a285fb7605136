// init_oracle.cpp — CPU ORACLE (TEST INFRASTRUCTURE ONLY, never shipped, never on the product path).
//
// Line-by-line restatement of ORBmatcher::SearchForInitialization (src/ORBmatcher1.cc:650-765, called by
// Tracking::MonocularInitialization, src/Tracking3.cc:740-741) over the projection oracle's own Frame / GetFeaturesInArea /
// ComputeThreeMaxima / DescriptorDistance, which this file compiles in unchanged (oracle/projection_oracle.cpp is included, not
// copied).  Built on demand by tests/init_oracle.py into build/.
#include <climits>

#include "../../oracle/projection_oracle.cpp"

namespace {
constexpr int TH_LOW = 50;            // src/ORBmatcher1.cc:37
}  // namespace

extern "C" {

// F1 = (kp1, desc1, n1): mvKeysUn / mDescriptors; F2 = (kp2, desc2, n2) on the grid bounds_grid (mnMinX, mnMinY, mnMaxX, mnMaxY,
// mfGridElementWidthInv, mfGridElementHeightInv).  vbPrevMatched = prev [n1][2], in/out.  Writes vnMatches12 [n1]; returns nmatches.
int orbo_search_for_initialization(const KeyPoint* kp1, const uint8_t* desc1, int n1, const KeyPoint* kp2, const uint8_t* desc2, int n2,
                                   const float* bounds_grid, float* prev, int windowSize, float mfNNratio, int mbCheckOrientation,
                                   int32_t* vnMatches12_out)
{
    Frame F2;
    fill_frame(F2, kp2, desc2, nullptr, n2, bounds_grid, nullptr);
    int nmatches = 0;
    std::vector<int> vnMatches12(n1, -1);
    std::vector<int> rotHist[HISTO_LENGTH];
    for (int i = 0; i < HISTO_LENGTH; i++) rotHist[i].reserve(500);
    const float factor = 1.0f / HISTO_LENGTH;
    std::vector<int> vMatchedDistance(n2, INT_MAX);
    std::vector<int> vnMatches21(n2, -1);
    for (int i1 = 0; i1 < n1; i1++) {
        const KeyPoint kp = kp1[i1];
        const int level1 = kp.octave;
        if (level1 > 0) continue;
        const std::vector<size_t> vIndices2 = F2.GetFeaturesInArea(prev[2 * i1], prev[2 * i1 + 1], windowSize, level1, level1);
        if (vIndices2.empty()) continue;
        const uint8_t* d1 = desc1 + (size_t)i1 * 32;
        int bestDist = INT_MAX;
        int bestDist2 = INT_MAX;
        int bestIdx2 = -1;
        for (auto vit = vIndices2.begin(); vit != vIndices2.end(); vit++) {
            const size_t i2 = *vit;
            const uint8_t* d2 = F2.mDescriptors + i2 * 32;
            const int dist = DescriptorDistance(d1, d2);
            if (vMatchedDistance[i2] <= dist) continue;
            if (dist < bestDist) {
                bestDist2 = bestDist;
                bestDist = dist;
                bestIdx2 = (int)i2;
            } else if (dist < bestDist2) {
                bestDist2 = dist;
            }
        }
        if (bestDist <= TH_LOW) {
            if (bestDist < (float)bestDist2 * mfNNratio) {
                if (vnMatches21[bestIdx2] >= 0) {
                    vnMatches12[vnMatches21[bestIdx2]] = -1;
                    nmatches--;
                }
                vnMatches12[i1] = bestIdx2;
                vnMatches21[bestIdx2] = i1;
                vMatchedDistance[bestIdx2] = bestDist;
                nmatches++;
                if (mbCheckOrientation) {
                    float rot = kp1[i1].angle - F2.mvKeysUn[bestIdx2].angle;
                    if (rot < 0.0) rot += 360.0f;
                    int bin = round(rot * factor);
                    if (bin == HISTO_LENGTH) bin = 0;
                    if (bin < 0 || bin >= HISTO_LENGTH) return -1;   // the reference asserts here
                    rotHist[bin].push_back(i1);
                }
            }
        }
    }
    if (mbCheckOrientation) {
        int ind1 = -1;
        int ind2 = -1;
        int ind3 = -1;
        ComputeThreeMaxima(rotHist, HISTO_LENGTH, ind1, ind2, ind3);
        for (int i = 0; i < HISTO_LENGTH; i++) {
            if (i == ind1 || i == ind2 || i == ind3) continue;
            for (size_t j = 0, jend = rotHist[i].size(); j < jend; j++) {
                const int idx1 = rotHist[i][j];
                if (vnMatches12[idx1] >= 0) {
                    vnMatches12[idx1] = -1;
                    nmatches--;
                }
            }
        }
    }
    // Update prev matched
    for (int i1 = 0; i1 < n1; i1++)
        if (vnMatches12[i1] >= 0) { prev[2 * i1] = F2.mvKeysUn[vnMatches12[i1]].x; prev[2 * i1 + 1] = F2.mvKeysUn[vnMatches12[i1]].y; }
    for (int i1 = 0; i1 < n1; i1++) vnMatches12_out[i1] = vnMatches12[i1];
    return nmatches;
}

}  // extern "C"
