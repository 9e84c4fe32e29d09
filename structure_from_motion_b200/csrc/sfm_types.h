// Plain types that the host code and the kernels of more than one stage share: the selection record, the model
// kinds, the pose candidates and the models of the model selection.  No device code, so host-only translation units
// (sfm_nccl.cpp, through sfm_host.h) can include it too.
#pragma once
#include <cstdint>

namespace sfm {

// The model K3 selects among: the essential matrix (8-point samples, SED in K-normalised coordinates) or the homography
// (4-point samples, symmetric transfer error in pixels; sfm_homography.cuh).  The kind fixes the sample size and the
// exact scorer of the sample rule and of the rescore; the selection rule itself is the same.
enum { MODEL_E = 0, MODEL_H = 1 };

struct Best {
    double err;
    long long idx;
    int count;
    int pad;
};

struct SelectRecord {
    Best best;
    long long num_invalid, first_invalid;
    double E[9];
    int32_t sample[8];  // the winner's minimal sample (its table row; ransac.py:63), -1 without a table or a winner
};

// The four pose candidates in the reference's enumeration order
// (lib/epipolar/eight_point.py:210-212): (R1,t), (R1,-t), (R2,t), (R2,-t).
struct PoseSet {
    double R[4][9];
    double t[4][3];
    double sv[3];  // singular values of E, descending
    long long counts[4];
    int best;  // argmax of counts (first maximum), -1 until voted
    int pad;
};

// the models of one pair, row-major; a model not given is never read
struct SelectModels {
    double E[9], H[9], K[9];
    int have_e, have_h;
};

}  // namespace sfm
