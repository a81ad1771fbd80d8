// Builds: 8 warps per utterance, ONE bin per thread, chunk = 16 frames -- long filters (the per-bin state W_p, X[t-p],
// C_p of a 16-partition Kalman filter is 81 registers).
#include "stage1_launch.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
using Build = N512Build<NW, P, ALGO, ECHO, REGS, false>;
}

Stage1Launch stage1_build_nw8(int P, int algo, bool echo, int nw, int regs) {
    AEC_STAGE1_BUILD(8, 16, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoKalman, true, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoNlms, true, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoKalman, true, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoNlms, true, 128)
    return nullptr;
}

}  // namespace aec
