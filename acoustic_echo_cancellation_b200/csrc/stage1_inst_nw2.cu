// Builds: 2 warps per utterance (2 mirrored-bin pairs per thread), chunk = 4 frames.  128 registers is the largest cap
// that keeps 7 two-warp utterances resident per SM (16 K registers per scheduler).
#include "stage1_launch.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
using Build = N512Build<NW, P, ALGO, ECHO, REGS, false>;
}

Stage1Launch stage1_build_nw2(int P, int algo, bool echo, int nw, int regs) {
    AEC_STAGE1_BUILD(2, 4, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoNlms, false, 168)
    AEC_STAGE1_BUILD(2, 4, kAlgoNlms, true, 168)       // echo output: 33 KB smem -> 6 per SM anyway
    AEC_STAGE1_BUILD(2, 4, kAlgoKalman, false, 168)
    AEC_STAGE1_BUILD(2, 4, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoKalman, true, 200)
    AEC_STAGE1_BUILD(2, 1, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoNlms, true, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoKalman, true, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoNlms, true, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoKalman, true, 128)
    return nullptr;
}

}  // namespace aec
