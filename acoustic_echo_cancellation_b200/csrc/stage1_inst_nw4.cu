// Builds: 4 warps per utterance (1 mirrored-bin pair per thread), chunk = 8 frames.
#include "stage1_launch.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
using Build = N512Build<NW, P, ALGO, ECHO, REGS, false>;
}

Stage1Launch stage1_build_nw4(int P, int algo, bool echo, int nw, int regs) {
    AEC_STAGE1_BUILD(4, 8, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoNlms, false, 168)
    AEC_STAGE1_BUILD(4, 8, kAlgoNlms, true, 168)
    AEC_STAGE1_BUILD(4, 8, kAlgoKalman, false, 168)
    AEC_STAGE1_BUILD(4, 8, kAlgoKalman, true, 168)
    AEC_STAGE1_BUILD(4, 16, kAlgoNlms, false, 255)
    AEC_STAGE1_BUILD(4, 16, kAlgoNlms, true, 255)
    AEC_STAGE1_BUILD(4, 16, kAlgoKalman, false, 255)
    AEC_STAGE1_BUILD(4, 16, kAlgoKalman, true, 255)
    AEC_STAGE1_BUILD(4, 4, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(4, 4, kAlgoNlms, false, 96)
    return nullptr;
}

}  // namespace aec
