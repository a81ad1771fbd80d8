// Builds: 1 warp per utterance (4 mirrored-bin pairs per thread, no block barriers beyond the warp), chunk = 2 frames.
// Tuning variants for short filters.
#include "stage1_launch.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
using Build = N512Build<NW, P, ALGO, ECHO, REGS, false>;
}

Stage1Launch stage1_build_nw1(int P, int algo, bool echo, int nw, int regs) {
    AEC_STAGE1_BUILD(1, 4, kAlgoNlms, false, 255)
    AEC_STAGE1_BUILD(1, 4, kAlgoNlms, false, 200)
    return nullptr;
}

}  // namespace aec
