// Builds of the two-warp kernel WITH the fused Stage-2 feature epilogue (SURVEY 8f rank 2): the error signal is
// re-analysed on chip one frame behind its synthesis and cat[err_erb, |err_erb - far_erb|] is emitted next to it.
// 43.9 KB of shared memory per utterance -> 5 utterances per SM; the register cap that goes with five two-warp
// utterances is 168: registers are per scheduler (16 K each) and five utterances put three warps on two of the four
// schedulers -- at the first cut's cap of 200 ncu showed 4 utterances per SM (profiles/r2_fused_ncu_summary.md).
// (The plain kernel runs seven per SM at 128.)  The Kalman filter spills at 168 and stays at 200.  Which of the two
// 4-partition NLMS builds runs follows from the batch size (stage1_run_impl in aec_capi.cu).
#include "stage1_launch.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
using Build = N512Build<NW, P, ALGO, ECHO, REGS, true>;
}

Stage1Launch stage1_build_feat(int P, int algo, bool echo, int nw, int regs) {
    AEC_STAGE1_BUILD(2, 4, kAlgoNlms, false, 168)
    AEC_STAGE1_BUILD(2, 4, kAlgoNlms, false, 200)
    AEC_STAGE1_BUILD(2, 4, kAlgoKalman, false, 200)
    AEC_STAGE1_BUILD(2, 2, kAlgoNlms, false, 168)
    AEC_STAGE1_BUILD(2, 1, kAlgoNlms, false, 168)
    return nullptr;
}

}  // namespace aec
