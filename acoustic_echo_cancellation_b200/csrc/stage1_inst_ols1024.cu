// Builds of the frame-1024 overlap-save PBFDAF kernel (kAlgoPbfdaf / kAlgoPbfkf; 4 partitions: four warps per
// utterance, 8: eight).
#include "stage1_launch.cuh"
#include "stage1_ols1024_kernel.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
struct Build {
    static_assert(NW == Ols1024Shape<P>::NW, "the frame-1024 overlap-save warp count follows from P");
    static constexpr void (*kernel)(Stage1Params) = stage1_ols1024_kernel<P, ALGO == kAlgoPbfkf, ECHO, REGS>;
    static constexpr size_t smem = Ols1024Shape<P>::total;
};
}

Stage1Launch stage1_build_ols1024(int P, int algo, bool echo, int nw, int regs) {
    AEC_STAGE1_BUILD(8, 8, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoPbfkf, true, 128)
    AEC_STAGE1_BUILD(4, 4, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(4, 4, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(4, 4, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(4, 4, kAlgoPbfkf, true, 128)
    return nullptr;
}

}  // namespace aec
