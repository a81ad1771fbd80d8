// Builds of the frame-1024 (48 kHz) kernel: 8 warps, one mirrored pair per thread.
#include "stage1_kernel_1024.cuh"
#include "stage1_launch.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
struct Build {
    static_assert(NW == Stage1Smem1024::NW, "the frame-1024 kernel runs 8 warps per utterance");
    static constexpr void (*kernel)(Stage1Params) = stage1_n1024_kernel<P, ALGO, ECHO, REGS>;
    static constexpr size_t smem = Stage1Smem1024::total(ECHO, P);
};
}

Stage1Launch stage1_build_1024(int P, int algo, bool echo, int nw, int regs) {
    AEC_STAGE1_BUILD(8, 8, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoNlms, true, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(8, 8, kAlgoKalman, true, 128)
    AEC_STAGE1_BUILD(8, 4, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(8, 4, kAlgoNlms, true, 128)
    AEC_STAGE1_BUILD(8, 4, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(8, 4, kAlgoKalman, true, 128)
    AEC_STAGE1_BUILD(8, 2, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(8, 2, kAlgoNlms, true, 128)
    AEC_STAGE1_BUILD(8, 2, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(8, 2, kAlgoKalman, true, 128)
    AEC_STAGE1_BUILD(8, 1, kAlgoNlms, false, 128)
    AEC_STAGE1_BUILD(8, 1, kAlgoNlms, true, 128)
    AEC_STAGE1_BUILD(8, 1, kAlgoKalman, false, 128)
    AEC_STAGE1_BUILD(8, 1, kAlgoKalman, true, 128)
    return nullptr;
}

}  // namespace aec
