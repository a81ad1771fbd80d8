// Builds of the overlap-save PBFDAF kernel (kAlgoPbfdaf: NLMS step, kAlgoPbfkf: Kalman step): two warps per utterance
// for 1-4 partitions, four for 8, eight for 16 (OlsShape).
#include "stage1_ols_kernel.cuh"
#include "stage1_launch.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
struct Build {
    static_assert(NW == OlsShape<P>::NW, "the overlap-save warp count follows from P");
    static constexpr bool KAL = ALGO == kAlgoPbfkf;
    static constexpr void (*kernel)(Stage1Params) = stage1_ols_kernel<P, KAL, ECHO, REGS>;
    static constexpr size_t smem = OlsSmem::total(P, KAL);
};
}

Stage1Launch stage1_build_ols(int P, int algo, bool echo, int nw, int regs) {
    // 128 registers (8 utterances per SM) by default.  The Kalman step keeps the far-end history in shared memory
    // (OlsSmem::ring), which is what lets its 20 extra state registers fit: 2.85 ms per 1024 x 10 s, 11.5 ms per 4096
    // (history in registers: 3.4 / 12.4 ms at 128 registers with spills, 4.7 / 11.9 ms at 168 without).
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfkf, true, 128)
    // The 168-register Kalman builds stay available as variant 2168.
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfkf, false, 168)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfkf, true, 168)
    // NLMS step at 168 registers, spill-free: 6 % shorter block latency -- 3660 against 3900 cycles alone on an SM --
    // which does not pay for 6 instead of 8 resident utterances; variant 2168.
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfdaf, false, 168)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfdaf, true, 168)
    AEC_STAGE1_BUILD(8, 16, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoPbfkf, true, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoPbfkf, true, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoPbfkf, true, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoPbfkf, true, 128)
    return nullptr;
}

}  // namespace aec
