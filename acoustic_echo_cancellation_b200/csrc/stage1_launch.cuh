// Launcher glue between the C ABI and the templated stage-1 kernels.  The kernels are built in the nine
// stage1_inst_*.cu units (split so that the build parallelises); each unit is one look-up function that lists its
// builds, one AEC_STAGE1_BUILD line per build, and returns the launch function of the build a call asks for.
#pragma once
#include <cuda_runtime.h>

#include "stage1_kernel.cuh"

namespace aec {

using Stage1Launch = cudaError_t (*)(const Stage1Params& prm, cudaStream_t s);

// Configures KERNEL once per device and thread, then launches one CTA of NT threads per utterance.  KERNEL is a template
// argument so that every build keeps its own "configured" state: all builds of a kernel family share one function type.
template <void (*KERNEL)(Stage1Params), int NT, size_t SMEM>
cudaError_t launch_stage1(const Stage1Params& prm, cudaStream_t s) {
    static thread_local int configured_dev = -1;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (configured_dev != dev) {
        e = cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
        if (e != cudaSuccess) return e;
        // The kernels keep their tables in shared memory / registers and do not need L1: ask for the largest carve-out
        // so that 7 two-warp utterances (31.8 KB each) fit on one SM ...
        e = cudaFuncSetAttribute(KERNEL, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e != cudaSuccess) return e;
        // ... but no larger than the resident utterances need: the long-filter kernels (2 utterances of 60-90 KB per SM)
        // and the 128-register overlap-save builds still spill a few registers, and what is left of the 256 KB array
        // serves those reloads from L1 instead of L2.
        int resident = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, KERNEL, NT, SMEM);
        if (e != cudaSuccess) return e;
        if (resident > 0) {
            const size_t need = size_t(resident) * (SMEM + 1024);
            int pct = static_cast<int>((need * 100 + 228 * 1024 - 1) / (228 * 1024));
            pct = pct > 100 ? 100 : pct;
            e = cudaFuncSetAttribute(KERNEL, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
            if (e != cudaSuccess) return e;
        }
        configured_dev = dev;
    }
    KERNEL<<<dim3((unsigned)prm.B), dim3(NT), SMEM, s>>>(prm);
    return cudaGetLastError();
}

// The look-up of one unit: the launch function of the first build listed for (P, algo, echo) whose warp count equals nw
// and whose register cap equals regs, where nw = 0 or regs = 0 accepts any; nullptr when no build matches.  The first
// build listed for (P, algo, echo) is therefore its default.
Stage1Launch stage1_build_nw1(int P, int algo, bool echo, int nw, int regs);
Stage1Launch stage1_build_nw2(int P, int algo, bool echo, int nw, int regs);
Stage1Launch stage1_build_nw4(int P, int algo, bool echo, int nw, int regs);
Stage1Launch stage1_build_nw8(int P, int algo, bool echo, int nw, int regs);
Stage1Launch stage1_build_1024(int P, int algo, bool echo, int nw, int regs);
Stage1Launch stage1_build_feat(int P, int algo, bool echo, int nw, int regs);     // with the fused Stage-2 features
Stage1Launch stage1_build_ols(int P, int algo, bool echo, int nw, int regs);
Stage1Launch stage1_build_ols1024(int P, int algo, bool echo, int nw, int regs);
// streaming overlap-save builds (frame 512; the filter state crosses the call, OlsStreamState) and their state set-up:
// rows b with mask null or mask[b] != 0 of the B states at state + b * stride are reset (one launch)
Stage1Launch stage1_build_ols_stream(int P, int algo, bool echo, int nw, int regs);
cudaError_t ols_stream_state_init(void* state, long long B, long long stride, const uint8_t* mask, int P, bool kalman,
                                  float c0, cudaStream_t s);

// One build of a unit: NW warps per utterance, P partitions, algorithm, echo-estimate output, register cap.  Build<...>
// is the unit's kernel family: its kernel and dynamic shared memory, and, where the kernel fixes its warp count, a
// static_assert that NW is that count.
#define AEC_STAGE1_BUILD(NW_, P_, ALGO_, ECHO_, REGS_)                                                                  \
    if (P == (P_) && algo == (ALGO_) && echo == (ECHO_) && (nw == 0 || nw == (NW_)) && (regs == 0 || regs == (REGS_))) { \
        using B = Build<NW_, P_, ALGO_, ECHO_, REGS_>;                                                                  \
        return &launch_stage1<B::kernel, 32 * (NW_), B::smem>;                                                          \
    }

// Kernel family of the frame-512 STFT-domain units (stage1_inst_nw*.cu, and stage1_inst_feat.cu with FEAT)
template <int NW, int P, int ALGO, bool ECHO, int REGS, bool FEAT>
struct N512Build {
    static constexpr void (*kernel)(Stage1Params) = stage1_n512_kernel<NW, P, ALGO, ECHO, REGS, FEAT>;
    static constexpr size_t smem = FEAT ? Stage1Smem<NW, P>::total_feat(ECHO) : Stage1Smem<NW, P>::total(ECHO);
};

}  // namespace aec
