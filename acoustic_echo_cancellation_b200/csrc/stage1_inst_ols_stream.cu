// Builds of the streaming overlap-save kernel (stage1_ols_stream_kernel: the body of stage1_ols_kernel with the filter
// state loaded from and stored to HBM, aec_stage1_run_stream), one per (P, algo, echo) at 128 registers, and the kernel
// that initialises the state blocks (aec_stage1_state_init).
#include "stage1_ols_kernel.cuh"
#include "stage1_launch.cuh"

namespace aec {
namespace {
template <int NW, int P, int ALGO, bool ECHO, int REGS>
struct Build {
    static_assert(NW == OlsShape<P>::NW, "the overlap-save warp count follows from P");
    static constexpr bool KAL = ALGO == kAlgoPbfkf;
    static constexpr void (*kernel)(Stage1Params) = stage1_ols_stream_kernel<P, KAL, ECHO, REGS>;
    static constexpr size_t smem = OlsSmem::total(P, KAL);
};

// Row b (where mask is null or mask[b] != 0): every byte of the state zero, except C = c0 (Kalman step).
__global__ void __launch_bounds__(256) ols_state_init_kernel(unsigned char* state, long long stride, const uint8_t* mask,
                                                             int P, int kalman, float c0) {
    const long long b = blockIdx.x;
    if (mask && !mask[b]) return;
    float* row = reinterpret_cast<float*>(state + b * stride);
    const long long n = OlsStreamState::bytes(P, kalman != 0) / 4;
    const long long c_begin = OlsStreamState::C(P) / 4, c_end = c_begin + (long long)P * OlsStreamState::K;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) row[i] = (kalman && i >= c_begin && i < c_end) ? c0 : 0.f;
}
}  // namespace

Stage1Launch stage1_build_ols_stream(int P, int algo, bool echo, int nw, int regs) {
    AEC_STAGE1_BUILD(2, 1, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(2, 1, kAlgoPbfkf, true, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(2, 2, kAlgoPbfkf, true, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(2, 4, kAlgoPbfkf, true, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(4, 8, kAlgoPbfkf, true, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoPbfdaf, false, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoPbfdaf, true, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoPbfkf, false, 128)
    AEC_STAGE1_BUILD(8, 16, kAlgoPbfkf, true, 128)
    return nullptr;
}

cudaError_t ols_stream_state_init(void* state, long long B, long long stride, const uint8_t* mask, int P, bool kalman,
                                  float c0, cudaStream_t s) {
    ols_state_init_kernel<<<dim3((unsigned)B), dim3(256), 0, s>>>(static_cast<unsigned char*>(state), stride, mask, P,
                                                                   kalman ? 1 : 0, c0);
    return cudaGetLastError();
}

}  // namespace aec
