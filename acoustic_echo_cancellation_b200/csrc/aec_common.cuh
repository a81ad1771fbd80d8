// Shared host-side helpers of the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/aec_b200.h"

namespace aec {

// Constant tables living in device global memory (one copy per device / context).
struct Tables {
    const float2* tw256;   // [16][16]  exp(-2 pi i h q / 256) at [q*16 + h]
    const float2* tw512;   // [129]     exp(-2 pi i k / 512)
    const float2* win_a;   // [256]     0.5 * hann512[2m], 0.5 * hann512[2m+1]
    const float2* win_s;   // [256]     hann512[n] / (512 (coff[n] + 1e-8))
    const float2* win_r;   // [256]     hann512[n] / 512        (raw synthesis frame, for aec_istft)
    const float* hann512;  // [512]
    // frame-1024 kernels
    const float2* tw512w;  // [17][32]  rows 0..15: exp(-2 pi i l q / 512) at [q*32 + l]; row 16: exp(-2 pi i a / 32)
    const float2* tw1024;  // [257]     exp(-2 pi i k / 1024)
    const float2* win_a1k; // [256]     0.5 * hann1024[2m], 0.5 * hann1024[2m+1], m < 256
    const float2* win_s1k; // [512]     hann1024[n] / (1024 (coff[n] + 1e-8))
};

// Returns AEC_OK and the tables of the current device (lazily initialised, thread safe).
int get_tables(Tables* out);

void set_cuda_error(cudaError_t e, const char* where);
void count_launch(int n = 1);
// AEC_OK or AEC_EINVAL for an aec_delay_cfg (aec_delay.cu)
int validate_delay_cfg(const aec_delay_cfg* dcfg);

#define AEC_CUDA_CHECK(expr)                          \
    do {                                              \
        cudaError_t _e = (expr);                      \
        if (_e != cudaSuccess) {                      \
            ::aec::set_cuda_error(_e, #expr);         \
            return AEC_ECUDA;                         \
        }                                             \
    } while (0)

}  // namespace aec
