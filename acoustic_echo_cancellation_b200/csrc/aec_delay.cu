// Far-end bulk-delay estimator (GCC-PHAT over the whole utterance) and far-end shift: aec_delay_estimate,
// aec_delay_align.  Definition: oracle/delay_oracle.py and DESIGN.md "Far-end delay estimation".
//
// Estimator: one CTA per utterance, so a row's outputs never depend on the batch around it.  For every block s of
// D samples the CTA transforms the far-end window x~[(s-1)D, (s+1)D) and the microphone window [0_D, y~[sD, (s+1)D)]
// (M = 2D real points each) as two D-point complex FFTs (even samples real, odd samples imaginary) in shared memory,
// splits them into the real spectra X_s, Y_s and adds Y_s conj(X_s) to S.  Thread t owns the bins k = t + i T of S in
// registers for the whole utterance (the block sum runs in one fixed order: deterministic).  The far-end samples of the
// current block stay in registers as the first half of the next window, so each input sample is read once.  After the
// last block: PHAT (G = S / |S|, DC and Nyquist zero), one inverse D-point FFT with the inverse real split, and a
// block argmax of |r[l]|, l = 0..D, with ties going to the smaller lag.
#include <cmath>

#include "aec_common.cuh"
#include "fft_warp.cuh"

namespace aec {
namespace {

constexpr int kDelayMinLog = 8;    // D = 256
constexpr int kDelayMaxLog = 13;   // D = 8192

template <int LOGD>
struct DelayShape {
    static constexpr int D = 1 << LOGD;                 // complex FFT length = half the real window M = 2D
    static constexpr int T = D / 2 < 1024 ? D / 2 : 1024;
    static constexpr int KPT = D / T;                   // bins of S per thread
    static constexpr int HP = (D / 2) / T;              // complex points (sample pairs) of one block per thread
    static constexpr size_t kSmem = 3 * (size_t)D * sizeof(float2);   // far FFT, mic FFT, twiddles w_M^k (k < D)
};

__device__ __forceinline__ float2 conjf2(float2 a) { return make_float2(a.x, -a.y); }

// In-place radix-2 DIT FFT of length D on one or two bit-reversed buffers; tw[k] = exp(-2 pi i k / 2D).
// Ends with a __syncthreads.
template <int LOGD, bool INV, bool TWO>
__device__ __forceinline__ void block_fft(float2* a, float2* c, const float2* tw, int tid) {
    using S = DelayShape<LOGD>;
#pragma unroll 1
    for (int h = 1; h < S::D; h <<= 1) {
        const int tstride = S::D / h;                   // w_{2h}^j = w_{2D}^{j D / h}
#pragma unroll
        for (int i = 0; i < S::HP; ++i) {
            const int q = tid + i * S::T;
            const int j = q & (h - 1);
            const int i0 = ((q - j) << 1) + j;
            float2 w = tw[j * tstride];
            if (INV) w.y = -w.y;
            {
                const float2 u = a[i0], v = cmul(a[i0 + h], w);
                a[i0] = cadd(u, v);
                a[i0 + h] = csub(u, v);
            }
            if (TWO) {
                const float2 u = c[i0], v = cmul(c[i0 + h], w);
                c[i0] = cadd(u, v);
                c[i0 + h] = csub(u, v);
            }
        }
        __syncthreads();
    }
}

template <int LOGD>
__device__ __forceinline__ int brev(int m) {
    return (int)(__brev((unsigned)m) >> (32 - LOGD));
}

// Real spectrum bin k (0 <= k < D) of the 2D-point real sequence whose even / odd samples are the real / imaginary
// parts of the D-point transform Z: U[k] = (Z[k] + conj Z[D-k]) / 2 - i w^k (Z[k] - conj Z[D-k]) / 2, w = e^{-2 pi i/2D}.
__device__ __forceinline__ float2 real_split(float2 zk, float2 zr, float2 w) {
    const float2 bc = conjf2(zr);
    const float2 e = make_float2(0.5f * (zk.x + bc.x), 0.5f * (zk.y + bc.y));
    const float2 o = make_float2(0.5f * (zk.y - bc.y), -0.5f * (zk.x - bc.x));   // -i (zk - bc) / 2
    return cadd(e, cmul(w, o));
}

// (value, lag) pair: b beats a when |r| is larger, or equal at a smaller lag
__device__ __forceinline__ bool beats(float bv, int bl, float av, int al) { return bv > av || (bv == av && bl < al); }

template <int LOGD>
__global__ void __launch_bounds__(DelayShape<LOGD>::T)
delay_estimate_kernel(const float* __restrict__ far, const float* __restrict__ mic, const long long* __restrict__ n_samples,
                      long long L, long long in_stride, int margin, float min_peak, int* __restrict__ delay_out,
                      int* __restrict__ shift_out, float* __restrict__ peak_out, float* __restrict__ corr) {
    using S = DelayShape<LOGD>;
    constexpr int D = S::D;
    extern __shared__ float2 smem[];
    float2* zf = smem;            // far-end window transform (later: G in natural order)
    float2* zm = smem + D;        // microphone window transform (later: the inverse transform)
    float2* tw = smem + 2 * D;    // w_M^k, k = 0..D-1
    __shared__ float red_v[32];
    __shared__ int red_l[32];

    const int tid = threadIdx.x;
    const long long b = blockIdx.x;
    long long n = L;
    if (n_samples) {
        n = n_samples[b];
        n = n < 0 ? 0 : (n > L ? L : n);
    }
    const float* x = far + b * in_stride;
    const float* y = mic + b * in_stride;

    for (int k = tid; k < D; k += S::T) {
        float sn, cs;
        sincospif((float)k / (float)D, &sn, &cs);       // angle -2 pi k / 2D, k / D exact
        tw[k] = make_float2(cs, -sn);
    }

    float2 acc[S::KPT];
#pragma unroll
    for (int i = 0; i < S::KPT; ++i) acc[i] = make_float2(0.f, 0.f);
    float2 prev[S::HP];           // far-end pairs of the previous block (x~ = 0 before the utterance)
#pragma unroll
    for (int i = 0; i < S::HP; ++i) prev[i] = make_float2(0.f, 0.f);

    const long long nblk = (n + D - 1) / D;
#pragma unroll 1
    for (long long s = 0; s < nblk; ++s) {
#pragma unroll
        for (int i = 0; i < S::HP; ++i) {
            const int m = tid + i * S::T;                     // pair index inside the block, 0 .. D/2 - 1
            const long long p = s * D + 2 * m;
            const float2 xv = make_float2(p < n ? x[p] : 0.f, p + 1 < n ? x[p + 1] : 0.f);
            const float2 yv = make_float2(p < n ? y[p] : 0.f, p + 1 < n ? y[p + 1] : 0.f);
            zf[brev<LOGD>(m)] = prev[i];
            zf[brev<LOGD>(m + D / 2)] = xv;
            zm[brev<LOGD>(m)] = make_float2(0.f, 0.f);
            zm[brev<LOGD>(m + D / 2)] = yv;
            prev[i] = xv;
        }
        __syncthreads();
        block_fft<LOGD, false, true>(zf, zm, tw, tid);
#pragma unroll
        for (int i = 0; i < S::KPT; ++i) {
            const int k = tid + i * S::T;
            const int kr = (D - k) & (D - 1);
            const float2 w = tw[k];
            const float2 X = real_split(zf[k], zf[kr], w);
            const float2 Y = real_split(zm[k], zm[kr], w);
            acc[i].x = fmaf(Y.y, X.y, fmaf(Y.x, X.x, acc[i].x));     // += Y conj(X)
            acc[i].y = fmaf(Y.y, X.x, fmaf(-Y.x, X.y, acc[i].y));
        }
        __syncthreads();
    }

    // PHAT weighting; G[0] = 0 (bin 0 is owned by thread 0, i = 0), G[D] is never formed
#pragma unroll
    for (int i = 0; i < S::KPT; ++i) {
        const int k = tid + i * S::T;
        const float a = hypotf(acc[i].x, acc[i].y);
        acc[i] = (k == 0 || !(a > 0.f)) ? make_float2(0.f, 0.f) : make_float2(acc[i].x / a, acc[i].y / a);
        zf[k] = acc[i];
    }
    __syncthreads();
    // inverse real split: Z'[k] = (G[k] + conj G[D-k]) + i w^-k (G[k] - conj G[D-k]); z = IFFT_D(Z') gives
    // r[2m] + i r[2m+1] = z[m] / M  (G[D] = 0, so bin 0 reads G[0] for it: both zero)
#pragma unroll
    for (int i = 0; i < S::KPT; ++i) {
        const int k = tid + i * S::T;
        const float2 g = acc[i];
        const float2 bc = conjf2(zf[(D - k) & (D - 1)]);
        const float2 e = cadd(g, bc), o = csub(g, bc);
        const float2 wo = cmulc(o, tw[k]);                         // o * conj(w)
        zm[brev<LOGD>(k)] = make_float2(e.x - wo.y, e.y + wo.x);   // e + i wo
    }
    __syncthreads();
    block_fft<LOGD, true, false>(zm, nullptr, tw, tid);

    constexpr float kInvM = 1.0f / (float)(2 * D);
    float best_v = -1.f;
    int best_l = 0x7fffffff;
    float* crow = corr ? corr + b * (long long)(D + 1) : nullptr;
    for (int m = tid; m <= D / 2; m += S::T) {
        const float2 z = zm[m];
        const float r0 = z.x * kInvM, r1 = z.y * kInvM;
        const int l0 = 2 * m;
        if (beats(fabsf(r0), l0, best_v, best_l)) { best_v = fabsf(r0); best_l = l0; }
        if (crow) crow[l0] = r0;
        if (l0 + 1 <= D) {
            if (beats(fabsf(r1), l0 + 1, best_v, best_l)) { best_v = fabsf(r1); best_l = l0 + 1; }
            if (crow) crow[l0 + 1] = r1;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best_v, o);
        const int ol = __shfl_xor_sync(0xffffffffu, best_l, o);
        if (beats(ov, ol, best_v, best_l)) { best_v = ov; best_l = ol; }
    }
    constexpr int kWarps = S::T / 32;
    if ((tid & 31) == 0) {
        red_v[tid >> 5] = best_v;
        red_l[tid >> 5] = best_l;
    }
    __syncthreads();
    if (tid == 0) {
        float bv = red_v[0];
        int bl = red_l[0];
        for (int w = 1; w < kWarps; ++w)
            if (beats(red_v[w], red_l[w], bv, bl)) { bv = red_v[w]; bl = red_l[w]; }
        const int sh = bv >= min_peak ? (bl - margin > 0 ? bl - margin : 0) : 0;
        if (delay_out) delay_out[b] = bl;
        if (peak_out) peak_out[b] = bv;
        shift_out[b] = sh;
    }
}

// far_out[b][n] = far[b][n - shift[b]] for shift[b] <= n < L, 0 below; grid (B, column chunks)
__global__ void __launch_bounds__(256)
delay_align_kernel(const float* __restrict__ far, float* __restrict__ far_out, const int* __restrict__ shift,
                   long long L, long long in_stride, long long out_stride) {
    const long long b = blockIdx.x;
    long long s = shift[b];
    if (s < 0) s = 0;
    const float* x = far + b * in_stride;
    float* o = far_out + b * out_stride;
    const long long step = (long long)gridDim.y * blockDim.x;
    for (long long i = (long long)blockIdx.y * blockDim.x + threadIdx.x; i < L; i += step)
        o[i] = i >= s ? x[i - s] : 0.f;
}

template <int LOGD>
cudaError_t launch_estimate(const float* far, const float* mic, const long long* n, long long B, long long L,
                            long long in_stride, int margin, float min_peak, int* delay, int* shift, float* peak,
                            float* corr, cudaStream_t s) {
    using S = DelayShape<LOGD>;
    static_assert(S::kSmem <= 227 * 1024 - 256, "shared memory");
    auto k = delay_estimate_kernel<LOGD>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::kSmem);
    if (e != cudaSuccess) return e;
    k<<<(unsigned)B, S::T, S::kSmem, s>>>(far, mic, n, L, in_stride, margin, min_peak, delay, shift, peak, corr);
    return cudaGetLastError();
}

}  // namespace

int validate_delay_cfg(const aec_delay_cfg* dcfg) {
    if (!dcfg) return AEC_EINVAL;
    const int D = dcfg->max_delay;
    if (D < (1 << kDelayMinLog) || D > (1 << kDelayMaxLog) || (D & (D - 1))) return AEC_EINVAL;
    if (dcfg->margin < 0) return AEC_EINVAL;
    if (std::isnan(dcfg->min_peak)) return AEC_EINVAL;
    return AEC_OK;
}

}  // namespace aec

using namespace aec;

extern "C" int aec_delay_cfg_default(aec_delay_cfg* dcfg) {
    if (!dcfg) return AEC_EINVAL;
    *dcfg = aec_delay_cfg{};
    dcfg->max_delay = 8192;
    dcfg->margin = 128;
    dcfg->min_peak = 0.1f;
    return AEC_OK;
}

extern "C" int aec_delay_estimate(const float* far, const float* mic, const int64_t* n_samples, int64_t B, int64_t L,
                                  int64_t in_stride, const aec_delay_cfg* dcfg, int32_t* delay, int32_t* shift,
                                  float* peak, float* corr, void* cuda_stream) {
    const int rc = validate_delay_cfg(dcfg);
    if (rc != AEC_OK) return rc;
    if (B < 0 || L < 0 || in_stride < L) return AEC_EINVAL;
    if (B == 0) return AEC_OK;
    if (!far || !mic || !shift) return AEC_EINVAL;
    if (B > 0x7fffffffLL) return AEC_EINVAL;
    cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
    const long long* n = reinterpret_cast<const long long*>(n_samples);
    cudaError_t e = cudaErrorInvalidValue;
    switch (__builtin_ctz((unsigned)dcfg->max_delay)) {
        case 8: e = launch_estimate<8>(far, mic, n, B, L, in_stride, dcfg->margin, dcfg->min_peak, delay, shift, peak, corr, s); break;
        case 9: e = launch_estimate<9>(far, mic, n, B, L, in_stride, dcfg->margin, dcfg->min_peak, delay, shift, peak, corr, s); break;
        case 10: e = launch_estimate<10>(far, mic, n, B, L, in_stride, dcfg->margin, dcfg->min_peak, delay, shift, peak, corr, s); break;
        case 11: e = launch_estimate<11>(far, mic, n, B, L, in_stride, dcfg->margin, dcfg->min_peak, delay, shift, peak, corr, s); break;
        case 12: e = launch_estimate<12>(far, mic, n, B, L, in_stride, dcfg->margin, dcfg->min_peak, delay, shift, peak, corr, s); break;
        case 13: e = launch_estimate<13>(far, mic, n, B, L, in_stride, dcfg->margin, dcfg->min_peak, delay, shift, peak, corr, s); break;
    }
    if (e != cudaSuccess) {
        set_cuda_error(e, "aec_delay_estimate launch");
        return AEC_ECUDA;
    }
    count_launch();
    return AEC_OK;
}

extern "C" int aec_delay_align(const float* far, float* far_out, const int32_t* shift, int64_t B, int64_t L,
                               int64_t in_stride, int64_t out_stride, void* cuda_stream) {
    if (B < 0 || L < 0 || in_stride < L || out_stride < L) return AEC_EINVAL;
    if (B == 0) return AEC_OK;
    if (!far || !far_out || !shift || far == far_out) return AEC_EINVAL;
    if (B > 0x7fffffffLL) return AEC_EINVAL;
    if (L == 0) return AEC_OK;
    long long chunks = (L + 2047) / 2048;
    if (chunks > 65535) chunks = 65535;
    delay_align_kernel<<<dim3((unsigned)B, (unsigned)chunks), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        far, far_out, reinterpret_cast<const int*>(shift), L, in_stride, out_stride);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_cuda_error(e, "aec_delay_align launch");
        return AEC_ECUDA;
    }
    count_launch();
    return AEC_OK;
}
