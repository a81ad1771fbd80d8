// Streaming Stage 2: the whole Little_net suppressor (aec_features + aec_stage2_mask + aec_stage2_synth, in_norm off) for
// the new hops of many live streams in one launch, with each stream's GRU state, last input hop and pending overlap-add
// half-frame carried in caller-owned device memory from one call to the next.
//
// Frame t of the reference STFT covers hops t-1 and t (hop -1 is zero); output block g is the second half of frame g plus
// the first half of frame g+1.  A row that consumes n hops computes frames T0 .. T0+n-1 and emits blocks T0-1 .. T0+n-2
// (block -1 is not part of the signal).  Every frame is computed with the arithmetic, in the order, of the one-shot
// kernels: the features of features512_kernel, the GRU / linears of stage2_mask_kernel, the gain, inverse transform and
// overlap-add of stage2_synth_kernel.  Where a frame falls in a call changes nothing, so a chunked stream gives the bits
// of one call over the whole stream.  (Against LittleNetInference(in_norm=False) the outputs agree to ~1e-7 relative, not
// always bit for bit: this unit is compiled on its own.)
//
// What is per frame -- the Little_net arithmetic shared with the one-shot kernels -- is defined once in stage2_net.cuh;
// this unit holds what streaming adds: the state layout, the persistent per-stream loop, framing from the carried
// previous hop, the overlap-add with the carried half-frame and the state epilogue.
#include <cstdint>

#include "aec_common.cuh"
#include "fft_warp.cuh"
#include "stage2_net.cuh"

namespace aec {
namespace {

using namespace s2;

constexpr int kHop = 256;
constexpr int kSW = 4;          // streams (warps) per CTA
constexpr int kCtasPerSm = 2;   // persistent grid: at most this many CTAs per SM, each walking streams

// One stream's state (include/aec_b200.h): byte offsets
struct S2State {
    static constexpr int kFrames = 0;      // int64 frames consumed (+ 8 reserved bytes)
    static constexpr int kHid = 16;        // float h[32]
    static constexpr int kMicPrev = 144;   // float mic_prev[256]
    static constexpr int kRefPrev = 1168;  // float ref_prev[256]
    static constexpr int kOla = 2192;      // float ola[256]
    static constexpr int kBytes = 3216;
};
static_assert(S2State::kBytes % 16 == 0 && S2State::kMicPrev % 16 == 0 && S2State::kRefPrev % 16 == 0 &&
              S2State::kOla % 16 == 0, "state fields on 16-byte boundaries");

// shared memory, in floats: CTA-wide weights and bank ranges, then one region per warp
constexpr int kBankFloats = 2 * kK + 2 * kK + 2 * kH;                     // c2 float2[257], blo/bhi[257], lo/hi[32]
constexpr int kTileF = 2 * 2 * kTilePitch;                                // two half-warp FFT tiles (float2)
constexpr int kMagP = 260;                                                // magnitude row pitch
constexpr int kWarpFloats = kTileF + 2 * kMagP + kCh * kIn + 3 * kCh * kH + kH + kHop;
constexpr size_t kSmemBytes = (size_t)(kWFloats + kBankFloats + kSW * kWarpFloats) * sizeof(float);
static_assert(kWFloats % 4 == 0 && kBankFloats % 4 == 0 && kWarpFloats % 4 == 0 && (kTileF + 2 * kMagP) % 4 == 0,
              "float4 / float2 regions must stay aligned");

// Windowed analysis of one frame into the half-warp's tile (tile[k] = Zc[k]): samples 0..255 from p0 (the previous hop),
// 256..511 from p1.  `vec`: both pointers 8-byte aligned.
__device__ __forceinline__ void analyse_hops(const float* p0, const float* p1, bool vec, float2* tile, const Tables& tab,
                                             int h) {
    float2 v[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float* p = (j < 8 ? p0 : p1) + 2 * h + 32 * (j & 7);
        const float2 wv = __ldg(&tab.win_a[h + 16 * j]);
        const float2 xv = vec ? *reinterpret_cast<const float2*>(p) : make_float2(p[0], p[1]);
        v[j] = make_float2(xv.x * wv.x, xv.y * wv.y);
    }
    __syncwarp();
    fft256_halfwarp<false>(v, tile, tab.tw256, h);
#pragma unroll
    for (int p = 0; p < 16; ++p) tile[h + 16 * fft16_index(p)] = v[p];
    __syncwarp();
}

__global__ void __launch_bounds__(kSW * 32, kCtasPerSm) stage2_stream_kernel(
    const float* __restrict__ mic, const float* __restrict__ ref, const float* __restrict__ erb, aec_stage2_weights w,
    float* __restrict__ out, const int64_t* __restrict__ n_samples, long long B, long long L, long long in_stride,
    long long out_stride, unsigned char* __restrict__ state, long long state_stride, Tables tab) {
    extern __shared__ __align__(16) float sm[];
    float2* c2 = reinterpret_cast<float2*>(sm + kWFloats);        // [257] first two coefficients of bin k's band range
    int* blo = reinterpret_cast<int*>(c2 + kK);                    // [257] band range of bin k
    int* bhi = blo + kK;
    int* lo = bhi + kK;                                            // [32]  bin range of band j
    int* hi = lo + kH;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = lane >> 4, h = lane & 15;
    // ---- weights and bank ranges, once per CTA ----
    stage_weights(sm, w, tid, blockDim.x);
    const BinBands bank{blo, bhi, c2, erb};
    bank.stage(tid, blockDim.x);
    band_bin_ranges(erb, kH, lo, hi, tid, blockDim.x);
    __syncthreads();

    float* wreg = sm + kWFloats + kBankFloats + warp * kWarpFloats;
    float2* tiles = reinterpret_cast<float2*>(wreg);               // [2][kTilePitch]: half-warp tiles
    float2* tile = tiles + half * kTilePitch;
    float* mag = wreg + kTileF;                                    // [2][kMagP]   |Z| of the mic / ref frame
    float* xs = mag + 2 * kMagP;                                   // [kCh][64]   the chunk's feature vectors
    float* hb = xs + kCh * kIn;                                    // [kCh][32]   h_t of the chunk
    float* os = hb + kCh * kH;                                     // [kCh][32]   linear1 outputs
    float* es = os + kCh * kH;                                     // [kCh][32]   est_erb of the chunk
    float* hs = es + kCh * kH;                                     // [32]        h_{t-1} broadcast buffer
    float* ola = hs + kH;                                          // [256]       pending second half-frame
    const NetLane net = NetLane::load(sm, w, lane);

    for (long long b = (long long)blockIdx.x * kSW + warp; b < B; b += (long long)gridDim.x * kSW) {
        long long n = n_samples ? n_samples[b] : L;
        n = n < 0 ? 0 : (n > L ? L : n);
        const long long nh = n / kHop;
        const float* xm = mic + b * in_stride;
        const float* xr = ref + b * in_stride;
        float* yb = out + b * out_stride;
        unsigned char* st = state + b * state_stride;
        float* st_h = reinterpret_cast<float*>(st + S2State::kHid);
        float* st_mp = reinterpret_cast<float*>(st + S2State::kMicPrev);
        float* st_rp = reinterpret_cast<float*>(st + S2State::kRefPrev);
        float* st_ola = reinterpret_cast<float*>(st + S2State::kOla);
        long long emitted = 0;
        if (nh > 0) {
            const long long T0 = *reinterpret_cast<const long long*>(st + S2State::kFrames);
            const long long g_first = T0 > 0 ? T0 - 1 : 0;      // the first block this call writes, at column 0
            const bool vec = (reinterpret_cast<uintptr_t>(xm) & 7) == 0 && (reinterpret_cast<uintptr_t>(xr) & 7) == 0;
            const float* xb = half == 0 ? xm : xr;
            const float* prev = half == 0 ? st_mp : st_rp;
            float hcur = st_h[lane];
#pragma unroll
            for (int i = 0; i < kHop / 32; ++i) ola[lane + 32 * i] = st_ola[lane + 32 * i];
            for (long long f0 = 0; f0 < nh; f0 += kCh) {
                const int nf = (int)((nh - f0) < kCh ? (nh - f0) : kCh);
                // ---- features of the chunk's frames (features512_kernel): half-warp 0 the mic, 1 the ref ----
                for (int f = 0; f < kCh; ++f) {
                    if (f < nf) {
                        const long long i = f0 + f;
                        analyse_hops(i == 0 ? prev : xb + (i - 1) * kHop, xb + i * kHop, vec, tile, tab, h);
                        float* mrow = mag + half * kMagP;
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const int k = h + 16 * q;
                            float2 xk, xm2;
                            unpack_pair(tile[k], tile[(256 - k) & 255], __ldg(&tab.tw512[k]), xk, xm2);
                            if (k == 0) {
                                xk.y = 0.f;
                                xm2.y = 0.f;
                            }
                            mrow[k] = sqrt_approx(fmaf(xk.x, xk.x, fmaf(xk.y, xk.y, 1e-9f)));        // ERB.py:277-278
                            mrow[256 - k] = sqrt_approx(fmaf(xm2.x, xm2.x, fmaf(xm2.y, xm2.y, 1e-9f)));
                        }
                        if (h == 0) {
                            float2 xk, xm2;
                            unpack_pair(tile[128], tile[128], make_float2(0.f, -1.f), xk, xm2);
                            mrow[128] = sqrt_approx(fmaf(xk.x, xk.x, fmaf(xk.y, xk.y, 1e-9f)));
                        }
                        __syncwarp();
                        // ERB projection, lane = band (ERB.py:282-283), then cat[mic_erb, |mic_erb - ref_erb|]
                        float am = 0.f, ar = 0.f;
                        for (int k = lo[lane]; k < hi[lane]; ++k) {
                            const float c = __ldg(erb + k * kH + lane);
                            am = fmaf(mag[k], c, am);
                            ar = fmaf(mag[kMagP + k], c, ar);
                        }
                        xs[f * kIn + lane] = am;
                        xs[f * kIn + kH + lane] = fabsf(am - ar);                                  // ERB.py:287-290
                        __syncwarp();
                    } else {
                        xs[f * kIn + lane] = 0.f;
                        xs[f * kIn + kH + lane] = 0.f;
                    }
                }
                __syncwarp();
                // ---- the GRU and linear layers of the chunk ----
                float gr[kCh], gz[kCh], gn[kCh], a1[kCh], a2[kCh];
                gru_inputs(net, sm, xs, lane, gr, gz, gn);
                gru_chunk(net, gr, gz, gn, hs, hb, hcur, nf, lane);
                __syncwarp();
                net_outputs(net, sm, xs, hb, os, lane, a1, a2);
#pragma unroll
                for (int f = 0; f < kCh; ++f) es[f * kH + lane] = sigmoidf_(a2[f]) * xs[f * kIn + lane];
                __syncwarp();
                // ---- synthesis (stage2_synth_kernel), two frames at a time: half-warp 0 frame f, 1 frame f + 1 ----
                for (int f = 0; f < nf; f += 2) {
                    const int ff = (f + half < nf) ? f + half : f;         // an odd last pair: both halves on frame f
                    const long long i = f0 + ff;
                    analyse_hops(i == 0 ? st_mp : xm + (i - 1) * kHop, xm + i * kHop, vec, tile, tab, h);
                    float2 v[16];
                    synth_frame(tile, bank, es, ff, tab, h, v);
                    __syncwarp();
#pragma unroll
                    for (int p = 0; p < 16; ++p) {
                        const int r = fft16_index(p);
                        const float2 wv = __ldg(&tab.win_s[h + 16 * r]);
                        tile[h + 16 * r] = make_float2(v[p].x * wv.x, v[p].y * wv.y);
                    }
                    __syncwarp();
                    // overlap-add (ERB.py:315-316): block t-1 = pending half + first half of frame t, + 1e-9
                    for (int s = 0; s < 2 && f + s < nf; ++s) {
                        const long long t = T0 + f0 + f + s;
                        const float2* fr = tiles + s * kTilePitch;
                        float2* ola2 = reinterpret_cast<float2*>(ola);
#pragma unroll
                        for (int m = lane; m < 128; m += 32) {
                            const float2 a = ola2[m], c = fr[m];
                            if (t >= 1) {
                                float* y = yb + (t - 1 - g_first) * kHop + 2 * m;
                                y[0] = a.x + c.x + 1e-9f;
                                y[1] = a.y + c.y + 1e-9f;
                            }
                            ola2[m] = fr[128 + m];
                        }
                        __syncwarp();
                    }
                }
            }
            // ---- epilogue: the state after frame T0 + nh - 1 ----
            st_h[lane] = hcur;
#pragma unroll
            for (int i = 0; i < kHop / 32; ++i) {
                const int m = lane + 32 * i;
                st_mp[m] = xm[(nh - 1) * kHop + m];
                st_rp[m] = xr[(nh - 1) * kHop + m];
                st_ola[m] = ola[m];
            }
            if (lane == 0) *reinterpret_cast<long long*>(st + S2State::kFrames) = T0 + nh;
            emitted = (T0 > 0 ? nh : nh - 1) * kHop;
            __syncwarp();
        }
        for (long long c = emitted + lane; c < L; c += 32) yb[c] = 0.f;      // zero past the row's blocks
    }
}

__global__ void stage2_stream_state_init_kernel(unsigned char* __restrict__ state, long long B, long long stride,
                                                const uint8_t* __restrict__ mask) {
    constexpr int kVec = S2State::kBytes / 16;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < B * kVec; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / kVec;
        if (mask && !mask[b]) continue;
        reinterpret_cast<int4*>(state + b * stride)[i % kVec] = make_int4(0, 0, 0, 0);
    }
}

int check_state(const void* state, int64_t state_stride) {
    if (!state || (reinterpret_cast<uintptr_t>(state) & 15) != 0) return AEC_EINVAL;
    if (state_stride < S2State::kBytes || (state_stride % 16) != 0) return AEC_EINVAL;
    return AEC_OK;
}

bool aligned4(const void* p) { return p && (reinterpret_cast<uintptr_t>(p) & 3) == 0; }

}  // namespace
}  // namespace aec

using namespace aec;

extern "C" int64_t aec_stage2_state_bytes(void) { return S2State::kBytes; }

extern "C" int aec_stage2_state_init(void* state, int64_t B, int64_t state_stride, const uint8_t* reset_mask,
                                     void* cuda_stream) {
    const int rc = check_state(state, state_stride);
    if (rc != AEC_OK) return rc;
    if (B < 0 || B > 0x7fffffffLL) return AEC_EINVAL;
    if (B == 0) return AEC_OK;
    Tables tab;
    const int rc2 = get_tables(&tab);                 // device check (sm_100 only)
    if (rc2 != AEC_OK) return rc2;
    const long long n = B * (S2State::kBytes / 16);
    const unsigned grid = (unsigned)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
    stage2_stream_state_init_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        static_cast<unsigned char*>(state), B, state_stride, reset_mask);
    AEC_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return AEC_OK;
}

extern "C" int aec_stage2_run_stream(const float* mic, const float* ref, const float* erb, const aec_stage2_weights* w,
                                     float* out, const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride,
                                     int64_t out_stride, void* state, int64_t state_stride, int32_t bands,
                                     void* cuda_stream) {
    if (bands != kH) return AEC_EUNSUPPORTED;         // Little_net is built for 32 ERB bands (configs.py:21-27)
    int rc = check_state(state, state_stride);
    if (rc != AEC_OK) return rc;
    if (!w || !aligned4(w->gru_w_ih) || !aligned4(w->gru_w_hh) || !aligned4(w->gru_b_ih) || !aligned4(w->gru_b_hh) ||
        !aligned4(w->lin1_w) || !aligned4(w->lin1_b) || !aligned4(w->lin2_w) || !aligned4(w->lin2_b))
        return AEC_EINVAL;
    if (B < 0 || L < 0 || in_stride < L || out_stride < L) return AEC_EINVAL;
    if (B == 0 || L == 0) return AEC_OK;
    if (!mic || !ref || !aligned4(erb) || !out) return AEC_EINVAL;
    Tables tab;
    rc = get_tables(&tab);
    if (rc != AEC_OK) return rc;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    AEC_CUDA_CHECK(cudaFuncSetAttribute(stage2_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)kSmemBytes));
    // persistent grid: a CTA stages the weights once and its warps walk streams b, b + gridDim.x * kSW, ...
    const long long ctas = (B + kSW - 1) / kSW;
    const unsigned grid = (unsigned)(ctas < (long long)kCtasPerSm * sms ? ctas : (long long)kCtasPerSm * sms);
    stage2_stream_kernel<<<grid, kSW * 32, kSmemBytes, static_cast<cudaStream_t>(cuda_stream)>>>(
        mic, ref, erb, *w, out, n_samples, B, L, in_stride, out_stride, static_cast<unsigned char*>(state), state_stride,
        tab);
    AEC_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return AEC_OK;
}
