// Stage-2 residual-echo suppressor inference (the consumer of the stage-1 output):
//   aec_stage2_mask   <-> Little_net.forward lines Stage2_lhm/scripts/network/ERB.py:293-304
//                         (GRU 64->32, Linear 64->32 + ReLU, Linear 32->32 + sigmoid, mask * mic_erb)
//   aec_stage2_synth  <-> ERB.py:306-316 (est_erb @ erb^T applied to the microphone spectrum, iSTFT, + 1e-9)
// The feature tensor fed to the GRU comes from aec_features (ERB.py:262-290).  Pinned by
// tests/golden/reference_stage2.npz (the reference module itself, seeded weights).
#include <cstdint>
#include <type_traits>

#include "aec_common.cuh"
#include "fft_warp.cuh"
#include "stage2_net.cuh"

namespace aec {
namespace {

using namespace s2;

// utterances (= warps) per CTA: 4 for large batches (the 45 KB of weights are staged once per CTA), 1 for batches that would
// otherwise leave SMs empty -- the recurrence streams ~400 shared-memory wavefronts per utterance per frame, and four
// utterances on one SM pay them one after the other while other SMs sit idle

// One warp per utterance, lane j = hidden unit / band j, the frames in chunks of kCh (stage2_net.cuh).
constexpr int kScratch = kCh * kIn + 2 * kCh * kH + kH;   // floats per warp: xs[8][64] + hb[8][32] + os[8][32] + hs[32]

template <int kMaskWarps>
__global__ void __launch_bounds__(kMaskWarps * 32) stage2_mask_kernel(const float* __restrict__ feat,
                                                                      aec_stage2_weights w, float* __restrict__ est,
                                                                      long long B, long long T) {
    extern __shared__ __align__(16) float sm[];
    float* scratch = sm + kWFloats;        // per warp: kScratch floats
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    stage_weights(sm, w, tid, blockDim.x);
    __syncthreads();
    const long long b = (long long)blockIdx.x * kMaskWarps + warp;
    if (b >= B) return;
    float* xs = scratch + warp * kScratch;          // [kCh][64] the chunk's feature vectors
    float* hb = xs + kCh * kIn;                      // [kCh][32] h_t of the chunk
    float* os = hb + kCh * kH;                       // [kCh][32] linear1 outputs
    float* hs = os + kCh * kH;                       // [32]      h_{t-1}, broadcast buffer of the recurrence
    const float* fb = feat + b * T * kIn;
    float* eb = est + b * T * kH;
    const NetLane net = NetLane::load(sm, w, lane);
    float h = 0.f;
    for (long long t0 = 0; t0 < T; t0 += kCh) {
        const int nf = (int)((T - t0) < kCh ? (T - t0) : kCh);
        __syncwarp();
        // ---- stage the chunk's feature vectors (coalesced; frames past the end read as zero) ----
#pragma unroll
        for (int r = 0; r < 2 * kCh; ++r) {
            const int f = r >> 1, col = lane + 32 * (r & 1);
            xs[f * kIn + col] = (f < nf) ? __ldg(fb + (t0 + f) * kIn + col) : 0.f;
        }
        __syncwarp();
        float gr[kCh], gz[kCh], gn[kCh], a1[kCh], a2[kCh];
        gru_inputs(net, sm, xs, lane, gr, gz, gn);
        gru_chunk(net, gr, gz, gn, hs, hb, h, nf, lane);
        __syncwarp();
        net_outputs(net, sm, xs, hb, os, lane, a1, a2);
#pragma unroll
        for (int f = 0; f < kCh; ++f)
            if (f < nf) eb[(t0 + f) * kH + lane] = sigmoidf_(a2[f]) * xs[f * kIn + lane];   // est_erb = mask * mic_erb
    }
}

// ---- synthesis: out = iSTFT((est_erb @ erb^T) * STFT(mic - shift)) + 1e-9 -------------------
constexpr int kTT = 16, kThreads = 128;
static_assert(((8 * kTilePitch + kTT * 256) * 8 + kTT * kH * 4 + 2 * kK * 4) % 8 == 0, "coefficient pairs must be 8-byte aligned");

// (round 2: the dense bank is no longer staged in shared memory -- 33 KB per CTA for ~2 non-zeros per bin, re-staged by
//  every CTA for a single 15-hop tile --; a CTA now walks several tiles, reads the two or three coefficients of a bin
//  through L1, and needs 54 KB instead of 87: four CTAs per SM instead of two.)
__global__ void __launch_bounds__(kThreads, 4) stage2_synth_kernel(const float* __restrict__ mic,
                                                                   const float* __restrict__ est,
                                                                   const float* __restrict__ erb, float* __restrict__ y,
                                                                   long long L, long long in_stride, long long out_stride,
                                                                   long long T, float shift_val,
                                                                   const float* __restrict__ shift_dev, Tables tab) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tiles = reinterpret_cast<float2*>(smem);                                   // [8][kTilePitch]
    float2* fr = tiles + 8 * kTilePitch;                                               // [kTT][256]
    float* es = reinterpret_cast<float*>(fr + kTT * 256);                              // [kTT][32]
    int* blo = reinterpret_cast<int*>(es + kTT * kH);                                  // [257]
    int* bhi = blo + kK;                                                               // [257]
    float2* c2 = reinterpret_cast<float2*>(bhi + kK);                                  // [257]  (offset 54280: 8-byte aligned)
    const int tid = threadIdx.x, lane = tid & 31, hw = tid >> 4, h = lane & 15;
    const long long b = blockIdx.y;
    const float shift = shift_dev ? __ldg(shift_dev) : shift_val;      // ERB.py:254, by value or from aec_batch_shift
    const BinBands bank{blo, bhi, c2, erb};
    bank.stage(tid, kThreads);
    const float* xb = mic + b * in_stride;
    float* yb = y + b * out_stride;
    float2* tile = tiles + hw * kTilePitch;
    const long long n_tiles = (T - 1 + kTT - 2) / (kTT - 1);
    for (long long tile_i = blockIdx.x; tile_i < n_tiles; tile_i += gridDim.x) {
        const long long g0 = tile_i * (kTT - 1);
        __syncthreads();                           // previous tile's overlap-add finished (and blo / bhi visible)
        for (int i = tid; i < kTT * kH; i += kThreads) {
            const long long t = g0 + i / kH;
            es[i] = t < T ? __ldg(est + (b * T + t) * kH + (i % kH)) : 0.f;
        }
        __syncthreads();
        for (int i = 0; i < 2; ++i) {
            const int tt = hw + 8 * i;
            const long long t = g0 + tt;
            // ---- analysis of the (shifted) microphone frame ----
            {
                float2 v[16];
                const long long base = (t - 1) * 256;
                const long long Lv = t < T ? L : 0;
                // interior frames of 8-byte aligned rows: unpredicated 64-bit loads (the common case; the scalar
                // predicated form made this kernel wait on global loads: long_scoreboard 7.8 per issue)
                if (t >= 1 && base + 512 <= Lv && ((reinterpret_cast<uintptr_t>(xb) & 7) == 0)) {
                    const float2* xp = reinterpret_cast<const float2*>(xb + base) + h;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float2 wv = __ldg(&tab.win_a[h + 16 * j]);
                        const float2 xv = __ldg(xp + 16 * j);
                        v[j] = make_float2((xv.x - shift) * wv.x, (xv.y - shift) * wv.y);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const long long s = base + 2 * h + 32 * j;
                        const float2 wv = __ldg(&tab.win_a[h + 16 * j]);
                        const float x0 = (s >= 0 && s < Lv) ? __ldg(xb + s) - shift : 0.f;
                        const float x1 = (s + 1 >= 0 && s + 1 < Lv) ? __ldg(xb + s + 1) - shift : 0.f;
                        v[j] = make_float2(x0 * wv.x, x1 * wv.y);
                    }
                }
                __syncwarp();
                fft256_halfwarp<false>(v, tile, tab.tw256, h);
#pragma unroll
                for (int p = 0; p < 16; ++p) tile[h + 16 * fft16_index(p)] = v[p];
                __syncwarp();
            }
            // ---- per-bin gain, inverse transform, synthesis window ----
            float2 v[16];
            synth_frame(tile, bank, es, tt, tab, h, v);
#pragma unroll
            for (int p = 0; p < 16; ++p) {
                const int r = fft16_index(p);
                const float2 wv = __ldg(&tab.win_s[h + 16 * r]);
                fr[tt * 256 + h + 16 * r] = make_float2(v[p].x * wv.x, v[p].y * wv.y);
            }
            __syncwarp();
        }
        __syncthreads();
        for (int idx = tid; idx < (kTT - 1) * 128; idx += kThreads) {
            const int tt = idx / 128, m = idx % 128;
            const long long g = g0 + tt;
            if (g + 1 <= T - 1) {
                const float2 a = fr[tt * 256 + 128 + m];
                const float2 c = fr[(tt + 1) * 256 + m];
                yb[g * 256 + 2 * m] = a.x + c.x + 1e-9f;                     // ERB.py:316
                yb[g * 256 + 2 * m + 1] = a.y + c.y + 1e-9f;
            }
        }
    }
}

}  // namespace
}  // namespace aec

using namespace aec;

extern "C" int aec_stage2_mask(const float* feat, const aec_stage2_weights* w, float* est_erb, int64_t B, int64_t T,
                               int32_t bands, void* cuda_stream) {
    if (B < 0 || T < 0 || !w) return AEC_EINVAL;
    if (bands != kH) return AEC_EUNSUPPORTED;        // Little_net is built for 32 ERB bands (configs.py:21-27)
    if (B == 0 || T == 0) return AEC_OK;
    if (!feat || !est_erb || !w->gru_w_ih || !w->gru_w_hh || !w->gru_b_ih || !w->gru_b_hh || !w->lin1_w ||
        !w->lin1_b || !w->lin2_w || !w->lin2_b)
        return AEC_EINVAL;
    Tables tab;
    int rc = get_tables(&tab);                        // device check (sm_100 only)
    if (rc != AEC_OK) return rc;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    auto launch = [&](auto warps_tag) -> int {
        constexpr int kW = decltype(warps_tag)::value;
        const size_t smem = (size_t)(kIn * 96 + kIn * kH + kH * kH + 256 + kW * kScratch) * sizeof(float);
        AEC_CUDA_CHECK(cudaFuncSetAttribute(stage2_mask_kernel<kW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const unsigned grid = (unsigned)((B + kW - 1) / kW);
        stage2_mask_kernel<kW><<<grid, kW * 32, smem, static_cast<cudaStream_t>(cuda_stream)>>>(feat, *w, est_erb, B, T);
        return AEC_OK;
    };
    rc = (B <= 4LL * sms) ? launch(std::integral_constant<int, 1>{}) : launch(std::integral_constant<int, 4>{});
    if (rc != AEC_OK) return rc;
    AEC_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return AEC_OK;
}

static int synth_impl(const float* mic, const float* est_erb, const float* erb, float* out, int64_t B, int64_t L,
                      int64_t in_stride, int64_t out_stride, int32_t frame, int32_t bands, float shift_mic,
                      const float* shift_mic_dev, void* cuda_stream) {
    if (B < 0 || L < 0 || in_stride < L) return AEC_EINVAL;
    if (frame != 512 || bands != kH) return AEC_EUNSUPPORTED;
    const long long T = aec_num_frames(L, frame);
    if (T >= 1 && out_stride < (T - 1) * 256) return AEC_EINVAL;
    if (B == 0 || T <= 1) return AEC_OK;
    if (!mic || !est_erb || !erb || !out) return AEC_EINVAL;
    if (B > 65535) {            // grid.y carries the utterance index: larger batches go in slices
        for (int64_t off = 0; off < B; off += 65535) {
            const int rc2 = synth_impl(mic + off * in_stride, est_erb + off * T * kH, erb, out + off * out_stride,
                                       (B - off < 65535) ? B - off : 65535, L, in_stride, out_stride, frame, bands,
                                       shift_mic, shift_mic_dev, cuda_stream);
            if (rc2 != AEC_OK) return rc2;
        }
        return AEC_OK;
    }
    Tables tab;
    int rc = get_tables(&tab);
    if (rc != AEC_OK) return rc;
    const size_t smem = (size_t)(8 * kTilePitch + kTT * 256) * sizeof(float2) + (size_t)(kTT * kH) * sizeof(float) +
                        (size_t)(2 * kK) * sizeof(int) + (size_t)kK * sizeof(float2);
    AEC_CUDA_CHECK(cudaFuncSetAttribute(stage2_synth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // a CTA walks several tiles of one utterance, so that the per-CTA set-up (band ranges) is not paid per tile
    const long long n_tiles = (T - 1 + kTT - 2) / (kTT - 1);
    long long per_utt = n_tiles;
    if (B >= 512) per_utt = 2; else if (B >= 64) per_utt = 8;
    if (per_utt > n_tiles) per_utt = n_tiles;
    if (per_utt < 1) per_utt = 1;
    dim3 grid((unsigned)per_utt, (unsigned)B);
    stage2_synth_kernel<<<grid, kThreads, smem, static_cast<cudaStream_t>(cuda_stream)>>>(
        mic, est_erb, erb, out, L, in_stride, out_stride, T, shift_mic, shift_mic_dev, tab);
    AEC_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return AEC_OK;
}

extern "C" int aec_stage2_synth(const float* mic, const float* est_erb, const float* erb, float* out, int64_t B,
                                int64_t L, int64_t in_stride, int64_t out_stride, int32_t frame, int32_t bands,
                                float shift_mic, void* cuda_stream) {
    return synth_impl(mic, est_erb, erb, out, B, L, in_stride, out_stride, frame, bands, shift_mic, nullptr, cuda_stream);
}

extern "C" int aec_stage2_synth_dev(const float* mic, const float* est_erb, const float* erb, float* out, int64_t B,
                                    int64_t L, int64_t in_stride, int64_t out_stride, int32_t frame, int32_t bands,
                                    const float* shift_mic_dev, void* cuda_stream) {
    return synth_impl(mic, est_erb, erb, out, B, L, in_stride, out_stride, frame, bands, 0.f, shift_mic_dev, cuda_stream);
}
