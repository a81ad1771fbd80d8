// Stand-alone spectral operators behind the reference's operator seams (frame = 512):
//   aec_stft      <-> ConvSTFT.forward      Stage2_lhm/scripts/network/attention_ccrn.py:45-52
//   aec_istft     <-> ConviSTFT.forward     Stage2_lhm/scripts/network/attention_ccrn.py:82-101
//   aec_features  <-> Little_net.forward    Stage2_lhm/scripts/network/ERB.py:262-290
// All three reuse the half-warp FFT-256 of the fused stage-1 kernel; a CTA works on a tile of
// 16 frames so the reference's [B, 2K, T] (T innermost) layout is read / written in 64-byte
// runs through a shared-memory transpose.
#include <cstdint>

#include "aec_common.cuh"
#include "fft_warp.cuh"

namespace aec {

namespace {

constexpr int kTT = 16;        // frames per CTA tile
constexpr int kThreads = 128;  // 8 half-warps, 2 frames each
constexpr int kK = 257;
constexpr int kPitch = kTT + 1;

__device__ __forceinline__ void unpack_pair_s(float2 fa, float2 fb, float2 w, float2& xk, float2& xm) {
    const float2 a = make_float2(fa.x + fb.x, fa.y - fb.y);
    const float2 d = make_float2(fa.y + fb.y, fb.x - fa.x);
    const float2 t = cmul(w, d);
    xk = make_float2(a.x + t.x, a.y + t.y);
    xm = make_float2(a.x - t.x, t.y - a.y);
}
__device__ __forceinline__ void pack_pair_s(float2 ek, float2 em, float2 w, float2& gk, float2& gm) {
    const float2 a = make_float2(ek.x + em.x, ek.y - em.y);
    const float2 d = make_float2(ek.x - em.x, ek.y + em.y);
    const float2 t = cmulc(d, w);
    gk = make_float2(a.x - t.y, a.y + t.x);
    gm = make_float2(a.x + t.y, t.x - a.y);
}

// Windowed analysis of frame t of one row into the half-warp's tile: tile[k] = Zc[k].
// `shift` is subtracted from in-range samples only (the zero pad stays zero, as in the
// reference where the shift precedes ConvSTFT's F.pad).
__device__ __forceinline__ void analyse_frame(const float* __restrict__ x, long long L, long long t, float shift,
                                              float2* tile, const Tables& tab, int h) {
    float2 v[16];
    const long long base = (t - 1) * 256;
    // interior frames of 8-byte aligned rows: unpredicated 64-bit loads (the common case)
    const bool fast = t >= 1 && base + 512 <= L && ((reinterpret_cast<uintptr_t>(x) & 7) == 0);
    if (fast) {
        const float2* xp = reinterpret_cast<const float2*>(x + base) + h;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const float2 w = __ldg(&tab.win_a[h + 16 * j]);
            const float2 xv = __ldg(xp + 16 * j);
            v[j] = make_float2((xv.x - shift) * w.x, (xv.y - shift) * w.y);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const long long s = base + 2 * h + 32 * j;
            const float2 w = __ldg(&tab.win_a[h + 16 * j]);
            const float x0 = (s >= 0 && s < L) ? __ldg(x + s) - shift : 0.f;
            const float x1 = (s + 1 >= 0 && s + 1 < L) ? __ldg(x + s + 1) - shift : 0.f;
            v[j] = make_float2(x0 * w.x, x1 * w.y);
        }
    }
    __syncwarp();
    fft256_halfwarp<false>(v, tile, tab.tw256, h);
#pragma unroll
    for (int p = 0; p < 16; ++p) tile[h + 16 * fft16_index(p)] = v[p];
    __syncwarp();
}

// ---------------------------------------------------------------------------------------
// STFT: x [B][in_stride] -> spec [B][514][T]
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) stft512_kernel(const float* __restrict__ x, float* __restrict__ spec,
                                                           long long L, long long in_stride, long long T, Tables tab) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tiles = reinterpret_cast<float2*>(smem);                       // [8][kTilePitch]
    float* outt = reinterpret_cast<float*>(smem + 8 * kTilePitch * sizeof(float2));  // [514][kPitch]
    const int tid = threadIdx.x, lane = tid & 31, hw = tid >> 4, h = lane & 15;
    const long long b = blockIdx.y, t0 = (long long)blockIdx.x * kTT;
    const float* xb = x + b * in_stride;
    float2* tile = tiles + hw * kTilePitch;
    for (int i = 0; i < 2; ++i) {
        const int tt = hw + 8 * i;
        const long long t = t0 + tt;
        {   // frames beyond T are analysed as zeros (loads predicated off) and never stored
            analyse_frame(xb, t < T ? L : 0, t, 0.f, tile, tab, h);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int k = h + 16 * q;
                float2 xk, xm;
                unpack_pair_s(tile[k], tile[(256 - k) & 255], __ldg(&tab.tw512[k]), xk, xm);
                outt[k * kPitch + tt] = xk.x;
                outt[(kK + k) * kPitch + tt] = (k == 0) ? 0.f : xk.y;
                outt[(256 - k) * kPitch + tt] = xm.x;
                outt[(kK + 256 - k) * kPitch + tt] = (k == 0) ? 0.f : xm.y;
            }
            if (h == 0) {
                float2 xk, xm;
                unpack_pair_s(tile[128], tile[128], make_float2(0.f, -1.f), xk, xm);
                outt[128 * kPitch + tt] = xk.x;
                outt[(kK + 128) * kPitch + tt] = xk.y;
            }
        }
    }
    __syncthreads();
    float* sb = spec + b * (2 * kK) * T;
    for (int idx = tid; idx < 2 * kK * kTT; idx += kThreads) {
        const int c = idx / kTT, tt = idx % kTT;
        if (t0 + tt < T) sb[(long long)c * T + t0 + tt] = outt[c * kPitch + tt];
    }
}

// ---------------------------------------------------------------------------------------
// iSTFT: spec [B][514][T] -> y [B][out_stride], (T-1)*256 samples per row.
// CTA emits output hops [g0, g0+15): needs frames g0 .. g0+15 (16 frames).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) istft512_kernel(const float* __restrict__ spec, float* __restrict__ y,
                                                            long long T, long long out_stride, Tables tab) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tiles = reinterpret_cast<float2*>(smem);                        // [8][256]
    float* inn = reinterpret_cast<float*>(smem + 8 * kTilePitch * sizeof(float2));    // [514][kPitch], later frames [16][512]
    const int tid = threadIdx.x, lane = tid & 31, hw = tid >> 4, h = lane & 15;
    const long long b = blockIdx.y, g0 = (long long)blockIdx.x * (kTT - 1);   // first output hop == first frame
    const float* sb = spec + b * (2 * kK) * T;
    for (int idx = tid; idx < 2 * kK * kTT; idx += kThreads) {
        const int c = idx / kTT, tt = idx % kTT;
        inn[c * kPitch + tt] = (g0 + tt < T) ? __ldg(sb + (long long)c * T + g0 + tt) : 0.f;
    }
    __syncthreads();
    float2* tile = tiles + hw * kTilePitch;
    float2 u[2][16];
    for (int i = 0; i < 2; ++i) {
        const int tt = hw + 8 * i;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int k = h + 16 * q;
            float2 ek = make_float2(inn[k * kPitch + tt], inn[(kK + k) * kPitch + tt]);
            float2 em = make_float2(inn[(256 - k) * kPitch + tt], inn[(kK + 256 - k) * kPitch + tt]);
            if (k == 0) {   // imaginary parts of DC / Nyquist have zero rows in the synthesis kernel
                ek.y = 0.f;
                em.y = 0.f;
            }
            float2 gk, gm;
            pack_pair_s(ek, em, __ldg(&tab.tw512[k]), gk, gm);
            tile[k] = gk;
            tile[(256 - k) & 255] = gm;
        }
        if (h == 0) {
            const float2 e = make_float2(inn[128 * kPitch + tt], inn[(kK + 128) * kPitch + tt]);
            float2 gk, gm;
            pack_pair_s(e, e, make_float2(0.f, -1.f), gk, gm);
            tile[128] = gk;
        }
        __syncwarp();
        float2 v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = tile[h + 16 * j];
        __syncwarp();
        fft256_halfwarp<true>(v, tile, tab.tw256, h);
#pragma unroll
        for (int p = 0; p < 16; ++p) {
            const int r = fft16_index(p);
            const float2 w = __ldg(&tab.win_s[h + 16 * r]);
            u[i][r] = make_float2(v[p].x * w.x, v[p].y * w.y);
        }
        __syncwarp();
    }
    __syncthreads();   // spectra consumed: reuse `inn` for the windowed frames
    float2* fr = reinterpret_cast<float2*>(inn);   // [16][256] float2 (sample pairs)
    for (int i = 0; i < 2; ++i) {
        const int tt = hw + 8 * i;
#pragma unroll
        for (int r = 0; r < 16; ++r) fr[tt * 256 + h + 16 * r] = u[i][r];
    }
    __syncthreads();
    float* yb = y + b * out_stride;
    // output hop g (samples g*256 ..) = second half of frame g + first half of frame g+1
    for (int idx = tid; idx < (kTT - 1) * 128; idx += kThreads) {
        const int tt = idx / 128, m = idx % 128;
        const long long g = g0 + tt;
        if (g + 1 <= T - 1) {
            const float2 a = fr[tt * 256 + 128 + m];
            const float2 c = fr[(tt + 1) * 256 + m];
            yb[g * 256 + 2 * m] = a.x + c.x;
            yb[g * 256 + 2 * m + 1] = a.y + c.y;
        }
    }
}

// ---------------------------------------------------------------------------------------
// Stage-2 feature front end: feat [B][T][2*bands]   (Stage2_lhm/scripts/network/ERB.py:262-290)
//
// A CTA walks tiles of 16 frames of one utterance.  Per tile: (1) a warp transforms one frame at a
// time, lanes 0-15 the microphone and 16-31 the reference signal (same half-warp FFT as the stage-1
// kernel), and stores the magnitudes; (2) the ERB projection runs with lane = (signal, frame) and the
// band warp-uniform, looping only over the band's non-zero bin range [lo_b, hi_b) -- the bank is ~2
// non-zeros per bin, so this is ~16x less work than the dense [T,257] @ [257,32] product the
// reference does -- and (3) the [16][2*bands] tile is written out coalesced.  The bank and its
// non-zero ranges are staged in shared memory once per CTA.
// ---------------------------------------------------------------------------------------
constexpr int kFeatMP = 259;   // magnitude row pitch (odd: lanes = frames read one bin conflict-free)

// (round 2: the bank is no longer staged densely in shared memory -- 33 KB for 483 non-zeros --; the projection reads
//  its coefficients through L1 (one broadcast load per bin, ~15 KB of sectors) and the output tile lives in the FFT
//  tiles, which are dead by then: 51 KB per CTA instead of 88, four CTAs per SM instead of two.)
__device__ __forceinline__ float sqrt_fast(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));     // 1 ulp; the arguments are >= 1e-9
    return r;
}

__global__ void __launch_bounds__(kThreads, 4) features512_kernel(const float* __restrict__ mic,
                                                               const float* __restrict__ ref,
                                                               const float* __restrict__ erb, float* __restrict__ feat,
                                                               long long L, long long in_stride, long long T, int bands,
                                                               float shift_mic, float shift_ref,
                                                               const float* __restrict__ shift_mic_dev,
                                                               const float* __restrict__ shift_ref_dev, Tables tab) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tiles = reinterpret_cast<float2*>(smem);                                  // [8][kTilePitch]
    float* mag = reinterpret_cast<float*>(smem + 8 * kTilePitch * sizeof(float2));    // [2][kTT][kFeatMP]
    int* lo = reinterpret_cast<int*>(mag + 2 * kTT * kFeatMP);                        // [bands]
    int* hi = lo + bands;                                                             // [bands]
    float* outt = reinterpret_cast<float*>(tiles);                                    // [kTT][2*bands], aliases the (dead) tiles
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = lane >> 4, h = lane & 15;
    const long long b = blockIdx.y;
    const long long n_tiles = (T + kTT - 1) / kTT;

    // non-zero bin range of every band (the cosine bank is ~2 non-zeros per bin)
    for (int j = tid; j < bands; j += kThreads) {
        int l = kK, u = 0;
        for (int k = 0; k < kK; ++k)
            if (__ldg(erb + k * bands + j) != 0.f) {
                l = l < k ? l : k;
                u = k + 1;
            }
        lo[j] = l;
        hi[j] = u;
    }
    const float* xb = (half == 0 ? mic : ref) + b * in_stride;
    // the batch-global scalar of ERB.py:254-255, by value or -- no host round trip -- from aec_batch_shift's output
    const float shift = half == 0 ? (shift_mic_dev ? __ldg(shift_mic_dev) : shift_mic)
                                  : (shift_ref_dev ? __ldg(shift_ref_dev) : shift_ref);
    float2* tile = tiles + (2 * warp + half) * kTilePitch;
    float* fb = feat + b * T * (2 * bands);

    for (long long tile_i = blockIdx.x; tile_i < n_tiles; tile_i += gridDim.x) {
        const long long t0 = tile_i * kTT;
        __syncthreads();                       // previous tile's projection / copy-out finished (and lo / hi visible)
        // ---- (1) analysis + magnitudes: warp w takes frames w, w+4, w+8, w+12 ----
        for (int i = 0; i < kTT / 4; ++i) {
            const int tt = warp + 4 * i;
            const long long t = t0 + tt;
            analyse_frame(xb, t < T ? L : 0, t, shift, tile, tab, h);
            float* mrow = mag + (half * kTT + tt) * kFeatMP;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int k = h + 16 * q;
                float2 xk, xm;
                unpack_pair_s(tile[k], tile[(256 - k) & 255], __ldg(&tab.tw512[k]), xk, xm);
                if (k == 0) {
                    xk.y = 0.f;
                    xm.y = 0.f;
                }
                mrow[k] = sqrt_fast(fmaf(xk.x, xk.x, fmaf(xk.y, xk.y, 1e-9f)));        // ERB.py:277-278
                mrow[256 - k] = sqrt_fast(fmaf(xm.x, xm.x, fmaf(xm.y, xm.y, 1e-9f)));
            }
            if (h == 0) {
                float2 xk, xm;
                unpack_pair_s(tile[128], tile[128], make_float2(0.f, -1.f), xk, xm);
                mrow[128] = sqrt_fast(fmaf(xk.x, xk.x, fmaf(xk.y, xk.y, 1e-9f)));
            }
            __syncwarp();
        }
        __syncthreads();
        // ---- (2) ERB projection: lane = (signal, frame), band uniform per warp ----
        {
            const float* mrow = mag + lane * kFeatMP;      // lane = half*16 + frame  ==  (sig*kTT + tt)
            for (int band = warp; band < bands; band += 4) {
                const int k0 = lo[band], k1 = hi[band];
                const float* cb = erb + band;
                float acc = 0.f;
                int k = k0;
                for (; k + 4 <= k1; k += 4) {                                              // ERB.py:282-283
                    const float c0 = __ldg(cb + k * bands), c1 = __ldg(cb + (k + 1) * bands);
                    const float c2 = __ldg(cb + (k + 2) * bands), c3 = __ldg(cb + (k + 3) * bands);
                    acc = fmaf(mrow[k], c0, acc);
                    acc = fmaf(mrow[k + 1], c1, acc);
                    acc = fmaf(mrow[k + 2], c2, acc);
                    acc = fmaf(mrow[k + 3], c3, acc);
                }
                for (; k < k1; ++k) acc = fmaf(mrow[k], __ldg(cb + k * bands), acc);
                // mic projection in lanes 0-15, ref projection in lanes 16-31 of the same frame
                const float other = __shfl_xor_sync(0xffffffffu, acc, 16);
                if (half == 0) {
                    outt[h * 2 * bands + band] = acc;
                    outt[h * 2 * bands + bands + band] = fabsf(acc - other);              // ERB.py:287-290
                }
            }
        }
        __syncthreads();
        // ---- (3) coalesced copy-out ----
        const int row_len = 2 * bands;
        for (int idx = tid; idx < kTT * row_len; idx += kThreads) {
            const int tt = idx / row_len;
            if (t0 + tt < T) fb[(t0 + tt) * row_len + (idx - tt * row_len)] = outt[idx];
        }
    }
}

// ---------------------------------------------------------------------------------------
// Frame 1024 (hop 512, 513 bins): one warp per frame, 512-point complex FFT (fft512_warp_regs)
// ---------------------------------------------------------------------------------------
constexpr int kK1k = 513;
constexpr int kFP1k = 2 * kTilePitch;   // float2 per warp tile

__global__ void __launch_bounds__(kThreads) stft1024_kernel(const float* __restrict__ x, float* __restrict__ spec,
                                                            long long L, long long in_stride, long long T, Tables tab) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tiles = reinterpret_cast<float2*>(smem);                              // [4][kFP1k]
    float* outt = reinterpret_cast<float*>(smem + 4 * kFP1k * sizeof(float2));    // [1026][kPitch]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, h = lane & 15, hb = lane >> 4;
    const long long b = blockIdx.y, t0 = (long long)blockIdx.x * kTT;
    const float* xb = x + b * in_stride;
    float2* tile = tiles + warp * kFP1k;
    const TwiddleRegs512 twr = TwiddleRegs512::load(tab.tw512w, lane);
    for (int i = 0; i < 4; ++i) {
        const int tt = warp + 4 * i;
        const long long t = t0 + tt;
        const long long Lv = t < T ? L : 0;          // frames beyond T: zeros, never stored
        float2 v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const long long sidx = (t - 1) * 512 + 2 * lane + 64 * j;
            float2 w = __ldg(&tab.win_a1k[lane + 32 * (j & 7)]);
            if (j >= 8) w = make_float2(0.5f - w.x, 0.5f - w.y);
            const float x0 = (sidx >= 0 && sidx < Lv) ? __ldg(xb + sidx) : 0.f;
            const float x1 = (sidx + 1 >= 0 && sidx + 1 < Lv) ? __ldg(xb + sidx + 1) : 0.f;
            v[j] = make_float2(x0 * w.x, x1 * w.y);
        }
        __syncwarp();
        fft512_warp_regs<false>(v, tile, twr, lane);
#pragma unroll
        for (int p = 0; p < 16; ++p) tile[h + 16 * hb + 32 * fft16_index(p)] = v[p];
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int k = lane + 32 * q;
            float2 xk, xm;
            unpack_pair_s(tile[k], tile[(512 - k) & 511], __ldg(&tab.tw1024[k]), xk, xm);
            outt[k * kPitch + tt] = xk.x;
            outt[(kK1k + k) * kPitch + tt] = (k == 0) ? 0.f : xk.y;
            outt[(512 - k) * kPitch + tt] = xm.x;
            outt[(kK1k + 512 - k) * kPitch + tt] = (k == 0) ? 0.f : xm.y;
        }
        if (lane == 0) {
            float2 xk, xm;
            unpack_pair_s(tile[256], tile[256], make_float2(0.f, -1.f), xk, xm);
            outt[256 * kPitch + tt] = xk.x;
            outt[(kK1k + 256) * kPitch + tt] = xk.y;
        }
        __syncwarp();
    }
    __syncthreads();
    float* sb = spec + b * (2 * kK1k) * T;
    for (int idx = tid; idx < 2 * kK1k * kTT; idx += kThreads) {
        const int c = idx / kTT, tt = idx % kTT;
        if (t0 + tt < T) sb[(long long)c * T + t0 + tt] = outt[c * kPitch + tt];
    }
}

__global__ void __launch_bounds__(kThreads) istft1024_kernel(const float* __restrict__ spec, float* __restrict__ y,
                                                             long long T, long long out_stride, Tables tab) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tiles = reinterpret_cast<float2*>(smem);                                           // [4][kFP1k]
    float* inn = reinterpret_cast<float*>(smem + 4 * kFP1k * sizeof(float2));                  // [1026][kPitch]
    float2* fr = reinterpret_cast<float2*>(smem + 4 * kFP1k * sizeof(float2) + (size_t)2 * kK1k * kPitch * sizeof(float));  // [16][512]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, h = lane & 15, hb = lane >> 4;
    const long long b = blockIdx.y, g0 = (long long)blockIdx.x * (kTT - 1);
    const float* sb = spec + b * (2 * kK1k) * T;
    for (int idx = tid; idx < 2 * kK1k * kTT; idx += kThreads) {
        const int c = idx / kTT, tt = idx % kTT;
        inn[c * kPitch + tt] = (g0 + tt < T) ? __ldg(sb + (long long)c * T + g0 + tt) : 0.f;
    }
    __syncthreads();
    float2* tile = tiles + warp * kFP1k;
    const TwiddleRegs512 twr = TwiddleRegs512::load(tab.tw512w, lane);
    for (int i = 0; i < 4; ++i) {
        const int tt = warp + 4 * i;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int k = lane + 32 * q;
            float2 ek = make_float2(inn[k * kPitch + tt], inn[(kK1k + k) * kPitch + tt]);
            float2 em = make_float2(inn[(512 - k) * kPitch + tt], inn[(kK1k + 512 - k) * kPitch + tt]);
            if (k == 0) {
                ek.y = 0.f;
                em.y = 0.f;
            }
            float2 gk, gm;
            pack_pair_s(ek, em, __ldg(&tab.tw1024[k]), gk, gm);
            tile[k] = gk;
            tile[(512 - k) & 511] = gm;
        }
        if (lane == 0) {
            const float2 e = make_float2(inn[256 * kPitch + tt], inn[(kK1k + 256) * kPitch + tt]);
            float2 gk, gm;
            pack_pair_s(e, e, make_float2(0.f, -1.f), gk, gm);
            tile[256] = gk;
        }
        __syncwarp();
        float2 v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = tile[lane + 32 * j];
        __syncwarp();
        fft512_warp_regs<true>(v, tile, twr, lane);
#pragma unroll
        for (int p = 0; p < 16; ++p) {
            const int m = h + 16 * hb + 32 * fft16_index(p);
            const float2 w = __ldg(&tab.win_s1k[m]);
            fr[tt * 512 + m] = make_float2(v[p].x * w.x, v[p].y * w.y);
        }
        __syncwarp();
    }
    __syncthreads();
    float* yb = y + b * out_stride;
    for (int idx = tid; idx < (kTT - 1) * 256; idx += kThreads) {
        const int tt = idx / 256, m = idx % 256;
        const long long g = g0 + tt;
        if (g + 1 <= T - 1) {
            const float2 a = fr[tt * 512 + 256 + m];
            const float2 c = fr[(tt + 1) * 512 + m];
            yb[g * 512 + 2 * m] = a.x + c.x;
            yb[g * 512 + 2 * m + 1] = a.y + c.y;
        }
    }
}

template <typename K>
int set_smem(K kern, size_t bytes) {
    AEC_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return AEC_OK;
}

}  // namespace
}  // namespace aec

using namespace aec;

static constexpr int64_t kMaxGridY = 65535;

extern "C" int aec_stft(const float* x, float* spec, int64_t B, int64_t L, int64_t in_stride, int32_t frame,
                        void* cuda_stream) {
    if (B < 0 || L < 0 || in_stride < L) return AEC_EINVAL;
    if (frame != 512 && frame != 1024) return AEC_EINVAL;
    if (B == 0) return AEC_OK;
    if (!x || !spec) return AEC_EINVAL;
    if (B > kMaxGridY) {        // grid.y carries the utterance index: larger batches go in slices
        const long long per = 2LL * (frame / 2 + 1) * aec_num_frames(L, frame);
        for (int64_t off = 0; off < B; off += kMaxGridY) {
            const int rc2 = aec_stft(x + off * in_stride, spec + off * per, (B - off < kMaxGridY) ? B - off : kMaxGridY, L,
                                     in_stride, frame, cuda_stream);
            if (rc2 != AEC_OK) return rc2;
        }
        return AEC_OK;
    }
    Tables tab;
    int rc = get_tables(&tab);
    if (rc != AEC_OK) return rc;
    const long long T = aec_num_frames(L, frame);
    if (frame == 1024) {
        const size_t smem1k = 4 * kFP1k * sizeof(float2) + (size_t)2 * kK1k * kPitch * sizeof(float);
        rc = set_smem(stft1024_kernel, smem1k);
        if (rc != AEC_OK) return rc;
        dim3 grid1k((unsigned)((T + kTT - 1) / kTT), (unsigned)B);
        stft1024_kernel<<<grid1k, kThreads, smem1k, static_cast<cudaStream_t>(cuda_stream)>>>(x, spec, L, in_stride, T, tab);
        AEC_CUDA_CHECK(cudaGetLastError());
        count_launch();
        return AEC_OK;
    }
    const size_t smem = 8 * kTilePitch * sizeof(float2) + (size_t)2 * kK * kPitch * sizeof(float);
    rc = set_smem(stft512_kernel, smem);
    if (rc != AEC_OK) return rc;
    dim3 grid((unsigned)((T + kTT - 1) / kTT), (unsigned)B);
    stft512_kernel<<<grid, kThreads, smem, static_cast<cudaStream_t>(cuda_stream)>>>(x, spec, L, in_stride, T, tab);
    AEC_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return AEC_OK;
}

extern "C" int aec_istft(const float* spec, float* y, int64_t B, int64_t T, int64_t out_stride, int32_t frame,
                         void* cuda_stream) {
    if (B < 0 || T < 0) return AEC_EINVAL;
    if (frame != 512 && frame != 1024) return AEC_EINVAL;
    if (T >= 1 && out_stride < (T - 1) * (frame / 2)) return AEC_EINVAL;
    if (B == 0 || T <= 1) return AEC_OK;
    if (!spec || !y) return AEC_EINVAL;
    if (B > kMaxGridY) {
        const long long per = 2LL * (frame / 2 + 1) * T;
        for (int64_t off = 0; off < B; off += kMaxGridY) {
            const int rc2 = aec_istft(spec + off * per, y + off * out_stride, (B - off < kMaxGridY) ? B - off : kMaxGridY, T,
                                      out_stride, frame, cuda_stream);
            if (rc2 != AEC_OK) return rc2;
        }
        return AEC_OK;
    }
    Tables tab;
    int rc = get_tables(&tab);
    if (rc != AEC_OK) return rc;
    if (frame == 1024) {
        const size_t smem1k = 4 * kFP1k * sizeof(float2) + (size_t)2 * kK1k * kPitch * sizeof(float) +
                              (size_t)kTT * 512 * sizeof(float2);
        rc = set_smem(istft1024_kernel, smem1k);
        if (rc != AEC_OK) return rc;
        dim3 grid1k((unsigned)((T - 1 + kTT - 2) / (kTT - 1)), (unsigned)B);
        istft1024_kernel<<<grid1k, kThreads, smem1k, static_cast<cudaStream_t>(cuda_stream)>>>(spec, y, T, out_stride, tab);
        AEC_CUDA_CHECK(cudaGetLastError());
        count_launch();
        return AEC_OK;
    }
    const size_t smem = 8 * kTilePitch * sizeof(float2) + (size_t)2 * kK * kPitch * sizeof(float);
    rc = set_smem(istft512_kernel, smem);
    if (rc != AEC_OK) return rc;
    const long long hops = T - 1;
    dim3 grid((unsigned)((hops + kTT - 2) / (kTT - 1)), (unsigned)B);
    istft512_kernel<<<grid, kThreads, smem, static_cast<cudaStream_t>(cuda_stream)>>>(spec, y, T, out_stride, tab);
    AEC_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return AEC_OK;
}

namespace aec {
namespace {
// ---------------------------------------------------------------------------------------
// Batch-global shift mean(x) / std(x) (unbiased, torch.std) of ERB.py:254-256, on the device: per-CTA partial sums
// in double (fixed order -> deterministic), one finishing CTA; the scalar stays in device memory.
// ---------------------------------------------------------------------------------------
constexpr int kShiftCtas = 592, kShiftThreads = 256;

__global__ void __launch_bounds__(kShiftThreads) shift_partial_kernel(const float* __restrict__ x, long long B, long long L,
                                                                      long long stride, double* __restrict__ part) {
    double s = 0.0, q = 0.0;
    const bool vec = (L % 4 == 0) && (stride % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
    if (vec) {
        const long long per_row = L / 4, total = B * per_row;
        for (long long i = (long long)blockIdx.x * kShiftThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kShiftThreads) {
            const long long r = i / per_row, c = i - r * per_row;
            const float4 v = __ldg(reinterpret_cast<const float4*>(x + r * stride) + c);
            const float a = (v.x + v.y) + (v.z + v.w);
            const float b2 = fmaf(v.x, v.x, v.y * v.y) + fmaf(v.z, v.z, v.w * v.w);
            s += (double)a;
            q += (double)b2;
        }
    } else {
        const long long total = B * L;
        for (long long i = (long long)blockIdx.x * kShiftThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kShiftThreads) {
            const long long r = i / L, c = i - r * L;
            const float v = __ldg(x + r * stride + c);
            s += (double)v;
            q += (double)v * (double)v;
        }
    }
    __shared__ double sh[2][kShiftThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if ((threadIdx.x & 31) == 0) {
        sh[0][threadIdx.x >> 5] = s;
        sh[1][threadIdx.x >> 5] = q;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ts = 0.0, tq = 0.0;
        for (int w = 0; w < kShiftThreads / 32; ++w) {
            ts += sh[0][w];
            tq += sh[1][w];
        }
        part[2 * blockIdx.x] = ts;
        part[2 * blockIdx.x + 1] = tq;
    }
}

__global__ void __launch_bounds__(32) shift_finish_kernel(const double* __restrict__ part, int n_part, double count,
                                                          float* __restrict__ out) {
    if (threadIdx.x != 0) return;
    double s = 0.0, q = 0.0;
    for (int i = 0; i < n_part; ++i) {
        s += part[2 * i];
        q += part[2 * i + 1];
    }
    const double mean = s / count;
    const double var = count > 1.0 ? (q - s * mean) / (count - 1.0) : 0.0;       // unbiased, like torch.std
    out[0] = (float)(mean / sqrt(var > 0.0 ? var : 0.0));                          // (std = 0 -> inf / nan, as in torch)
}

}  // namespace
}  // namespace aec

using namespace aec;

extern "C" int64_t aec_batch_shift_workspace_bytes(void) { return (int64_t)kShiftCtas * 2 * sizeof(double); }

extern "C" int aec_batch_shift(const float* x, int64_t B, int64_t L, int64_t stride, float* shift_dev, void* workspace,
                               int64_t workspace_bytes, void* cuda_stream) {
    if (B <= 0 || L <= 0 || stride < L || !x || !shift_dev || !workspace) return AEC_EINVAL;
    if (workspace_bytes < aec_batch_shift_workspace_bytes() || (reinterpret_cast<uintptr_t>(workspace) & 7)) return AEC_EINVAL;
    Tables tab;
    const int rc = get_tables(&tab);                  // device check (sm_100 only)
    if (rc != AEC_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
    shift_partial_kernel<<<kShiftCtas, kShiftThreads, 0, s>>>(x, B, L, stride, static_cast<double*>(workspace));
    shift_finish_kernel<<<1, 32, 0, s>>>(static_cast<const double*>(workspace), kShiftCtas, (double)B * (double)L, shift_dev);
    AEC_CUDA_CHECK(cudaGetLastError());
    count_launch(2);
    return AEC_OK;
}

static int features_impl(const float* mic, const float* ref, const float* erb, float* feat, int64_t B, int64_t L,
                         int64_t in_stride, int32_t frame, int32_t bands, float shift_mic, float shift_ref,
                         const float* shift_mic_dev, const float* shift_ref_dev, void* cuda_stream) {
    if (B < 0 || L < 0 || in_stride < L || bands < 1 || bands > 64) return AEC_EINVAL;
    if (frame != 512) return frame == 1024 ? AEC_EUNSUPPORTED : AEC_EINVAL;
    if (B == 0) return AEC_OK;
    if (!mic || !ref || !erb || !feat) return AEC_EINVAL;
    if (B > kMaxGridY) {
        const long long per = 2LL * bands * aec_num_frames(L, frame);
        for (int64_t off = 0; off < B; off += kMaxGridY) {
            const int rc2 = features_impl(mic + off * in_stride, ref + off * in_stride, erb, feat + off * per,
                                          (B - off < kMaxGridY) ? B - off : kMaxGridY, L, in_stride, frame, bands,
                                          shift_mic, shift_ref, shift_mic_dev, shift_ref_dev, cuda_stream);
            if (rc2 != AEC_OK) return rc2;
        }
        return AEC_OK;
    }
    Tables tab;
    int rc = get_tables(&tab);
    if (rc != AEC_OK) return rc;
    const long long T = aec_num_frames(L, frame);
    // FFT tiles (reused for the [kTT][2*bands] output tile: 16 x 128 floats at most), magnitudes, band ranges
    const size_t smem = 8 * kTilePitch * sizeof(float2) + (size_t)2 * kTT * kFeatMP * sizeof(float) +
                        (size_t)2 * bands * sizeof(int);
    rc = set_smem(features512_kernel, smem);
    if (rc != AEC_OK) return rc;
    // a CTA walks several tiles so that the ERB bank is staged once per CTA, not once per tile
    const long long n_tiles = (T + kTT - 1) / kTT;
    long long per_utt = n_tiles;
    if (B >= 512) per_utt = 2; else if (B >= 64) per_utt = 8;
    if (per_utt > n_tiles) per_utt = n_tiles;
    if (per_utt < 1) per_utt = 1;
    dim3 grid((unsigned)per_utt, (unsigned)B);
    features512_kernel<<<grid, kThreads, smem, static_cast<cudaStream_t>(cuda_stream)>>>(
        mic, ref, erb, feat, L, in_stride, T, bands, shift_mic, shift_ref, shift_mic_dev, shift_ref_dev, tab);
    AEC_CUDA_CHECK(cudaGetLastError());
    count_launch();
    return AEC_OK;
}

extern "C" int aec_features(const float* mic, const float* ref, const float* erb, float* feat, int64_t B, int64_t L,
                            int64_t in_stride, int32_t frame, int32_t bands, float shift_mic, float shift_ref,
                            void* cuda_stream) {
    return features_impl(mic, ref, erb, feat, B, L, in_stride, frame, bands, shift_mic, shift_ref, nullptr, nullptr,
                         cuda_stream);
}

extern "C" int aec_features_dev(const float* mic, const float* ref, const float* erb, float* feat, int64_t B, int64_t L,
                                int64_t in_stride, int32_t frame, int32_t bands, const float* shift_mic_dev,
                                const float* shift_ref_dev, void* cuda_stream) {
    return features_impl(mic, ref, erb, feat, B, L, in_stride, frame, bands, 0.f, 0.f, shift_mic_dev, shift_ref_dev,
                         cuda_stream);
}
