// Little_net, the Stage-2 residual-echo suppressor (Stage2_lhm/scripts/network/ERB.py:262-316), as both of its GPU forms
// compute it: the one-shot kernels (features512_kernel in aec_spectral.cu, stage2_mask_kernel and stage2_synth_kernel in
// aec_stage2.cu) and the streaming kernel (stage2_stream_kernel, aec_stage2_stream.cu).  The per-frame arithmetic they
// share is defined here once, so that a stream run in chunks computes every frame as the one-shot path does: the weight
// layout, the GRU and linear layers of a chunk, the bank's sparse ranges and the gain and inverse transform of a synthesis
// frame.
//
// Kept copies, because the shared form changes the SASS of the kernels in brackets (instruction order and registers; the
// outputs would not change).  A change to one of them has to be made at every call site.
//   accumulators      gr / gz / gn / a1 / a2 are declared by each caller of gru_inputs and net_outputs: declared inside a
//                     shared function they are allocated in the opposite order [stage2_mask_kernel<1>, <4>]
//   synthesis window  the multiply by tab.win_s after synth_frame [stage2_synth_kernel]
//   magnitudes        sqrt(re^2 + im^2 + 1e-9) of bins 0..256 of an analysed frame, in features512_kernel and
//                     stage2_stream_kernel [both]
// est_erb = sigmoidf_(a2) * mic_erb stays with the callers of net_outputs, which store it differently: to global memory
// for the real frames in stage2_mask_kernel, to the shared row es for every frame in stage2_stream_kernel.
#pragma once
#include <cuda_runtime.h>

#include "aec_common.cuh"
#include "fft_warp.cuh"

namespace aec {
namespace s2 {

constexpr int kH = 32;    // hidden units == ERB bands (Little_net: GRU(2*bands -> bands))
constexpr int kIn = 64;   // 2 * bands
constexpr int kCh = 8;    // frames per chunk of the recurrence
constexpr int kK = 257;   // bins of a frame-512 spectrum
// the staged weights, in floats (stage_weights)
constexpr int kWFloats = kIn * 96 + kIn * kH + kH * kH + 256;

// gate non-linearities on the frame-to-frame chain of the recurrence: MUFU.EX2 + MUFU.RCP forms (a few ulp; the pinned
// tolerance of the inference is 2e-4 relative) instead of the IEEE division and the branchy tanhf -- each of the three
// sits on the critical path of every time step
__device__ __forceinline__ float sigmoidf_(float v) { return __fdividef(1.f, 1.f + __expf(-v)); }
__device__ __forceinline__ float tanhf_(float v) { return 1.f - __fdividef(2.f, __expf(2.f * v) + 1.f); }

// The weights into kWFloats floats of shared memory, as float4 groups of four consecutive inputs per (gate, unit): one
// 16-byte load feeds four FFMAs.
//   wih : [gate 3][input/4 16][unit 32][4]     w1 : [input/4 16][unit 32][4]     w2 : [input/4 8][unit 32][4]
//   then b_ih[96] b_hh[96] b1[32] b2[32]
// By threads tid, tid + nt, ... of the CTA; the caller synchronises.
__device__ __forceinline__ void stage_weights(float* sm, const aec_stage2_weights& w, int tid, int nt) {
    float* wih = sm;
    float* w1 = wih + kIn * 96;
    float* w2 = w1 + kIn * kH;
    float* bias = w2 + kH * kH;
    for (int i = tid; i < 96 * kIn; i += nt) {
        const int row = i / kIn, col = i % kIn, g = row >> 5, j = row & 31;
        wih[(((g * (kIn / 4) + (col >> 2)) * 32 + j) << 2) + (col & 3)] = __ldg(w.gru_w_ih + i);
    }
    for (int i = tid; i < kH * kIn; i += nt) {
        const int j = i / kIn, col = i % kIn;
        w1[((((col >> 2)) * 32 + j) << 2) + (col & 3)] = __ldg(w.lin1_w + i);
    }
    for (int i = tid; i < kH * kH; i += nt) {
        const int j = i / kH, col = i % kH;
        w2[((((col >> 2)) * 32 + j) << 2) + (col & 3)] = __ldg(w.lin2_w + i);
    }
    for (int i = tid; i < 96; i += nt) {
        bias[i] = __ldg(w.gru_b_ih + i);
        bias[96 + i] = __ldg(w.gru_b_hh + i);
    }
    for (int i = tid; i < kH; i += nt) {
        bias[192 + i] = __ldg(w.lin1_b + i);
        bias[224 + i] = __ldg(w.lin2_b + i);
    }
}

// Lane j's share of the net (j = hidden unit / band): its biases, read from the staged weights, and its three rows of W_hh
// (gate order r, z, n), resident in registers for as long as the warp runs.
struct NetLane {
    float b_r, b_z, b_in, b_hn, b_1, b_2;
    float whr[kH], whz[kH], whn[kH];

    static __device__ __forceinline__ NetLane load(const float* sm, const aec_stage2_weights& w, int lane) {
        const float* wih = sm;
        const float* w1 = wih + kIn * 96;
        const float* w2 = w1 + kIn * kH;
        const float* bias = w2 + kH * kH;
        NetLane n;
        n.b_r = bias[lane] + bias[96 + lane];
        n.b_z = bias[32 + lane] + bias[128 + lane];
        n.b_in = bias[64 + lane];
        n.b_hn = bias[160 + lane];
        n.b_1 = bias[192 + lane];
        n.b_2 = bias[224 + lane];
#pragma unroll
        for (int i = 0; i < kH; ++i) {
            n.whr[i] = __ldg(w.gru_w_hh + (0 * kH + lane) * kH + i);
            n.whz[i] = __ldg(w.gru_w_hh + (1 * kH + lane) * kH + i);
            n.whn[i] = __ldg(w.gru_w_hh + (2 * kH + lane) * kH + i);
        }
        return n;
    }
};

// One warp per utterance or stream, lane j = hidden unit / band j, the frames in chunks of kCh (round 2: only what depends
// on h stays on the frame-to-frame chain):
//   phase 1  gru_inputs: W_ih x_t + b for the chunk's 8 frames at once -- no dependence on h, 24 independent accumulators
//            per lane, every weight load (float4 groups of four inputs per unit, staged transposed in shared memory) used 8
//            times;
//   phase 2  gru_chunk: the recurrence proper: W_hh h_{t-1} with lane j's three rows of W_hh held in REGISTERS (96
//            floats), the hidden state broadcast through 32 floats of shared memory (8 x LDS.128), gates, h_t -> per-chunk
//            buffer;
//   phase 3  net_outputs: Linear(64->32)+ReLU on cat[h_t, mic_erb_t] and Linear(32->32) for the 8 frames at once; the
//            caller stores est_erb = sigmoid(a2) * mic_erb.
// Before, every step ran all 18.4 k multiply-adds of the three layers (and ~400 shared-memory wavefronts of weights) as one
// dependent chain on a single warp: ~3 400 cycles per frame; the chain is now ~1/6 of that.
// xs [kCh][64] holds the chunk's feature vectors cat[mic_erb, |mic_erb - ref_erb|] (frames past the chunk's nf real ones
// zero), hb / os [kCh][32] and hs [32] are the warp's scratch.

// phase 1 into the caller's gr / gz / gn
__device__ __forceinline__ void gru_inputs(const NetLane& n, const float* sm, const float* xs, int lane, float (&gr)[kCh],
                                           float (&gz)[kCh], float (&gn)[kCh]) {
    const float4* wih4 = reinterpret_cast<const float4*>(sm) + lane;
#pragma unroll
    for (int f = 0; f < kCh; ++f) {
        gr[f] = n.b_r;
        gz[f] = n.b_z;
        gn[f] = n.b_in;
    }
#pragma unroll 2
    for (int i4 = 0; i4 < kIn / 4; ++i4) {
        const float4 wr = wih4[(0 * (kIn / 4) + i4) * 32], wz = wih4[(1 * (kIn / 4) + i4) * 32],
                     wn = wih4[(2 * (kIn / 4) + i4) * 32];
#pragma unroll
        for (int f = 0; f < kCh; ++f) {
            const float4 xv = *reinterpret_cast<const float4*>(xs + f * kIn + 4 * i4);
            gr[f] = fmaf(wr.w, xv.w, fmaf(wr.z, xv.z, fmaf(wr.y, xv.y, fmaf(wr.x, xv.x, gr[f]))));
            gz[f] = fmaf(wz.w, xv.w, fmaf(wz.z, xv.z, fmaf(wz.y, xv.y, fmaf(wz.x, xv.x, gz[f]))));
            gn[f] = fmaf(wn.w, xv.w, fmaf(wn.z, xv.z, fmaf(wn.y, xv.y, fmaf(wn.x, xv.x, gn[f]))));
        }
    }
}

// phase 2 for the first nf frames of the chunk: h_t into hb (zero for frames past nf); h is lane j's GRU state, carried
// from chunk to chunk
__device__ __forceinline__ void gru_chunk(const NetLane& n, const float (&gr)[kCh], const float (&gz)[kCh],
                                          const float (&gn)[kCh], float* hs, float* hb, float& h, int nf, int lane) {
    const float4* hs4 = reinterpret_cast<const float4*>(hs);
#pragma unroll
    for (int f = 0; f < kCh; ++f) {
        if (f < nf) {
            hs[lane] = h;
            __syncwarp();
            // four partial sums per gate: twelve independent chains of eight FFMAs
            float ar[4] = {0.f, 0.f, 0.f, 0.f}, az[4] = {0.f, 0.f, 0.f, 0.f}, an[4] = {n.b_hn, 0.f, 0.f, 0.f};
#pragma unroll
            for (int i4 = 0; i4 < kH / 4; ++i4) {
                const float4 hv = hs4[i4];
                ar[0] = fmaf(n.whr[4 * i4 + 0], hv.x, ar[0]); ar[1] = fmaf(n.whr[4 * i4 + 1], hv.y, ar[1]);
                ar[2] = fmaf(n.whr[4 * i4 + 2], hv.z, ar[2]); ar[3] = fmaf(n.whr[4 * i4 + 3], hv.w, ar[3]);
                az[0] = fmaf(n.whz[4 * i4 + 0], hv.x, az[0]); az[1] = fmaf(n.whz[4 * i4 + 1], hv.y, az[1]);
                az[2] = fmaf(n.whz[4 * i4 + 2], hv.z, az[2]); az[3] = fmaf(n.whz[4 * i4 + 3], hv.w, az[3]);
                an[0] = fmaf(n.whn[4 * i4 + 0], hv.x, an[0]); an[1] = fmaf(n.whn[4 * i4 + 1], hv.y, an[1]);
                an[2] = fmaf(n.whn[4 * i4 + 2], hv.z, an[2]); an[3] = fmaf(n.whn[4 * i4 + 3], hv.w, an[3]);
            }
            const float r = sigmoidf_(gr[f] + ((ar[0] + ar[1]) + (ar[2] + ar[3])));
            const float z = sigmoidf_(gz[f] + ((az[0] + az[1]) + (az[2] + az[3])));
            const float nn = tanhf_(fmaf(r, (an[0] + an[1]) + (an[2] + an[3]), gn[f]));
            h = fmaf(z, h - nn, nn);                 // (1 - z) n + z h
            hb[f * kH + lane] = h;
            __syncwarp();                            // every lane has read hs before the next step overwrites it
        } else {
            hb[f * kH + lane] = 0.f;
        }
    }
}

// phase 3 (ERB.py:295-304), with the caller's a1 / a2: on return os holds the ReLU outputs and a2 the mask logits
__device__ __forceinline__ void net_outputs(const NetLane& n, const float* sm, const float* xs, const float* hb, float* os,
                                            int lane, float (&a1)[kCh], float (&a2)[kCh]) {
    const float4* w14 = reinterpret_cast<const float4*>(sm + kIn * 96) + lane;
    const float4* w24 = reinterpret_cast<const float4*>(sm + kIn * 96 + kIn * kH) + lane;
#pragma unroll
    for (int f = 0; f < kCh; ++f) a1[f] = n.b_1;
#pragma unroll 2
    for (int i4 = 0; i4 < kH / 4; ++i4) {
        const float4 wa = w14[i4 * 32], wb = w14[(kH / 4 + i4) * 32];      // inputs 0..31 = h, 32..63 = mic_erb
#pragma unroll
        for (int f = 0; f < kCh; ++f) {
            const float4 hv = *reinterpret_cast<const float4*>(hb + f * kH + 4 * i4);
            const float4 xv = *reinterpret_cast<const float4*>(xs + f * kIn + 4 * i4);
            a1[f] = fmaf(wa.w, hv.w, fmaf(wa.z, hv.z, fmaf(wa.y, hv.y, fmaf(wa.x, hv.x, a1[f]))));
            a1[f] = fmaf(wb.w, xv.w, fmaf(wb.z, xv.z, fmaf(wb.y, xv.y, fmaf(wb.x, xv.x, a1[f]))));
        }
    }
#pragma unroll
    for (int f = 0; f < kCh; ++f) os[f * kH + lane] = fmaxf(a1[f], 0.f);
    __syncwarp();
#pragma unroll
    for (int f = 0; f < kCh; ++f) a2[f] = n.b_2;
#pragma unroll 2
    for (int i4 = 0; i4 < kH / 4; ++i4) {
        const float4 wv = w24[i4 * 32];
#pragma unroll
        for (int f = 0; f < kCh; ++f) {
            const float4 ov = *reinterpret_cast<const float4*>(os + f * kH + 4 * i4);
            a2[f] = fmaf(wv.w, ov.w, fmaf(wv.z, ov.z, fmaf(wv.y, ov.y, fmaf(wv.x, ov.x, a2[f]))));
        }
    }
}

// The bank erb [257][kH] in the sparse form the synthesis reads: the non-zero band range [blo[k], bhi[k]) of every bin
// (the reference's bank has <= 2 bands per bin) and the range's first two coefficients c2[k], all in shared memory; the
// coefficients of wider ranges come through L1.
struct BinBands {
    int* blo;
    int* bhi;
    float2* c2;
    const float* erb;

    // by threads tid, tid + nt, ... of the CTA; the caller synchronises
    __device__ __forceinline__ void stage(int tid, int nt) const {
        for (int k = tid; k < kK; k += nt) {
            int lo = kH, hi = 0;
            for (int j = 0; j < kH; ++j)
                if (__ldg(erb + k * kH + j) != 0.f) {
                    lo = min(lo, j);
                    hi = j + 1;
                }
            blo[k] = lo < kH ? lo : 0;
            bhi[k] = hi > lo ? hi : blo[k];
            c2[k] = make_float2(lo < hi ? __ldg(erb + k * kH + lo) : 0.f, lo + 1 < hi ? __ldg(erb + k * kH + lo + 1) : 0.f);
        }
    }
    // ERB.py:306-307 at bin k: (mask * mic_erb) @ erb^T of frame f, whose est_erb is es[f * kH ..]
    __device__ __forceinline__ float gain(const float* es, int f, int k) const {
        const int lo = blo[k], hi = bhi[k];
        const float2 c = c2[k];
        const float* e = es + f * kH + lo;
        float g = fmaf(e[0], c.x, 0.f);
        g = fmaf(e[lo + 1 < kH ? 1 : 0], c.y, g);   // (c.y is zero when the range has one band)
        for (int j = lo + 2; j < hi; ++j) g = fmaf(es[f * kH + j], __ldg(erb + k * kH + j), g);   // wider banks only
        return g;
    }
};

// Non-zero bin range [lo[j], hi[j]) of every band j of a bank erb [257][bands] (the cosine bank is ~2 non-zeros per bin),
// by threads tid, tid + nt, ... of the CTA; the caller synchronises.
__device__ __forceinline__ void band_bin_ranges(const float* erb, int bands, int* lo, int* hi, int tid, int nt) {
    for (int j = tid; j < bands; j += nt) {
        int l = kK, u = 0;
        for (int k = 0; k < kK; ++k)
            if (__ldg(erb + k * bands + j) != 0.f) {
                l = l < k ? l : k;
                u = k + 1;
            }
        lo[j] = l;
        hi[j] = u;
    }
}

// One synthesis frame (ERB.py:306-313), in the half-warp's tile holding the analysed microphone frame (tile[k] = Zc[k]):
// the per-bin gain of est_erb row f of es, the packing for the inverse transform (in place) and the inverse FFT-256.
// On return v[p] holds sample pair h + 16 fft16_index(p) of the frame before the synthesis window (tab.win_s, applied by
// the caller, which stores the frame where it needs it), and the tile is free once the half-warp has synchronised.  Lane
// h of the half-warp.
__device__ __forceinline__ void synth_frame(float2* tile, const BinBands& bb, const float* es, int f, const Tables& tab,
                                            int h, float2 (&v)[16]) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int k = h + 16 * q, km = (256 - k) & 255;
        const float2 wk = __ldg(&tab.tw512[k]);
        float2 xk, xm, gk, gm;
        unpack_pair(tile[k], tile[km], wk, xk, xm);
        const float ga = bb.gain(es, f, k), gb = bb.gain(es, f, 256 - k);
        xk = make_float2(ga * xk.x, k == 0 ? 0.f : ga * xk.y);       // ERB.py:309-310
        xm = make_float2(gb * xm.x, k == 0 ? 0.f : gb * xm.y);
        pack_pair(xk, xm, wk, gk, gm);
        tile[k] = gk;
        tile[km] = gm;
    }
    if (h == 0) {
        float2 xk, xm, gk, gm;
        unpack_pair(tile[128], tile[128], make_float2(0.f, -1.f), xk, xm);
        const float ga = bb.gain(es, f, 128);
        xk = make_float2(ga * xk.x, ga * xk.y);
        pack_pair(xk, xk, make_float2(0.f, -1.f), gk, gm);
        tile[128] = gk;
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = tile[h + 16 * j];
    __syncwarp();
    fft256_halfwarp<true>(v, tile, tab.tw256, h);
}

}  // namespace s2
}  // namespace aec
