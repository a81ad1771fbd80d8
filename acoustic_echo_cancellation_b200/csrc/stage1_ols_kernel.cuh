// Stage-1 linear echo canceller, algo = 2 / 3: overlap-save partitioned-block FDAF with the alternated gradient
// constraint (time-domain blocks of H = 256 new samples, FFT length 512, P partitions), NLMS step (algo 2) or the
// diagonal Kalman step of algo 1 (algo 3).  One persistent CTA of two warps per utterance; filter taps, far-end
// history and the power / covariance state stay in registers for the whole utterance, like the STFT-domain kernels
// (stage1_kernel.cuh), whose bin ownership it shares, and with their half-warp FFT-256 (fft_warp.cuh) and real-FFT split
// (stage1_common.cuh).
//
// Unlike them the recurrence crosses the transform every block -- e(t) needs W(t), W(t) needs E(t-1) = FFT(e(t-1)) --
// so there is no chunk of frames to batch and the length of the per-block dependency chain is what counts.  Five
// transforms per block (X, y, E and the two of the constraint) are arranged so that only TWO are on the chain:
//   * the constraint is applied to partition c = t mod P AS IT ENTERED the block (oracle/aec_oracle.py:pbfdaf_ols):
//     it does not wait for E, so IFFT(W_c) runs on the upper half-warp beside IFFT(Yhat) on the lower one, and
//     FFT(g) beside FFT([0, e]) -- one warp, two transform slots, both half-warps busy;
//   * X_{t+1} = FFT[x_t, x_{t+1}] does not depend on the filter at all: the OTHER warp computes it during the same phase,
//     two blocks at a time (X_{t+1} on its lower half-warp, X_{t+2} on the upper one, every second block).
// Per block t, two block barriers:
//   R  (64 threads, 4 bins each + bin 128): [t >= 1: E_{t-1}, constrained W_c back into registers, power / covariance,
//      weight update]  then  X_t into the history, Yhat = sum_p W_p X_{t-p} packed for the inverse transform, W_c packed
//   F  warp a = (slot + t) & 1:  y = IFFT(Yhat)[H:], e = d - y -> HBM, E = FFT[0, e]  ||  g = IFFT(W_c), g[H:] = 0, FFT(g)
//      warp a ^ 1, odd t:        X_{t+1} || X_{t+2}            (the forward transform is one shared body for both roles)
// (a thread touches only its own bins' tile entries in R, so the update of block t-1 and the estimate of block t need
// no barrier between them).  Far-end / microphone blocks are staged HBM -> shared memory with cp.async (LDGSTS, 16 B
// per thread, no registers) three / one blocks ahead.
// Register layout of the taps: position j holds partition (j + t) mod P -- the weight update writes its result one
// position down (a different destination register costs nothing), so the partition to constrain is always position 0;
// the far-end history is a ring indexed by block mod P, which position j meets at slot (-j) mod P in every block.  Neither
// the history nor the taps are ever shifted or selected by a run-time index; only the insertion of X_t is (P selects).
// Why it exists: the STFT-domain recurrence (Hann analysis window, no cross-band terms) cancels ~13 dB on the SURVEY 8d
// single-talk set; the exact linear convolution of this one reaches the 40 dB noise floor, and with the Kalman step it
// holds 14 dB through double talk (DESIGN.md section 2).
// stage1_ols_stream_kernel is the same body (stage1_ols_body.cuh) with the filter state loaded from and stored to HBM, so
// that a stream processed chunk by chunk gives the outputs of one call over the whole signal (DESIGN.md section 5d).
// BUILDER-AUTHORED (the reference has no stage-1 filter): restated by oracle/aec_oracle.py:pbfdaf_ols, parity unpinned.
#pragma once
#include "stage1_common.cuh"

namespace aec {

struct OlsSmem {
    static constexpr size_t tile_bytes = size_t(4) * kTilePitch * sizeof(float2);   // X [2], Yhat / E, W_c
    static constexpr size_t blk_bytes = size_t(4 + 2) * 256 * sizeof(float);        // far-end ring [4][256], microphone [2][256]
    // far-end history of the regular bins in shared memory: [P slots][256 bins] float2, one column per thread and bin,
    // copied into registers for the update / estimate phase only.  With the Kalman step (and at 16 partitions) the state
    // does not fit the registers next to the transform's 16 complex values (2.85 against 3.4 ms per 1024 x 10 s at P = 4);
    // for the NLMS step it removes the last spills of the 128-register builds (2.30 against 2.38 ms at P = 4, 3.64 against
    // 3.73 at P = 8); at 1 / 2 partitions the registers hold it for free.
    __host__ __device__ static constexpr bool ring(int P, bool kalman) { return kalman || P >= 4; }
    __host__ __device__ static constexpr size_t base(int P) {                            // + bin 128, ERLE partials, role word
        return tile_bytes + blk_bytes + (size_t(P) * 20 + 16 + 15) / 16 * 16 + 128;
    }
    __host__ __device__ static constexpr size_t total(int P, bool kalman) {
        return base(P) + (ring(P, kalman) ? size_t(P) * 256 * sizeof(float2) : 0);
    }
};

// Weight update of one bin with the error spectrum E of the block (operation order of oracle/aec_oracle.py).
// ROT: W / C are in rotating positions (position j = partition (j + t) mod P), X is the ring (slot = block mod P):
// position j meets slot (-j) mod P and the result goes one position down.  !ROT: W, C by partition, X by delay (bin 128).
template <int P, bool KAL, bool ROT>
__device__ __forceinline__ void ols_update(float2 (&W)[P], const float2 (&X)[P], float (&C)[KAL ? P : 1], float& sp,
                                           const float2 E, const Stage1Params& prm) {
    auto xs = [&](int j) -> const float2& { return X[ROT ? (P - j) % P : j]; };
    auto dst = [](int j) constexpr { return ROT ? (j + P - 1) % P : j; };
    float2 Wn[P];
    if constexpr (!KAL) {
        float s = 0.f;
#pragma unroll
        for (int p = 0; p < P; ++p) s = fmaf(X[p].x, X[p].x, fmaf(X[p].y, X[p].y, s));
        sp = fmaf(prm.pblam, sp, prm.pboml * s);
        const float g = prm.mu * rcp_fast(sp + prm.delta);
        const float2 ge = make_float2(g * E.x, g * E.y);
#pragma unroll
        for (int j = 0; j < P; ++j) Wn[dst(j)] = cfmac(xs(j), ge, W[j]);
    } else {
        float Cn[P];
        const float e2 = fmaf(E.x, E.x, E.y * E.y);
        sp = fmaf(prm.klam, sp, prm.koml * e2);
        float d = 0.f;
#pragma unroll
        for (int j = 0; j < P; ++j) d = fmaf(C[j], fmaf(xs(j).x, xs(j).x, xs(j).y * xs(j).y), d);
        d = d + sp + prm.keps;
        const float rd = __frcp_rn(d);
#pragma unroll
        for (int j = 0; j < P; ++j) {
            const float2 x = xs(j);
            const float x2 = fmaf(x.x, x.x, x.y * x.y);
            const float gs = C[j] * rd;
            const float2 g = make_float2(gs * x.x, -gs * x.y);            // C conj(X) / D
            float2 w = cfma(g, E, W[j]);
            w = make_float2(prm.ka * w.x, prm.ka * w.y);
            Wn[dst(j)] = w;
            Cn[dst(j)] = fmaf(prm.ka2 * (1.f - gs * x2), C[j], prm.kq * fmaf(w.x, w.x, w.y * w.y));
        }
#pragma unroll
        for (int j = 0; j < P; ++j) C[j] = Cn[j];
    }
#pragma unroll
    for (int j = 0; j < P; ++j) W[j] = Wn[j];
}

// The self-mirrored bin (128 at frame 512, 256 at frame 1024) for LONG filters, one lane per tap: lanes 0 .. P-1 of one
// warp (P = 8 / 16), state in shared memory.  The serial form (one lane, all taps) is on the critical path of the update
// phase -- ~600 cycles of a 16-tap Kalman step -- and its unrolled code is a tenth of the hot loop; this one is ~100
// instructions and a few shuffle reductions.  zY / zW / zX: the bin's entries of the E / W_c / X tiles (split and packing
// twiddle -i: the real-signal bin is 2 conj(Z), and back).  Block t of the call is block t0 + t of the stream (t0: its
// blocks before the call, mod P); !EST: the update with E_{t-1} only (the streaming kernel's last one, which has no
// block t).
template <int P, bool KAL, bool EST = true>
__device__ __forceinline__ void ols_mid_parallel(int p, int t, float2* midW, float2* midX, float* midC, float* midS, float2* zY,
                                                 float2* zW, const float2* zX, const Stage1Params& prm, int t0 = 0) {
    constexpr unsigned mask = P >= 32 ? 0xffffffffu : ((1u << P) - 1u);
    auto conj2 = [](float2 z) { return make_float2(2.f * z.x, -2.f * z.y); };
    auto sum = [&](float v) {
#pragma unroll
        for (int o = P / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
        return v;
    };
    const int c = (t0 + t) & (P - 1);
    float2 w = midW[p];
    float cc = KAL ? midC[p] : 0.f;
    const float2 xo = midX[(t0 + t - 1 - p) & (P - 1)];                   // partner of partition p in block t - 1
    __syncwarp(mask);                                                 // every lane has its X before slot c is overwritten
    if (t >= 1) {
        const float2 ek = conj2(*zY), ca = conj2(*zW);
        if (p == ((t0 + t - 1) & (P - 1))) w = ca;                         // the constrained partition
        const float x2 = fmaf(xo.x, xo.x, xo.y * xo.y);
        if constexpr (!KAL) {
            const float pw = fmaf(prm.pblam, *midS, prm.pboml * sum(x2));
            const float g = prm.mu * rcp_fast(pw + prm.delta);
            w = cfmac(xo, make_float2(g * ek.x, g * ek.y), w);
            __syncwarp(mask);
            if (p == 0) *midS = pw;
        } else {
            const float psi = fmaf(prm.klam, *midS, prm.koml * fmaf(ek.x, ek.x, ek.y * ek.y));
            const float rd = __frcp_rn(sum(cc * x2) + psi + prm.keps);
            const float gs = cc * rd;
            w = cfma(make_float2(gs * xo.x, -gs * xo.y), ek, w);
            w = make_float2(prm.ka * w.x, prm.ka * w.y);
            cc = fmaf(prm.ka2 * (1.f - gs * x2), cc, prm.kq * fmaf(w.x, w.x, w.y * w.y));
            midC[p] = cc;
            __syncwarp(mask);
            if (p == 0) *midS = psi;
        }
        midW[p] = w;
    }
    if constexpr (!EST) return;
    const float2 xk = conj2(*zX);
    if (p == 0) midX[c] = xk;
    const float2 xe = p == 0 ? xk : midX[(t0 + t - p) & (P - 1)];          // partner of partition p in block t
    const float2 yp = cmul(w, xe);
    const float2 y = make_float2(sum(yp.x), sum(yp.y));
    if (p == 0) *zY = conj2(y);
    if (p == c) *zW = conj2(w);
}

// Shape of the CTA: every thread keeps 16 bin-taps of state (taps, far-end history, covariances) in registers, so the
// number of warps grows with the filter: 1-4 partitions: 2 warps, two mirrored pairs (4 bins) per thread; 8 partitions:
// 4 warps, one pair per thread; 16 partitions: 8 warps, ONE bin per thread (lanes 2i / 2i+1 share the mirrored pair i: both
// do the split of the pair and keep their own bin, and swap their results by shuffle for the packing).  The transform
// phase is the same for all of them (one warp carries the chain, one the far-end transforms); the roles rotate over all
// warps of the CTA.
__host__ __device__ constexpr int ols_warps(int P) { return P <= 4 ? 2 : P / 2; }

template <int P>
struct OlsShape {
    static constexpr int NW = ols_warps(P);
    static constexpr int NT = 32 * NW;
    static constexpr bool kSplit = (NW == 8);
    static constexpr int PPT = kSplit ? 1 : 128 / NT;      // pair slots per thread
    static constexpr int NB = kSplit ? 1 : 2 * PPT;        // bins per thread
};

template <int P, bool KAL, bool ECHO, int REGS>
__global__ void __launch_bounds__(OlsShape<P>::NT) __maxnreg__(REGS) stage1_ols_kernel(const Stage1Params prm) {
    constexpr bool STREAM = false;
#include "stage1_ols_body.cuh"
}

// One chunk of each of B streams: row b continues from the state at prm.state + b * prm.state_stride and leaves it there.
template <int P, bool KAL, bool ECHO, int REGS>
__global__ void __launch_bounds__(OlsShape<P>::NT) __maxnreg__(REGS) stage1_ols_stream_kernel(const Stage1Params prm) {
    constexpr bool STREAM = true;
#include "stage1_ols_body.cuh"
}

}  // namespace aec
