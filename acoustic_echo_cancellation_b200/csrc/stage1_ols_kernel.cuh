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
// twiddle -i: the real-signal bin is 2 conj(Z), and back).
template <int P, bool KAL>
__device__ __forceinline__ void ols_mid_parallel(int p, int t, float2* midW, float2* midX, float* midC, float* midS, float2* zY,
                                                 float2* zW, const float2* zX, const Stage1Params& prm) {
    constexpr unsigned mask = P >= 32 ? 0xffffffffu : ((1u << P) - 1u);
    auto conj2 = [](float2 z) { return make_float2(2.f * z.x, -2.f * z.y); };
    auto sum = [&](float v) {
#pragma unroll
        for (int o = P / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
        return v;
    };
    const int c = t & (P - 1);
    float2 w = midW[p];
    float cc = KAL ? midC[p] : 0.f;
    const float2 xo = midX[(t - 1 - p) & (P - 1)];                   // partner of partition p in block t - 1
    __syncwarp(mask);                                                 // every lane has its X before slot c is overwritten
    if (t >= 1) {
        const float2 ek = conj2(*zY), ca = conj2(*zW);
        if (p == ((t - 1) & (P - 1))) w = ca;                         // the constrained partition
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
    const float2 xk = conj2(*zX);
    if (p == 0) midX[c] = xk;
    const float2 xe = p == 0 ? xk : midX[(t - p) & (P - 1)];          // partner of partition p in block t
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
    static_assert(P == 1 || P == 2 || P == 4 || P == 8 || P == 16, "partitions: a power of two, in registers");
    using SH = OlsShape<P>;
    constexpr int NW = SH::NW, NT = SH::NT, PPT = SH::PPT, NB = SH::NB;
    constexpr bool kSplit = SH::kSplit;
    constexpr int PC = KAL ? P : 1;
    constexpr bool kXs = OlsSmem::ring(P, KAL);                      // far-end history in shared memory instead of registers
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* tileX = reinterpret_cast<float2*>(smem_raw);             // [2] spectra of the far-end blocks, slot = block & 1
    float2* tileY = tileX + 2 * kTilePitch;
    float2* tileW = tileY + kTilePitch;
    float* xring = reinterpret_cast<float*>(tileW + kTilePitch);     // [4][256] far-end blocks, slot = block & 3
    float* dring = xring + 4 * 256;                                  // [2][256] microphone blocks, slot = block & 1
    float2* midW = reinterpret_cast<float2*>(dring + 2 * 256);       // [P] taps of bin 128 (its own mirror), by partition
    float2* midX = midW + P;                                         // [P] its far-end history, slot = block mod P
    float* midC = reinterpret_cast<float*>(midX + P);                // [P] covariances (Kalman)
    float* midS = midC + P;                                          // [1] smoothed power / Psi
    float* red = midS + 1;                                           // [2 NW] ERLE energies of the warps
    int* fft_warp_s = reinterpret_cast<int*>(red + 2 * NW);
    float2* xhist = reinterpret_cast<float2*>(smem_raw + OlsSmem::base(P));   // [P][NB][NT] (kXs), slot = block mod P

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = lane >> 4, h = lane & 15;
    const int side = tid & 1;                                        // kSplit: 0 = bin k, 1 = bin 256 - k of pair k = tid >> 1

    const int nblk = static_cast<int>(utterance_samples(prm, blockIdx.x) / 256);
    const float* far_b = prm.far + static_cast<long long>(blockIdx.x) * prm.in_stride;
    const float* mic_b = prm.mic + static_cast<long long>(blockIdx.x) * prm.in_stride;
    float* err_b = prm.err + static_cast<long long>(blockIdx.x) * prm.out_stride;
    float* echo_b = ECHO ? prm.echo + static_cast<long long>(blockIdx.x) * prm.out_stride : nullptr;

    // Warp w of a CTA sits on scheduler (slot + w) % 4, and the warp that carries the two-transform chain is the busier
    // one.  The roles rotate over the warps every block; for the two-warp CTAs (which only ever touch one scheduler pair)
    // the warp that starts with the chain follows the hardware warp slot, so that co-resident utterances on the same
    // scheduler pair load different schedulers (same device as the bin-128 owner of the STFT-domain kernel).
    if (tid == 0) {
        unsigned hw_warp;
        asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw_warp));
        *fft_warp_s = NW == 2 ? static_cast<int>((hw_warp >> 2) & 1u) : 0;
    }
    if (tid < P) {
        midW[tid] = make_float2(0.f, 0.f);
        midX[tid] = make_float2(0.f, 0.f);
        midC[tid] = prm.kc0;
    }
    if (tid == 0) *midS = 0.f;
    for (int i = tid; i < 256; i += NT) xring[3 * 256 + i] = 0.f;    // x_{-1} = 0 (slot of block -1)
    if constexpr (kXs)
        for (int i = tid; i < P * 256; i += NT) xhist[i] = make_float2(0.f, 0.f);
#ifdef AEC_PHASE_TIMING
    __shared__ long long dbg_sm[NW][12];
    if (lane == 0) {
        for (int i = 0; i < 11; ++i) dbg_sm[warp][i] = 0;
        dbg_sm[warp][11] = clock64();
    }
#endif
    // tuning (aec_cfg.stagger_ns > 0): start-up skew between the utterances that share an SM, so that the issue-bound
    // update phase of one meets the latency-bound transform phase of another instead of all of them running in step
    startup_skew(prm);
    __syncthreads();
    const int fw = *fft_warp_s;

    const TwiddleRegs twr = TwiddleRegs::load(prm.tw256, h);

    // ---- persistent per-bin state ----
    float2 W[NB][P], Xp[kXs ? 1 : NB][kXs ? 1 : P];
    float C[NB][PC], sp[NB];
    float2 wk[PPT];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        sp[b] = 0.f;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            W[b][p] = make_float2(0.f, 0.f);
            if constexpr (!kXs) Xp[b][p] = make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int p = 0; p < PC; ++p) C[b][p] = prm.kc0;
    }
#pragma unroll
    for (int i = 0; i < PPT; ++i) wk[i] = __ldg(&prm.tw512[kSplit ? (tid >> 1) : tid + NT * i]);

    // block staging: 64 threads x 4 samples per signal
    auto stage_block = [&](const float* row, float* dst, int blk) {
        if (blk < nblk && tid < 64) {
            const float* p = row + static_cast<long long>(blk) * 256 + 4 * tid;
            if (prm.use_tma) {
                cp_async16(dst + 4 * tid, p);
            } else {
                *reinterpret_cast<float4*>(dst + 4 * tid) = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
            }
        }
    };
    stage_block(far_b, xring, 0);
    stage_block(far_b, xring + 256, 1);
    cp_async_commit();

    float acc_m = 0.f, acc_e = 0.f;                                   // ERLE energies (lower half-warps)
    const float k512 = 1.0f / 512.0f;

    for (int t = -1; t < nblk; ++t) {
        stage_block(far_b, xring + ((t + 3) & 3) * 256, t + 3);
        stage_block(mic_b, dring + ((t + 1) & 1) * 256, t + 1);
        cp_async_commit();
        const int a = (fw + t) & (NW - 1);                            // the warp that carries the chain of this block
        // ---- R: update with E_{t-1}, echo estimate of block t ----
        if (t >= 0) {
            const int c = t & (P - 1);                                // partition constrained in this block = ring slot of X_t
            const float2* tX = tileX + (t & 1) * kTilePitch;
            // far-end history of this thread's bins: the persistent registers, or (kXs) a copy of the thread's columns of
            // the shared-memory ring that lives for this phase only
            float2 Xl[kXs ? NB : 1][kXs ? P : 1];
            float2 (&X)[NB][P] = *reinterpret_cast<float2 (*)[NB][P]>(kXs ? &Xl[0][0] : &Xp[0][0]);
            if constexpr (kXs) {
#pragma unroll
                for (int b = 0; b < NB; ++b)
#pragma unroll
                    for (int s2 = 0; s2 < P; ++s2) X[b][s2] = xhist[(s2 * NB + b) * NT + tid];
            }
#pragma unroll
            for (int i = 0; i < PPT; ++i) {
                const int k = kSplit ? (tid >> 1) : tid + NT * i, km = (256 - k) & 255;
                const int b0 = kSplit ? 0 : 2 * i, b1 = kSplit ? 0 : 2 * i + 1;     // this thread's bins k / 256 - k
                if (t >= 1) {
                    float2 ek, em, ca, cb;
                    unpack_pair(tileY[k], tileY[km], wk[i], ek, em);
                    unpack_pair(tileW[k], tileW[km], wk[i], ca, cb);                    // the constrained partition
                    if constexpr (kSplit) {
                        W[0][0] = side ? cb : ca;
                        ols_update<P, KAL, true>(W[0], X[0], C[0], sp[0], side ? em : ek, prm);
                    } else {
                        W[b0][0] = ca;
                        W[b1][0] = cb;
                        ols_update<P, KAL, true>(W[b0], X[b0], C[b0], sp[b0], ek, prm);
                        ols_update<P, KAL, true>(W[b1], X[b1], C[b1], sp[b1], em, prm);
                    }
                }
                float2 xk, xm, gk, gm;
                unpack_pair(tX[k], tX[km], wk[i], xk, xm);
                if constexpr (kSplit) xk = side ? xm : xk;
#pragma unroll
                for (int s = 0; s < P; ++s)
                    if (c == s) {
                        X[b0][s] = xk;
                        if constexpr (!kSplit) X[b1][s] = xm;
                    }
                if constexpr (kXs) {
                    xhist[(c * NB + b0) * NT + tid] = xk;
                    if constexpr (!kSplit) xhist[(c * NB + b1) * NT + tid] = xm;
                }
                float2 yk = make_float2(0.f, 0.f), ym = make_float2(0.f, 0.f), wa = W[b0][0], wb = W[b1][0];
#pragma unroll
                for (int j = 0; j < P; ++j) {
                    yk = cfma(W[b0][j], X[b0][(P - j) % P], yk);
                    if constexpr (!kSplit) ym = cfma(W[b1][j], X[b1][(P - j) % P], ym);
                }
                if constexpr (kSplit) {          // the partner lane holds the other bin of the pair
                    const float2 yo = make_float2(__shfl_xor_sync(0xffffffffu, yk.x, 1), __shfl_xor_sync(0xffffffffu, yk.y, 1));
                    const float2 wo = make_float2(__shfl_xor_sync(0xffffffffu, wa.x, 1), __shfl_xor_sync(0xffffffffu, wa.y, 1));
                    ym = side ? yk : yo;
                    yk = side ? yo : yk;
                    wb = side ? wa : wo;
                    wa = side ? wo : wa;
                }
                pack_pair(yk, ym, wk[i], gk, gm);
                if constexpr (kSplit) {
                    tileY[side ? km : k] = side ? gm : gk;
                } else {
                    tileY[k] = gk;
                    tileY[km] = gm;
                }
                pack_pair(wa, wb, wk[i], gk, gm);
                if constexpr (kSplit) {
                    tileW[side ? km : k] = side ? gm : gk;
                } else {
                    tileW[k] = gk;
                    tileW[km] = gm;
                }
            }
            if constexpr (P >= 16 || (KAL && P >= 8)) {               // bin 128, one lane per tap (long filters)
                if (warp == ((a + 1) & (NW - 1)) && lane < P)
                    ols_mid_parallel<P, KAL>(lane, t, midW, midX, midC, midS, tileY + 128, tileW + 128, tX + 128, prm);
            } else
            if (tid == ((a + 1) & (NW - 1)) * 32 + 31) {              // bin 128, on a warp with a light transform phase
                // its split / packing twiddle is -i: the real-signal bin is 2 conj(Z[128]), and back (mid_conj2)
                float2 mw[P], mx[P];                                  // by partition / by delay (as of block t - 1)
                float mc[PC], ms = *midS;
#pragma unroll
                for (int p = 0; p < P; ++p) {
                    mw[p] = midW[p];
                    mx[p] = midX[(t - 1 - p) & (P - 1)];
                }
#pragma unroll
                for (int p = 0; p < PC; ++p) mc[p] = midC[p];
                if (t >= 1) {
                    const float2 ek = mid_conj2(tileY[128]), ca = mid_conj2(tileW[128]);
                    const int cprev = (t - 1) & (P - 1);
#pragma unroll
                    for (int p = 0; p < P; ++p)
                        if (cprev == p) mw[p] = ca;
                    ols_update<P, KAL, false>(mw, mx, mc, ms, ek, prm);
                    *midS = ms;
#pragma unroll
                    for (int p = 0; p < PC; ++p) midC[p] = mc[p];
#pragma unroll
                    for (int p = 0; p < P; ++p) midW[p] = mw[p];
                }
                const float2 xk = mid_conj2(tX[128]);
#pragma unroll
                for (int p = P - 1; p > 0; --p) mx[p] = mx[p - 1];
                mx[0] = xk;
                midX[c] = xk;
                float2 y = make_float2(0.f, 0.f);
#pragma unroll
                for (int p = 0; p < P; ++p) y = cfma(mw[p], mx[p], y);
                tileY[128] = mid_conj2(y);
                float2 wc = mw[0];
#pragma unroll
                for (int p = 1; p < P; ++p)
                    if (c == p) wc = mw[p];
                tileW[128] = mid_conj2(wc);
            }
        }
        AEC_TICK(0);                                                  // R
        cp_async_wait<1>();                                           // blocks staged one iteration ago have landed
        __syncthreads();
        AEC_TICK(1);                                                  // wait after R
        // ---- F: the two transform slots of the chain on warp a; X_{t+1}, X_{t+2} on another warp (odd t) ----
        const bool chain = (warp == a) && (t >= 0);
        const bool xjob = (warp == ((a + NW / 2) & (NW - 1))) && (t & 1) && (t + 1 < nblk);
        if (chain || xjob) {
            float2 v[16];
            float2* tile;
            if (chain) {
                tile = half == 0 ? tileY : tileW;                     // lower half-warp: error path; upper: constraint
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = tile[h + 16 * j];
                __syncwarp();
                fft256_halfwarp_regs<true>(v, tile, twr, h);
                // register position p holds z[m], m = h + 16 r, r = fft16_index(p): samples 2m, 2m+1; the second half of
                // the 512 samples (r >= 8) is the linear-convolution part of y, the first half (r < 8) the part of g kept
                float2 u[16];
#pragma unroll
                for (int p = 0; p < 16; ++p) u[fft16_index(p)] = v[p];
                const float* dsrc = dring + (t & 1) * 256 + 2 * h;
                const float sg = half == 0 ? 0.f : 0.5f * k512;
                const bool st_v = half == 0 && prm.vec_out, st_s = half == 0 && !prm.vec_out;
                float em = 0.f, ee = 0.f;
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    const float2 y = make_float2(u[8 + r].x * k512, u[8 + r].y * k512);
                    const float2 d = *reinterpret_cast<const float2*>(dsrc + 32 * r);
                    const float2 e = make_float2(d.x - y.x, d.y - y.y);
                    {   // lower half-warp only: predicated stores, no divergent branch
                        float* dst = err_b + static_cast<long long>(t) * 256 + 2 * h + 32 * r;
                        st_stream_f2_if(dst, e, st_v);
                        st_stream_f1_if(dst, e.x, st_s);
                        st_stream_f1_if(dst + 1, e.y, st_s);
                        if constexpr (ECHO) {
                            float* dy = echo_b + static_cast<long long>(t) * 256 + 2 * h + 32 * r;
                            st_stream_f2_if(dy, y, st_v);
                            st_stream_f1_if(dy, y.x, st_s);
                            st_stream_f1_if(dy + 1, y.y, st_s);
                        }
                    }
                    em = fmaf(d.x, d.x, fmaf(d.y, d.y, em));
                    ee = fmaf(e.x, e.x, fmaf(e.y, e.y, ee));
                    v[r] = make_float2(u[r].x * sg, u[r].y * sg);                   // [g, 0_H] / [0_H, e]
                    v[8 + r] = half == 0 ? make_float2(0.5f * e.x, 0.5f * e.y) : make_float2(0.f, 0.f);
                }
                if (half == 0 && t >= prm.erle_skip_hops) {
                    acc_m += em;
                    acc_e += ee;
                }
            } else {
                // X_b = FFT[x_{b-1}, x_b], b = t + 1 (lower half-warp), t + 2 (upper); the 0.5 of the real-FFT split rides
                // on the input
                const int b1 = t + 1 + half;
                tile = tileX + (b1 & 1) * kTilePitch;
                const float* prev = xring + ((b1 - 1) & 3) * 256 + 2 * h;
                const float* cur = xring + (b1 & 3) * 256 + 2 * h;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float2 x = *reinterpret_cast<const float2*>((j < 8 ? prev : cur) + 32 * (j & 7));
                    v[j] = make_float2(0.5f * x.x, 0.5f * x.y);
                }
            }
            __syncwarp();
            fft256_halfwarp_regs<false>(v, tile, twr, h);             // one body for both roles
#pragma unroll
            for (int p = 0; p < 16; ++p) tile[h + 16 * fft16_index(p)] = v[p];
        }
#ifdef AEC_PHASE_TIMING
        if (warp == a) AEC_TICK(2); else AEC_TICK(4);                 // F as the chain warp / as another warp
#endif
        __syncthreads();
#ifdef AEC_PHASE_TIMING
        if (warp == a) AEC_TICK(3); else AEC_TICK(5);                 // wait after F
#endif
    }
    cp_async_wait<0>();

    // ---- epilogue: zero the output beyond the last whole block, ERLE ----
    zero_output_tail<ECHO>(err_b, echo_b, static_cast<long long>(nblk) * 256, prm, tid, NT);
    if (prm.erle_db != nullptr) {
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
            acc_m += __shfl_xor_sync(0xffffffffu, acc_m, o);
            acc_e += __shfl_xor_sync(0xffffffffu, acc_e, o);
        }
        if (lane == 0) {
            red[2 * warp] = acc_m;
            red[2 * warp + 1] = acc_e;
        }
        __syncthreads();
        if (tid == 0) store_erle(red, NW, prm, blockIdx.x);
    }
#ifdef AEC_PHASE_TIMING
    if (lane == 0 && prm.dbg)
        for (int i = 0; i < 12; ++i) prm.dbg[((long long)blockIdx.x * NW + warp) * 12 + i] = dbg_sm[warp][i];
#endif
}

}  // namespace aec
