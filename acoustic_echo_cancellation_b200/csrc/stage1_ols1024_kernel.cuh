// Overlap-save PBFDAF (algo 2 / 3, see stage1_ols_kernel.cuh for the recurrence and the phase structure) for frames of
// N = 1024 samples: blocks of H = 512 new samples, 513 bins -- the 48 kHz full-band configuration (BASELINE.json configs[3]).
// What differs from the frame-512 kernel is dictated by the doubled transform:
//   * a 1024-sample real transform is ONE 512-point complex FFT on a FULL warp (fft512_warp_regs), so the two chains of a
//     block run on two WARPS instead of two half-warps: warp a carries y = IFFT(Yhat)[H:], e = d - y -> HBM, E = FFT[0, e];
//     warp a + 1 carries g = IFFT(W_c), g[H:] = 0, FFT(g); warp a + 2 computes X_{t+1}.  One instruction stream serves both
//     chains (the role is a warp-uniform select), one forward-transform body serves all three warps;
//   * 4 partitions: 4 warps, two mirrored pairs (k, 512 - k) per thread; 8 partitions: 8 warps, one pair per thread (16
//     bin-taps of state per thread either way); the self-mirrored bin 256 is one lane's extra, its state in shared memory;
//   * the far-end history is the shared-memory ring of the frame-512 kernel (one float2 column per thread and bin, slot =
//     block mod P), the taps sit in rotating register positions (position j = partition (j + t) mod P).
// BUILDER-AUTHORED (the reference has no stage-1 filter): restated by oracle/aec_oracle.py:pbfdaf_ols with frame = 1024.
#pragma once
#include "stage1_ols_kernel.cuh"

namespace aec {

template <int P>
struct Ols1024Shape {
    static constexpr int NW = P;                           // 4 or 8 warps
    static constexpr int NT = 32 * NW;
    static constexpr int PPT = 256 / NT;                   // mirrored pairs per thread (2 or 1)
    static constexpr int NB = 2 * PPT;
    static constexpr int kFramePitch = 2 * kTilePitch;     // float2 per spectrum tile (512 entries + padding of the exchange)
    static constexpr size_t tile_bytes = size_t(3) * kFramePitch * sizeof(float2);        // X, Yhat / E, W_c
    static constexpr size_t blk_bytes = size_t(4 + 2) * 512 * sizeof(float);              // far-end ring [4][512], microphone [2][512]
    static constexpr size_t mid_bytes = (size_t(P) * 20 + 16 + 15) / 16 * 16 + 128;       // bin 256, ERLE partials
    static constexpr size_t hist_bytes = size_t(P) * 512 * sizeof(float2);                // far-end history ring
    static constexpr size_t total = tile_bytes + blk_bytes + mid_bytes + hist_bytes;
};

template <int P, bool KAL, bool ECHO, int REGS>
__global__ void __launch_bounds__(Ols1024Shape<P>::NT) __maxnreg__(REGS) stage1_ols1024_kernel(const Stage1Params prm) {
    static_assert(P == 4 || P == 8, "frame 1024: 4 or 8 partitions");
    using SH = Ols1024Shape<P>;
    constexpr int NW = SH::NW, NT = SH::NT, PPT = SH::PPT, NB = SH::NB, FP = SH::kFramePitch, HOP = 512;
    constexpr int PC = KAL ? P : 1;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* tileX = reinterpret_cast<float2*>(smem_raw);
    float2* tileY = tileX + FP;
    float2* tileW = tileY + FP;
    float* xring = reinterpret_cast<float*>(tileW + FP);             // [4][512] far-end blocks, slot = block & 3
    float* dring = xring + 4 * HOP;                                  // [2][512] microphone blocks, slot = block & 1
    float2* midW = reinterpret_cast<float2*>(dring + 2 * HOP);       // [P] taps of bin 256 (its own mirror), by partition
    float2* midX = midW + P;                                         // [P] its far-end history, slot = block mod P
    float* midC = reinterpret_cast<float*>(midX + P);                // [P] covariances (Kalman)
    float* midS = midC + P;                                          // [1] smoothed power / Psi
    float* red = midS + 1;                                           // [2 NW] ERLE energies of the warps
    float2* xhist = reinterpret_cast<float2*>(smem_raw + SH::tile_bytes + SH::blk_bytes + SH::mid_bytes);   // [P][NB][NT]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, h = lane & 15, hb = lane >> 4;

    const int nblk = static_cast<int>(utterance_samples(prm, blockIdx.x) / HOP);
    const float* far_b = prm.far + static_cast<long long>(blockIdx.x) * prm.in_stride;
    const float* mic_b = prm.mic + static_cast<long long>(blockIdx.x) * prm.in_stride;
    float* err_b = prm.err + static_cast<long long>(blockIdx.x) * prm.out_stride;
    float* echo_b = ECHO ? prm.echo + static_cast<long long>(blockIdx.x) * prm.out_stride : nullptr;

    if (tid < P) {
        midW[tid] = make_float2(0.f, 0.f);
        midX[tid] = make_float2(0.f, 0.f);
        midC[tid] = prm.kc0;
    }
    if (tid == 0) *midS = 0.f;
    for (int i = tid; i < HOP; i += NT) xring[3 * HOP + i] = 0.f;    // x_{-1} = 0 (slot of block -1)
    for (int i = tid; i < P * 512; i += NT) xhist[i] = make_float2(0.f, 0.f);
    __syncthreads();

    TwiddleRegs512 twr;
    twr.w1 = __ldg(&prm.tw256[1 * 32 + lane]);      // table for this kernel: [q][32] exp(-2 pi i l q / 512)
    twr.w2 = __ldg(&prm.tw256[2 * 32 + lane]);
    twr.w4 = __ldg(&prm.tw256[4 * 32 + lane]);
    twr.w8 = __ldg(&prm.tw256[8 * 32 + lane]);
    twr.wr = hb ? __ldg(&prm.tw256[16 * 32 + h]) : make_float2(1.f, 0.f);   // row 16: exp(-2 pi i a / 32)
    twr.sgn = hb ? -1.f : 1.f;

    // ---- persistent per-bin state: thread owns the mirrored pairs (k, 512 - k), k = tid + NT i ----
    float2 W[NB][P];
    float C[NB][PC], sp[NB];
    float2 wk[PPT];
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        sp[b] = 0.f;
#pragma unroll
        for (int p = 0; p < P; ++p) W[b][p] = make_float2(0.f, 0.f);
#pragma unroll
        for (int p = 0; p < PC; ++p) C[b][p] = prm.kc0;
    }
#pragma unroll
    for (int i = 0; i < PPT; ++i) wk[i] = __ldg(&prm.tw512[tid + NT * i]);      // exp(-2 pi i k / 1024)

    // block staging: 128 threads x 4 samples per signal
    auto stage_block = [&](const float* row, float* dst, int blk) {
        if (blk < nblk && tid < 128) {
            const float* p = row + static_cast<long long>(blk) * HOP + 4 * tid;
            if (prm.use_tma) {
                cp_async16(dst + 4 * tid, p);
            } else {
                *reinterpret_cast<float4*>(dst + 4 * tid) = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
            }
        }
    };
    stage_block(far_b, xring, 0);
    cp_async_commit();

    float acc_m = 0.f, acc_e = 0.f;                                   // ERLE energies (the warp of the error path)
    const float k1024 = 1.0f / 1024.0f;

    for (int t = -1; t < nblk; ++t) {
        stage_block(far_b, xring + ((t + 2) & 3) * HOP, t + 2);
        stage_block(mic_b, dring + ((t + 1) & 1) * HOP, t + 1);
        cp_async_commit();
        const int a = t & (NW - 1);                                   // error path; a + 1: constraint; a + 2: X_{t+1}
        // ---- R: update with E_{t-1}, echo estimate of block t ----
        if (t >= 0) {
            const int c = t & (P - 1);                                // partition constrained in this block = ring slot of X_t
            float2 X[NB][P];
#pragma unroll
            for (int b = 0; b < NB; ++b)
#pragma unroll
                for (int s2 = 0; s2 < P; ++s2) X[b][s2] = xhist[(s2 * NB + b) * NT + tid];
#pragma unroll
            for (int i = 0; i < PPT; ++i) {
                const int k = tid + NT * i, km = (512 - k) & 511;
                const int b0 = 2 * i, b1 = 2 * i + 1;
                if (t >= 1) {
                    float2 ek, em;
                    unpack_pair(tileY[k], tileY[km], wk[i], ek, em);
                    unpack_pair(tileW[k], tileW[km], wk[i], W[b0][0], W[b1][0]);          // the constrained partition
                    ols_update<P, KAL, true>(W[b0], X[b0], C[b0], sp[b0], ek, prm);
                    ols_update<P, KAL, true>(W[b1], X[b1], C[b1], sp[b1], em, prm);
                }
                float2 xk, xm, gk, gm;
                unpack_pair(tileX[k], tileX[km], wk[i], xk, xm);
#pragma unroll
                for (int s = 0; s < P; ++s)
                    if (c == s) {
                        X[b0][s] = xk;
                        X[b1][s] = xm;
                    }
                xhist[(c * NB + b0) * NT + tid] = xk;
                xhist[(c * NB + b1) * NT + tid] = xm;
                float2 yk = make_float2(0.f, 0.f), ym = make_float2(0.f, 0.f);
#pragma unroll
                for (int j = 0; j < P; ++j) {
                    yk = cfma(W[b0][j], X[b0][(P - j) % P], yk);
                    ym = cfma(W[b1][j], X[b1][(P - j) % P], ym);
                }
                pack_pair(yk, ym, wk[i], gk, gm);
                tileY[k] = gk;
                tileY[km] = gm;
                pack_pair(W[b0][0], W[b1][0], wk[i], gk, gm);
                tileW[k] = gk;
                tileW[km] = gm;
            }
            if constexpr (KAL && P >= 8) {                            // bin 256, one lane per tap (8-partition Kalman step)
                if (warp == ((a + 3) & (NW - 1)) && lane < P)
                    ols_mid_parallel<P, KAL>(lane, t, midW, midX, midC, midS, tileY + 256, tileW + 256, tileX + 256, prm);
            } else
            if (tid == ((a + 3) & (NW - 1)) * 32 + 31) {              // bin 256, on a warp without a transform
   // split / packing twiddle -i
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
                    const float2 ek = mid_conj2(tileY[256]), ca = mid_conj2(tileW[256]);
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
                const float2 xk = mid_conj2(tileX[256]);
#pragma unroll
                for (int p = P - 1; p > 0; --p) mx[p] = mx[p - 1];
                mx[0] = xk;
                midX[c] = xk;
                float2 y = make_float2(0.f, 0.f);
#pragma unroll
                for (int p = 0; p < P; ++p) y = cfma(mw[p], mx[p], y);
                tileY[256] = mid_conj2(y);
                float2 wc = mw[0];
#pragma unroll
                for (int p = 1; p < P; ++p)
                    if (c == p) wc = mw[p];
                tileW[256] = mid_conj2(wc);
            }
        }
        cp_async_wait<1>();                                           // blocks staged one iteration ago have landed
        __syncthreads();
        // ---- F: error path on warp a, constraint on warp a + 1, X_{t+1} on warp a + 2 ----
        const bool err_path = (warp == a) && (t >= 0);
        const bool cons_path = (warp == ((a + 1) & (NW - 1))) && (t >= 0);
        const bool xjob = (warp == ((a + 2) & (NW - 1))) && (t + 1 < nblk);
        if (err_path || cons_path || xjob) {
            float2 v[16];
            float2* tile;
            if (!xjob) {
                tile = cons_path ? tileW : tileY;
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = tile[lane + 32 * j];
                __syncwarp();
                fft512_warp_regs<true>(v, tile, twr, lane);
                // register position p holds z[m], m = lane + 32 s, s = fft16_index(p): samples 2m, 2m+1; the second half of
                // the 1024 samples (s >= 8) is the linear-convolution part of y, the first half (s < 8) the part of g kept
                float2 u[16];
#pragma unroll
                for (int p = 0; p < 16; ++p) u[fft16_index(p)] = v[p];
                const float* dsrc = dring + (t & 1) * HOP + 2 * lane;
                const float sg = cons_path ? 0.5f * k1024 : 0.f;
                const bool st_v = !cons_path && prm.vec_out, st_s = !cons_path && !prm.vec_out;
                float em = 0.f, ee = 0.f;
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    const float2 y = make_float2(u[8 + r].x * k1024, u[8 + r].y * k1024);
                    const float2 d = *reinterpret_cast<const float2*>(dsrc + 64 * r);
                    const float2 e = make_float2(d.x - y.x, d.y - y.y);
                    {   // error path only: predicated stores, no branches
                        float* dst = err_b + static_cast<long long>(t) * HOP + 2 * lane + 64 * r;
                        st_stream_f2_if(dst, e, st_v);
                        st_stream_f1_if(dst, e.x, st_s);
                        st_stream_f1_if(dst + 1, e.y, st_s);
                        if constexpr (ECHO) {
                            float* dy = echo_b + static_cast<long long>(t) * HOP + 2 * lane + 64 * r;
                            st_stream_f2_if(dy, y, st_v);
                            st_stream_f1_if(dy, y.x, st_s);
                            st_stream_f1_if(dy + 1, y.y, st_s);
                        }
                    }
                    em = fmaf(d.x, d.x, fmaf(d.y, d.y, em));
                    ee = fmaf(e.x, e.x, fmaf(e.y, e.y, ee));
                    v[r] = make_float2(u[r].x * sg, u[r].y * sg);                   // [g, 0_H] / [0_H, e]
                    v[8 + r] = cons_path ? make_float2(0.f, 0.f) : make_float2(0.5f * e.x, 0.5f * e.y);
                }
                if (!cons_path && t >= prm.erle_skip_hops) {
                    acc_m += em;
                    acc_e += ee;
                }
            } else {
                // X_{t+1} = FFT[x_t, x_{t+1}]  (the 0.5 of the real-FFT split rides on the input)
                tile = tileX;
                const float* prev = xring + (t & 3) * HOP + 2 * lane;
                const float* cur = xring + ((t + 1) & 3) * HOP + 2 * lane;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float2 x = *reinterpret_cast<const float2*>((j < 8 ? prev : cur) + 64 * (j & 7));
                    v[j] = make_float2(0.5f * x.x, 0.5f * x.y);
                }
            }
            __syncwarp();
            fft512_warp_regs<false>(v, tile, twr, lane);              // one body for the three roles
#pragma unroll
            for (int p = 0; p < 16; ++p) tile[lane + 32 * fft16_index(p)] = v[p];
        }
        __syncthreads();
    }
    cp_async_wait<0>();

    // ---- epilogue: zero the output beyond the last whole block, ERLE ----
    for (long long i = static_cast<long long>(nblk) * HOP + tid; i < prm.out_stride && i < prm.L; i += NT) {
        err_b[i] = 0.f;
        if constexpr (ECHO) echo_b[i] = 0.f;
    }
    if (prm.erle_db != nullptr) {
        warp_sum2<16>(acc_m, acc_e);
        if (lane == 0) {
            red[2 * warp] = acc_m;
            red[2 * warp + 1] = acc_e;
        }
        __syncthreads();
        if (tid == 0) store_erle(red, NW, prm, blockIdx.x);
    }
}

}  // namespace aec
