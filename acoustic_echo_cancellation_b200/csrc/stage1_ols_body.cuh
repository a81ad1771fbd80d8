// The body of both overlap-save kernels of stage1_ols_kernel.cuh, included INSIDE each __global__ function after
// `constexpr bool STREAM = ...;` (P, KAL, ECHO and prm are the kernel's).  Textual sharing rather than a __forceinline__
// function: the same body behind a call changes the one-shot kernel's instruction schedule.  Not a header of its own.
// STREAM (stage1_ols_stream_kernel): the utterance is the next chunk of a stream whose state
// (OlsStreamState) is loaded before the first block and stored after the last one.  Block t of the call is block
// T = T0 + t of the stream, and everything that depends on the block index through a partition or a ring slot -- the
// constrained partition, the history slots, the tap positions, bin 128's slots, the ERLE span -- follows T, so that every
// sum over the partitions runs in the order a single call over the whole stream would use (bit-identical outputs).
// The staging rings, output addresses and warp roles follow t.  The one-shot kernel never applies the update with the
// error of its last block; the streaming one does, in one more update-only R phase, before it stores the state.
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
    // STREAM: this row's state, the blocks it has consumed (T0), T0 mod P, and the first block of this call in the ERLE span
    unsigned char* st = STREAM ? prm.state + static_cast<long long>(blockIdx.x) * prm.state_stride : nullptr;
    const long long T0 = STREAM ? *reinterpret_cast<const long long*>(st) : 0;
    const int t0 = STREAM ? static_cast<int>(T0 & (P - 1)) : 0;
    const long long skip_rel = prm.erle_skip_hops - T0;
    const int erle_from = STREAM ? static_cast<int>(skip_rel < 0 ? 0 : (skip_rel > (1 << 30) ? (1 << 30) : skip_rel)) : 0;
    auto bin_of = [&](int b) {                                        // the bin a thread keeps in slot b of its state
        const int k = kSplit ? (tid >> 1) : tid + NT * (b >> 1);
        return (kSplit ? side : (b & 1)) ? 256 - k : k;               // k = 0: DC and Nyquist
    };
    const float2* sW = reinterpret_cast<const float2*>(st + OlsStreamState::W());
    const float2* sX = reinterpret_cast<const float2*>(st + OlsStreamState::X(P));
    const float* sS = reinterpret_cast<const float*>(st + OlsStreamState::S(P));
    const float* sC = reinterpret_cast<const float*>(st + OlsStreamState::C(P));
    constexpr int K = OlsStreamState::K;

    // Warp w of a CTA sits on scheduler (slot + w) % 4, and the warp that carries the two-transform chain is the busier
    // one.  The roles rotate over the warps every block; for the two-warp CTAs (which only ever touch one scheduler pair)
    // the warp that starts with the chain follows the hardware warp slot, so that co-resident utterances on the same
    // scheduler pair load different schedulers (same device as the bin-128 owner of the STFT-domain kernel).
    if (tid == 0) {
        unsigned hw_warp;
        asm volatile("mov.u32 %0, %%warpid;" : "=r"(hw_warp));
        *fft_warp_s = NW == 2 ? static_cast<int>((hw_warp >> 2) & 1u) : 0;
    }
    if constexpr (STREAM) {    // bin 128 by partition / ring slot (slot s holds delay (T0 - 1 - s) mod P), x_{-1}, the history
        if (tid < P) {
            midW[tid] = sW[tid * K + 128];
            midX[tid] = sX[((t0 - 1 - tid) & (P - 1)) * K + 128];
            midC[tid] = KAL ? sC[tid * K + 128] : prm.kc0;
        }
        if (tid == 0) *midS = sS[128];
        const float* sprev = reinterpret_cast<const float*>(st + OlsStreamState::prev());
        for (int i = tid; i < 256; i += NT) xring[3 * 256 + i] = sprev[i];
        if constexpr (kXs) {
#pragma unroll
            for (int s = 0; s < P; ++s)
#pragma unroll
                for (int b = 0; b < NB; ++b) xhist[(s * NB + b) * NT + tid] = sX[((t0 - 1 - s) & (P - 1)) * K + bin_of(b)];
        }
    } else {
        if (tid < P) {
            midW[tid] = make_float2(0.f, 0.f);
            midX[tid] = make_float2(0.f, 0.f);
            midC[tid] = prm.kc0;
        }
        if (tid == 0) *midS = 0.f;
        for (int i = tid; i < 256; i += NT) xring[3 * 256 + i] = 0.f;    // x_{-1} = 0 (slot of block -1)
        if constexpr (kXs)
            for (int i = tid; i < P * 256; i += NT) xhist[i] = make_float2(0.f, 0.f);
    }
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
        if constexpr (STREAM) {          // position j holds partition (j + T0) mod P; register slot s of X as xhist's
            const int k = bin_of(b);
            sp[b] = sS[k];
#pragma unroll
            for (int j = 0; j < P; ++j) {
                W[b][j] = sW[((j + t0) & (P - 1)) * K + k];
                if constexpr (!kXs) Xp[b][j] = sX[((t0 - 1 - j) & (P - 1)) * K + k];
            }
            if constexpr (KAL)
#pragma unroll
                for (int j = 0; j < P; ++j) C[b][j] = sC[((j + t0) & (P - 1)) * K + k];
        }
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

    for (int t = -1; t < nblk + (STREAM ? 1 : 0); ++t) {
        const bool fin = STREAM && t == nblk;                         // the update with E_{nblk-1} only
        stage_block(far_b, xring + ((t + 3) & 3) * 256, t + 3);
        stage_block(mic_b, dring + ((t + 1) & 1) * 256, t + 1);
        cp_async_commit();
        const int a = (fw + t) & (NW - 1);                            // the warp that carries the chain of this block
        // ---- R: update with E_{t-1}, echo estimate of block t ----
        if (t >= 0) {
            const int c = (t0 + t) & (P - 1);                         // partition constrained in this block = ring slot of X_t
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
                if (fin) continue;
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
                if (warp == ((a + 1) & (NW - 1)) && lane < P) {
                    if (fin)
                        ols_mid_parallel<P, KAL, false>(lane, t, midW, midX, midC, midS, tileY + 128, tileW + 128, tX + 128,
                                                        prm, t0);
                    else
                        ols_mid_parallel<P, KAL>(lane, t, midW, midX, midC, midS, tileY + 128, tileW + 128, tX + 128, prm, t0);
                }
            } else
            if (tid == ((a + 1) & (NW - 1)) * 32 + 31) {              // bin 128, on a warp with a light transform phase
                // its split / packing twiddle is -i: the real-signal bin is 2 conj(Z[128]), and back (mid_conj2)
                float2 mw[P], mx[P];                                  // by partition / by delay (as of block t - 1)
                float mc[PC], ms = *midS;
#pragma unroll
                for (int p = 0; p < P; ++p) {
                    mw[p] = midW[p];
                    mx[p] = midX[(t0 + t - 1 - p) & (P - 1)];
                }
#pragma unroll
                for (int p = 0; p < PC; ++p) mc[p] = midC[p];
                if (t >= 1) {
                    const float2 ek = mid_conj2(tileY[128]), ca = mid_conj2(tileW[128]);
                    const int cprev = (t0 + t - 1) & (P - 1);
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
                if (!fin) {
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
        }
        if (fin) break;
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
                if (half == 0 && t >= (STREAM ? erle_from : prm.erle_skip_hops)) {
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

    if constexpr (STREAM) {    // ---- the state after the update with E_{nblk-1}; a call without blocks leaves it ----
        if (nblk > 0) {
            __syncthreads();
            const int te = (t0 + nblk) & (P - 1);                     // positions and ring slots as of block T0 + nblk
            float2* dW = reinterpret_cast<float2*>(st + OlsStreamState::W());
            float2* dX = reinterpret_cast<float2*>(st + OlsStreamState::X(P));
            float* dS = reinterpret_cast<float*>(st + OlsStreamState::S(P));
            float* dC = reinterpret_cast<float*>(st + OlsStreamState::C(P));
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                const int k = bin_of(b);
                dS[k] = sp[b];
#pragma unroll
                for (int j = 0; j < P; ++j) {
                    dW[((j + te) & (P - 1)) * K + k] = W[b][j];
                    if constexpr (KAL) dC[((j + te) & (P - 1)) * K + k] = C[b][j];
                    if constexpr (kXs) {
                        dX[((te - 1 - j) & (P - 1)) * K + k] = xhist[(j * NB + b) * NT + tid];
                    } else {
                        dX[((te - 1 - j) & (P - 1)) * K + k] = Xp[b][j];
                    }
                }
            }
            if (tid < P) {
                dW[tid * K + 128] = midW[tid];
                dX[((te - 1 - tid) & (P - 1)) * K + 128] = midX[tid];
                if constexpr (KAL) dC[tid * K + 128] = midC[tid];
            }
            if (tid == 0) {
                dS[128] = *midS;
                *reinterpret_cast<long long*>(st) = T0 + nblk;
            }
            float* dprev = reinterpret_cast<float*>(st + OlsStreamState::prev());
            for (int i = tid; i < 256; i += NT) dprev[i] = xring[((nblk - 1) & 3) * 256 + i];
        }
    }

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
