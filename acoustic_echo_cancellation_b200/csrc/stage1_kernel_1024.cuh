// Stage-1 canceller for frames of N = 1024 samples (hop 512, 513 bins): the 48 kHz full-band
// configuration (BASELINE.json configs[3]).  Same three-phase structure as stage1_kernel.cuh;
// what differs is dictated by the doubled frame:
//   * a real frame is ONE 512-point complex FFT on a full warp (fft512_warp_regs), so the analysis
//     phase is two warp passes per frame (far end, microphone) and the synthesis phase one warp
//     pass per frame; every overlap between consecutive frames crosses warps and goes through the
//     dead spectrum tile of the earlier frame (the chunk's last tail through a 2 KB carry);
//   * 8 warps per utterance, 8 frames per chunk, every thread owns ONE mirrored pair (k, 512-k);
//     the self-mirrored bin 256 is the last thread's extra, its state in shared memory.
// STFT conventions: Stage2_lhm/scripts/network/attention_ccrn.py:8-25, 45-52, 82-101 with
// win_len = fft_len = 1024, win_inc = 512 (golden vectors: tests/golden, arrays *1024).
// The parameters, the PTX wrappers, the per-bin recurrence (BinState / bin_step) and the real-FFT split it shares with the
// frame-512 kernel live in stage1_common.cuh.
#pragma once
#include "stage1_common.cuh"

namespace aec {

struct Stage1Smem1024 {
    static constexpr int NW = 8, F = 8, R = F + 1;
    static constexpr int kFramePitch = 2 * kTilePitch;                                     // float2 per (frame, signal)
    static constexpr size_t zbuf_bytes = size_t(F) * 2 * kFramePitch * sizeof(float2);      // 69 632
    static constexpr size_t stage_bytes = size_t(2) * R * 512 * sizeof(float);              // 36 864
    static constexpr size_t win_bytes = size_t(256 + 512) * sizeof(float2);                 //  6 144
    __host__ __device__ static constexpr size_t tails_bytes(bool echo) { return size_t(echo ? 2 : 1) * 256 * sizeof(float2); }
    __host__ __device__ static constexpr size_t mid_bytes(int P) { return (size_t(P) * 20 + 4 + 15) / 16 * 16; }
    __host__ __device__ static constexpr size_t total(bool echo, int P) {
        return zbuf_bytes + stage_bytes + win_bytes + tails_bytes(echo) + mid_bytes(P) + 16;
    }
};

template <int P, int ALGO, bool ECHO, int REGS>
__global__ void __launch_bounds__(256) __maxnreg__(REGS) stage1_n1024_kernel(const Stage1Params prm) {
    using SM = Stage1Smem1024;
    constexpr int NW = SM::NW, F = SM::F, R = SM::R, NT = NW * 32, FP = SM::kFramePitch;
    constexpr int NSIG = ECHO ? 2 : 1;
    constexpr int HOP = 512;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    float2* zbuf = reinterpret_cast<float2*>(smem_raw);                                    // [F][2][FP]
    float* stage = reinterpret_cast<float*>(smem_raw + SM::zbuf_bytes);                    // [2][R][512]
    float2* win_a = reinterpret_cast<float2*>(smem_raw + SM::zbuf_bytes + SM::stage_bytes);   // [256]
    float2* win_s = win_a + 256;                                                           // [512]
    float2* carry = win_s + 512;                                                           // [NSIG][256]
    float* mid_state = reinterpret_cast<float*>(carry + NSIG * 256);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw + SM::zbuf_bytes + SM::stage_bytes + SM::win_bytes +
                                                 SM::tails_bytes(ECHO) + SM::mid_bytes(P));

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int h = lane & 15, hb = lane >> 4;
    const long long b = blockIdx.x;

    long long n_ll = prm.n_samples ? prm.n_samples[b] : prm.L;
    n_ll = n_ll < 0 ? 0 : (n_ll > prm.L ? prm.L : n_ll);
    const int n = static_cast<int>(n_ll);
    const int T = n / HOP + 1;
    const int n_chunks = (T + F - 1) / F;

    if (tid == 0) {
        mbar_init(mbar, 1);
        fence_mbar_init();
    }
    __syncthreads();

    auto row_off = [&](long long stride) {
        long long v = b * stride;
        asm volatile("" : "+l"(v));
        return v;
    };
    // hops [b0, b1] of the zero-padded signal -> staging ring (block beta = samples [(beta-1)*512, beta*512))
    auto produce = [&](int b0, int b1) {
        if (b1 > T) b1 = T;
        const long long in_off = row_off(prm.in_stride);
        const float* far_b = prm.far + in_off;
        const float* mic_b = prm.mic + in_off;
        if (lane == 0) {
            int nt = 0;
            for (int beta = b0; beta <= b1; ++beta) nt += (prm.use_tma && beta >= 1 && beta * HOP <= n) ? 1 : 0;
            fence_proxy_async();
            mbar_arrive_expect_tx(mbar, static_cast<uint32_t>(nt) * 4096u);
            for (int beta = b0; beta <= b1; ++beta) {
                if (prm.use_tma && beta >= 1 && beta * HOP <= n) {
                    const int slot = beta % R;
                    tma_load_1d(stage + (0 * R + slot) * HOP, far_b + (beta - 1) * HOP, 2048u, mbar);
                    tma_load_1d(stage + (1 * R + slot) * HOP, mic_b + (beta - 1) * HOP, 2048u, mbar);
                }
            }
        }
        for (int beta = b0; beta <= b1; ++beta) {
            if (!(prm.use_tma && beta >= 1 && beta * HOP <= n)) {
                const int slot = beta % R;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int o = lane + 32 * i;
                    const int idx = (beta - 1) * HOP + o;
                    const bool ok = beta >= 1 && idx < n;
                    stage[(0 * R + slot) * HOP + o] = ok ? __ldg(far_b + idx) : 0.f;
                    stage[(1 * R + slot) * HOP + o] = ok ? __ldg(mic_b + idx) : 0.f;
                }
            }
        }
    };
    if (warp == 0) produce(0, F);

    for (int i = tid; i < 256; i += NT) win_a[i] = __ldg(&prm.win_a[i]);
    for (int i = tid; i < 512; i += NT) win_s[i] = __ldg(&prm.win_s[i]);
    TwiddleRegs512 twr;
    twr.w1 = __ldg(&prm.tw256[1 * 32 + lane]);      // table for this kernel: [q][32] exp(-2 pi i l q / 512)
    twr.w2 = __ldg(&prm.tw256[2 * 32 + lane]);
    twr.w4 = __ldg(&prm.tw256[4 * 32 + lane]);
    twr.w8 = __ldg(&prm.tw256[8 * 32 + lane]);
    twr.wr = hb ? __ldg(&prm.tw256[16 * 32 + h]) : make_float2(1.f, 0.f);   // row 16: exp(-2 pi i a / 32)
    twr.sgn = hb ? -1.f : 1.f;

    // one mirrored pair (k, 512-k) per thread, k = tid; twiddle exp(-2 pi i k / 1024)
    BinState<P, ALGO> st[2];
    st[0].init(prm.kc0);
    st[1].init(prm.kc0);
    const float2 wk = __ldg(&prm.tw512[tid]);
    if (tid == NT - 1) {
        BinState<P, ALGO> st_mid;
        st_mid.init(prm.kc0);
        st_mid.store(mid_state);
    }
    static_assert(BinState<P, ALGO>::kFloats * sizeof(float) <= SM::mid_bytes(P), "mid-bin state does not fit");

    float acc_mic = 0.f, acc_err = 0.f;
    const bool want_erle = prm.erle_db != nullptr;

    for (int c = 0; c < n_chunks; ++c) {
        const int t0 = c * F;
        __syncthreads();
        mbar_wait(mbar, static_cast<uint32_t>(c & 1));

        // ================= phase A : analysis, 2F warp passes over 8 warps =================
#pragma unroll 1
        for (int job = warp; job < 2 * F; job += NW) {
            const int tl = job >> 1, sig = job & 1;
            const int t = t0 + tl;
            if (t < T) {
                const float* s0 = stage + (sig * R + (t % R)) * HOP + 2 * lane;
                const float* s1 = stage + (sig * R + ((t + 1) % R)) * HOP + 2 * lane;
                float2 v[16];
                float e_acc = 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float2 x = *reinterpret_cast<const float2*>((j < 8 ? s0 : s1) + 64 * (j & 7));
                    float2 w = win_a[lane + 32 * (j & 7)];               // 0.5 hann[n], n < 512
                    if (j >= 8) w = make_float2(0.5f - w.x, 0.5f - w.y);  // hann[n + 512] = 1 - hann[n]
                    v[j] = make_float2(x.x * w.x, x.y * w.y);
                    if (j >= 8) e_acc = fmaf(x.x, x.x, fmaf(x.y, x.y, e_acc));
                }
                if (want_erle && sig == 1 && t + 1 <= T - 1 && t >= prm.erle_skip_hops) acc_mic += e_acc;
                float2* tile = zbuf + (tl * 2 + sig) * FP;
                fft512_warp_regs<false>(v, tile, twr, lane);
#pragma unroll
                for (int p = 0; p < 16; ++p) tile[h + 16 * hb + 32 * fft16_index(p)] = v[p];
            }
        }
        __syncthreads();

        if (warp == 0 && c + 1 < n_chunks) produce(t0 + F + 1, t0 + 2 * F);

        // ================= phase B : per-bin recurrence =================
#pragma unroll 1
        for (int tl = 0; tl < F; ++tl) {
            if (t0 + tl < T) {
                float2* zf = zbuf + (tl * 2 + 0) * FP;
                float2* zm = zbuf + (tl * 2 + 1) * FP;
                const int k = tid, km = (512 - k) & 511;
                float2 xk, xm, yk, ym, ek, em, hk, hm, gk, gm;
                unpack_pair(zf[k], zf[km], wk, xk, xm);
                unpack_pair(zm[k], zm[km], wk, yk, ym);
                bin_step<P, ALGO>(st[0], xk, yk, prm, ek, hk);
                bin_step<P, ALGO>(st[1], xm, ym, prm, em, hm);
                pack_pair(ek, em, wk, gk, gm);
                zf[k] = gk;
                zf[km] = gm;
                if constexpr (ECHO) {
                    pack_pair(hk, hm, wk, gk, gm);
                    zm[k] = gk;
                    zm[km] = gm;
                }
                if (tid == NT - 1) {         // self-mirrored bin 256
                    xk = mid_conj2(zf[256]);
                    yk = mid_conj2(zm[256]);
                    BinState<P, ALGO> st_mid;
                    st_mid.load(mid_state);
                    bin_step<P, ALGO>(st_mid, xk, yk, prm, ek, hk);
                    st_mid.store(mid_state);
                    zf[256] = mid_conj2(ek);
                    if constexpr (ECHO) zm[256] = mid_conj2(hk);
                }
            }
        }
        __syncthreads();

        // ================= phase C : synthesis, one frame per warp =================
        const int tl = warp;
        const int t = t0 + tl;
        const long long out_off = row_off(prm.out_stride);
        float* out_b[2] = {prm.err + out_off, ECHO ? prm.echo + out_off : nullptr};
        float2 head[NSIG][8];
#pragma unroll
        for (int sgn = 0; sgn < NSIG; ++sgn) {
            float2 v[16];
            float2* tile = zbuf + (tl * 2 + sgn) * FP;
            if (t < T) {
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = tile[lane + 32 * j];
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = make_float2(0.f, 0.f);
            }
            __syncwarp();
            fft512_warp_regs<true>(v, tile, twr, lane);
            // position p holds z[m], m = h + 16 hb + 32 s, s = fft16_index(p): samples 2m, 2m+1
#pragma unroll
            for (int p = 0; p < 16; ++p) {
                const int s = fft16_index(p);
                const float2 w = win_s[h + 16 * hb + 32 * s];
                const float2 u = make_float2(v[p].x * w.x, v[p].y * w.y);
                if (s < 8) head[sgn][s] = u;
                else tile[h + 16 * hb + 32 * (s - 8)] = u;          // tail -> this frame's dead tile
            }
        }
        __syncthreads();
        // output hop t-1 = tail of frame t-1 + head of frame t
        if (t >= 1 && t <= T - 1) {
#pragma unroll
            for (int sgn = 0; sgn < NSIG; ++sgn) {
                const float2* tail_src = (warp == 0) ? carry + sgn * 256 : zbuf + ((tl - 1) * 2 + sgn) * FP;
                // conditions decided once, predicated straight-line loop body (see stage1_kernel.cuh)
                const bool vec = prm.vec_out != 0;
                float* dst = out_b[sgn] + (long long)(t - 1) * HOP + 2 * h + 32 * hb;
                float en = 0.f;
#pragma unroll
                for (int s = 0; s < 8; ++s) {
                    const float2 tl2 = tail_src[h + 16 * hb + 32 * s];
                    const float2 o = make_float2(head[sgn][s].x + tl2.x, head[sgn][s].y + tl2.y);
                    if (vec) st_stream_f2(dst + 64 * s, o);
                    else { st_stream_f1(dst + 64 * s, o.x); st_stream_f1(dst + 64 * s + 1, o.y); }
                    en = fmaf(o.x, o.x, fmaf(o.y, o.y, en));
                }
                if (sgn == 0 && t - 1 >= prm.erle_skip_hops) acc_err += en;
            }
        }
        // the last frame's tail crosses into the next chunk (warp 0 has consumed the old carry)
        if (warp == 0 && c + 1 < n_chunks) {
            __syncwarp();
#pragma unroll
            for (int sgn = 0; sgn < NSIG; ++sgn) {
                const float2* src = zbuf + ((F - 1) * 2 + sgn) * FP;
#pragma unroll
                for (int i = 0; i < 8; ++i) carry[sgn * 256 + lane + 32 * i] = src[lane + 32 * i];
            }
        }
    }

    {
        const long long valid = (long long)(T - 1) * HOP;
        float* out_b[2] = {prm.err + b * prm.out_stride, ECHO ? prm.echo + b * prm.out_stride : nullptr};
        for (long long i = valid + tid; i < prm.out_stride && i < prm.L; i += NT) {
            out_b[0][i] = 0.f;
            if constexpr (ECHO) out_b[1][i] = 0.f;
        }
    }
    if (want_erle) {
        __syncthreads();
        float* red = reinterpret_cast<float*>(zbuf);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            acc_mic += __shfl_xor_sync(0xffffffffu, acc_mic, o);
            acc_err += __shfl_xor_sync(0xffffffffu, acc_err, o);
        }
        if (lane == 0) {
            red[2 * warp] = acc_mic;
            red[2 * warp + 1] = acc_err;
        }
        __syncthreads();
        if (tid == 0) {
            float pm = 0.f, pe = 0.f;
            for (int w = 0; w < NW; ++w) {
                pm += red[2 * w];
                pe += red[2 * w + 1];
            }
            prm.erle_db[b] = 10.f * log10f(fmaxf(pm, 1e-20f) / fmaxf(pe, 1e-20f));
        }
    }
}

}  // namespace aec
