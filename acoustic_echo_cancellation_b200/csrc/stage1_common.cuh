// What the stage-1 kernel families share (stage1_kernel.cuh: STFT domain, frame 512; stage1_kernel_1024.cuh: frame 1024;
// stage1_ols_kernel.cuh / stage1_ols1024_kernel.cuh: overlap-save): the parameter block, the PTX wrappers, the per-bin
// recurrence of the STFT-domain kernels, and the per-utterance contract every kernel keeps: the
// sample count (utterance_samples), the zero output tail (zero_output_tail) and the ERLE (store_erle).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "fft_warp.cuh"

namespace aec {

enum { kAlgoNlms = 0, kAlgoKalman = 1, kAlgoPbfdaf = 2, kAlgoPbfkf = 3 };

struct Stage1Params {
    const float* far;
    const float* mic;
    float* err;
    float* echo;       // nullable (only read by ECHO instantiations)
    float* erle_db;    // nullable
    const long long* n_samples;  // nullable -> every utterance has L samples
    long long B, L, in_stride, out_stride;
    float mu, delta;                         // NLMS
    float ka, ka2, kq, klam, koml, kc0, keps;  // Kalman: A, A^2, 1-A^2, lambda, 1-lambda, c0, eps
    float pblam, pboml;                        // overlap-save PBFDAF (algo 2): power smoothing lambda, 1 - lambda
    int erle_skip_hops;
    int use_tma;      // inputs 16-byte aligned per hop -> bulk copies
    int vec_out;      // outputs 8-byte aligned -> float2 stores
    int stagger_ns;   // start-up skew between utterances sharing an SM (de-synchronises the phases)
    int num_sms;
    const float2* tw256;   // [16][16]  exp(-2 pi i h q / 256) at [q*16 + h]
    const float2* tw512;   // [129]     exp(-2 pi i k / 512)
    const float2* win_a;   // [256]     0.5 * hann[2m], 0.5 * hann[2m+1]
    const float2* win_s;   // [256]     hann[n] / (512 * (coff[n] + 1e-8)), n = 2m, 2m+1
    // fused Stage-2 feature epilogue (FEAT instantiations only; Stage2_lhm/scripts/network/ERB.py:262-290, in_norm off)
    float* feat;           // [B][feat_frames][64]  cat[err_erb, |err_erb - far_erb|]
    const float* erb;      // [257][32] dense cosine bank (ERB.py:10-71), device memory
    long long feat_frames; // rows per utterance (frames of an L-sample signal)
    // streaming overlap-save builds only (stage1_ols_stream_kernel): row b's filter state at state + b * state_stride,
    // laid out as OlsStreamState says
    unsigned char* state;
    long long state_stride;
#ifdef AEC_PHASE_TIMING
    long long* dbg;        // developer build only: [B][NW][12] cycles per phase (tools/phase_timing.py)
#endif
};

// State of one stream of the frame-512 overlap-save filter after T blocks (include/aec_b200.h, DESIGN.md section 5d): the
// quantities of oracle/aec_oracle.py:pbfdaf_ols in its rfft units, K = 257 bins, every array on a 16-byte boundary.
//   blocks int64 (+ 8 reserved bytes) | prev float[256] = x_{T-1} | W complex[P][K] by partition | X complex[P][K],
//   X[p] = rfft([x_{T-2-p}, x_{T-1-p}]) | algo 2: Pw float[K] | algo 3: Psi float[K], C float[P][K] by partition
struct OlsStreamState {
    static constexpr int K = 257;
    __host__ __device__ static constexpr long long a16(long long n) { return (n + 15) / 16 * 16; }
    __host__ __device__ static constexpr long long prev() { return 16; }
    __host__ __device__ static constexpr long long W() { return prev() + 256 * 4; }
    __host__ __device__ static constexpr long long X(int P) { return W() + a16(8LL * P * K); }
    __host__ __device__ static constexpr long long S(int P) { return X(P) + a16(8LL * P * K); }     // Pw / Psi
    __host__ __device__ static constexpr long long C(int P) { return S(P) + a16(4LL * K); }         // algo 3
    __host__ __device__ static constexpr long long bytes(int P, bool kalman) {
        return kalman ? C(P) + a16(4LL * P * K) : C(P);
    }
};

// Developer instrumentation (compiled out of the product library): lane 0 of every warp accumulates
// the cycles between consecutive AEC_TICK points in shared memory.
#ifdef AEC_PHASE_TIMING
#define AEC_TICK(i)                                                   \
    do {                                                              \
        if (lane == 0) {                                              \
            const long long now_ = clock64();                         \
            dbg_sm[warp][i] += now_ - dbg_sm[warp][11];               \
            dbg_sm[warp][11] = now_;                                  \
        }                                                             \
    } while (0)
#else
#define AEC_TICK(i) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------
// mbarrier / bulk-copy (TMA) wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "AEC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra AEC_DONE;\n"
        "bra AEC_WAIT;\n"
        "AEC_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// one lane of a converged warp (SASS: ELECT); keeps the bulk-copy operands in uniform registers
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void st_stream_f2(float* p, float2 v) {
    asm volatile("st.global.cs.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream_f1(float* p, float v) {
    asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
// predicated forms: a store that only part of a warp performs, without a divergent branch around it (eight
// BSSY / BRA / BSYNC regions in the overlap-save kernels' transform chain cost ~40 cycles of branch resolution each)
__device__ __forceinline__ void st_stream_f2_if(float* p, float2 v, bool on) {
    asm volatile("{\n.reg .pred q;\nsetp.ne.u32 q, %3, 0;\n@q st.global.cs.v2.f32 [%0], {%1, %2};\n}" ::"l"(p), "f"(v.x), "f"(v.y),
                 "r"(static_cast<unsigned>(on))
                 : "memory");
}
__device__ __forceinline__ void st_stream_f1_if(float* p, float v, bool on) {
    asm volatile("{\n.reg .pred q;\nsetp.ne.u32 q, %2, 0;\n@q st.global.cs.f32 [%0], %1;\n}" ::"l"(p), "f"(v),
                 "r"(static_cast<unsigned>(on))
                 : "memory");
}

// cp.async (LDGSTS): 16 bytes global -> shared per thread without passing through registers
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src_gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// MUFU.RCP without the range fix-up code of __fdividef / the Newton step of 1.0f / x (the argument
// is a regularised power, far from the denormal / overflow ranges; 1 ulp is ample for 1e-4 parity)
__device__ __forceinline__ float rcp_fast(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// ------------------------------------------------------------------------------------------
// per-bin recurrence state, resident in registers
// ------------------------------------------------------------------------------------------
template <int P, int ALGO>
struct BinState {
    float2 W[P];   // filter taps
    float2 X[P];   // X[p] = far-end spectrum p hops ago (X[0] = current after the shift)
    float C[ALGO == kAlgoKalman ? P : 1];
    float psi;
    __device__ __forceinline__ void init(float c0) {
#pragma unroll
        for (int p = 0; p < P; ++p) {
            W[p] = make_float2(0.f, 0.f);
            X[p] = make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int p = 0; p < (ALGO == kAlgoKalman ? P : 1); ++p) C[p] = c0;
        psi = 0.f;
    }
    static constexpr int kFloats = 4 * P + (ALGO == kAlgoKalman ? P : 1) + 1;
    __device__ __forceinline__ void store(float* m) const {
#pragma unroll
        for (int p = 0; p < P; ++p) {
            m[4 * p + 0] = W[p].x; m[4 * p + 1] = W[p].y; m[4 * p + 2] = X[p].x; m[4 * p + 3] = X[p].y;
        }
#pragma unroll
        for (int p = 0; p < (ALGO == kAlgoKalman ? P : 1); ++p) m[4 * P + p] = C[p];
        m[kFloats - 1] = psi;
    }
    __device__ __forceinline__ void load(const float* m) {
#pragma unroll
        for (int p = 0; p < P; ++p) {
            W[p] = make_float2(m[4 * p + 0], m[4 * p + 1]);
            X[p] = make_float2(m[4 * p + 2], m[4 * p + 3]);
        }
#pragma unroll
        for (int p = 0; p < (ALGO == kAlgoKalman ? P : 1); ++p) C[p] = m[4 * P + p];
        psi = m[kFloats - 1];
    }
};

// One frame of the recurrence for one bin.  Operation order mirrors oracle/aec_oracle.py
// (fdaf_nlms / fdaf_kalman).
// SHIFT = false: the caller has already placed X[t-1..t-P+1] in s.X[1..P-1] (history kept in a
// shared-memory ring for long filters, so that it is not live in registers across the FFT phases).
template <int P, int ALGO, bool SHIFT = true>
__device__ __forceinline__ void bin_step(BinState<P, ALGO>& s, const float2 Xn, const float2 Y,
                                         const Stage1Params& prm, float2& E, float2& Yh) {
    if constexpr (SHIFT) {
#pragma unroll
        for (int p = P - 1; p > 0; --p) s.X[p] = s.X[p - 1];
    }
    s.X[0] = Xn;
    float2 yh = make_float2(0.f, 0.f);
#pragma unroll
    for (int p = 0; p < P; ++p) yh = cfma(s.W[p], s.X[p], yh);
    const float2 e = csub(Y, yh);
    if constexpr (ALGO == kAlgoNlms) {
        float pw = 0.f;
#pragma unroll
        for (int p = 0; p < P; ++p) pw = fmaf(s.X[p].x, s.X[p].x, fmaf(s.X[p].y, s.X[p].y, pw));
        const float g = prm.mu * rcp_fast(pw + prm.delta);
        const float2 ge = make_float2(g * e.x, g * e.y);
#pragma unroll
        for (int p = 0; p < P; ++p) s.W[p] = cfmac(s.X[p], ge, s.W[p]);
    } else {
        const float e2 = fmaf(e.x, e.x, e.y * e.y);
        s.psi = fmaf(prm.klam, s.psi, prm.koml * e2);
        // |X|^2 is recomputed in the update loop rather than kept in a P-entry array: two more
        // instructions per tap, P fewer live registers (what decides spilling at P = 16)
        float d = 0.f;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const float x2 = fmaf(s.X[p].x, s.X[p].x, s.X[p].y * s.X[p].y);
            d = fmaf(s.C[p], x2, d);
        }
        d = d + s.psi + prm.keps;
        const float rd = __frcp_rn(d);
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const float x2 = fmaf(s.X[p].x, s.X[p].x, s.X[p].y * s.X[p].y);
            const float gs = s.C[p] * rd;
            const float2 g = make_float2(gs * s.X[p].x, -gs * s.X[p].y);   // C conj(X) / D
            float2 w = cfma(g, e, s.W[p]);
            w = make_float2(prm.ka * w.x, prm.ka * w.y);
            s.W[p] = w;
            const float w2 = fmaf(w.x, w.x, w.y * w.y);
            s.C[p] = fmaf(prm.ka2 * (1.f - gs * x2), s.C[p], prm.kq * w2);
        }
    }
    E = e;
    Yh = yh;
}

// The self-mirrored bin (k = N/4 on the half-size spectrum) has the split / packing twiddle -i, for which unpack_pair /
// pack_pair reduce to 2 conj(.) -- the same values, without their multiplies by 0 and -1.
__device__ __forceinline__ float2 mid_conj2(float2 z) { return make_float2(2.f * z.x, -2.f * z.y); }

// ------------------------------------------------------------------------------------------
// per-utterance contract
// ------------------------------------------------------------------------------------------
// Copies that stay in the kernels, because calling the shared definition changes the SASS of the builds in brackets
// (instruction order and registers; the outputs would not change).  A change to a rule has to be made there too.
//   sample count        stage1_n1024_kernel [1], re-read in stage1_n512_kernel's producer [all 40]
//   zero tail           stage1_n1024_kernel [1], stage1_ols1024_kernel [6]
//   ERLE                stage1_n1024_kernel [1], stage1_n512_kernel [35] (partials per half-warp, slot half ^ 1)
//   ERLE partials       two-value lane sums in stage1_n1024_kernel [16] and stage1_ols_kernel [24] (warp_sum2)
//   hop staging         stage1_n1024_kernel's producer [16] (stage_hops)
//   block staging       the stage_block lambdas of stage1_ols_kernel [24, with its sample count folded] and
//                       stage1_ols1024_kernel [8]
//   serial mid bin      the bin-128 / bin-256 step of stage1_ols_kernel [14] and stage1_ols1024_kernel [6]
//   mid_conj2           the conj2 lambda of ols_mid_parallel (stage1_ols_kernel.cuh) [8]
//   twiddle registers   stage1_n1024_kernel [1], stage1_ols1024_kernel [8] (TwiddleRegs512::load, fft_warp.cuh)
// Samples of utterance b: n_samples[b] clamped to [0, L]; every utterance has L samples without n_samples.  (prm by value:
// inlined, the reads come straight from the kernel parameters, and the kernels' code is what it was with the clamp inline.)
__device__ __forceinline__ long long utterance_samples(const Stage1Params prm, long long b) {
    const long long n = prm.n_samples ? prm.n_samples[b] : prm.L;
    return n < 0 ? 0 : (n > prm.L ? prm.L : n);
}

// Start-up skew (stagger_ns > 0): CTA b sleeps ((b / num_sms) mod 8) * stagger_ns, so that the utterances resident on
// one SM, which start together, do not run their phases in lock-step.
__device__ __forceinline__ void startup_skew(const Stage1Params& prm) {
    if (prm.stagger_ns > 0) {
        const unsigned slot = (unsigned)(blockIdx.x / (unsigned)prm.num_sms) & 7u;
        if (slot) __nanosleep(slot * (unsigned)prm.stagger_ns);
    }
}

// The output rows are exactly zero from `valid` (the end of the utterance's last whole hop / block) up to
// min(out_stride, L).  All NT threads of the CTA.
template <bool ECHO>
__device__ __forceinline__ void zero_output_tail(float* err_row, float* echo_row, long long valid, const Stage1Params& prm,
                                                 int tid, int NT) {
    for (long long i = valid + tid; i < prm.out_stride && i < prm.L; i += NT) {
        err_row[i] = 0.f;
        if constexpr (ECHO) echo_row[i] = 0.f;
    }
}

// ERLE of utterance b, written by one thread once red[2 w] / red[2 w + 1] hold warp w's microphone / error energy over
// the hops of the ERLE span: 10 log10(max(mic, 1e-20) / max(err, 1e-20)) with the energies summed over the NW warps.
__device__ __forceinline__ void store_erle(const float* red, int NW, const Stage1Params& prm, long long b) {
    float pm = 0.f, pe = 0.f;
    for (int w = 0; w < NW; ++w) {
        pm += red[2 * w];
        pe += red[2 * w + 1];
    }
    prm.erle_db[b] = 10.f * log10f(fmaxf(pm, 1e-20f) / fmaxf(pe, 1e-20f));
}

// Hops [b0, b1] of the zero-padded far-end / microphone rows -> the staging ring stage[2][R][HOP], slot = hop mod R.
// Hop beta holds samples [(beta - 1) HOP, beta HOP); hop 0 is the left zero pad.  With use_tma a hop inside the n samples
// is one bulk copy per signal, issued by lane 0 and completed on mbar; the warp loads the other hops, zero beyond n.
template <int HOP, int R>
__device__ __forceinline__ void stage_hops(float* stage, uint64_t* mbar, const float* far_b, const float* mic_b, int b0,
                                           int b1, int n, const Stage1Params& prm, int lane) {
    if (lane == 0) {
        int nt = 0;
        for (int beta = b0; beta <= b1; ++beta) nt += (prm.use_tma && beta >= 1 && beta * HOP <= n) ? 1 : 0;
        fence_proxy_async();
        mbar_arrive_expect_tx(mbar, static_cast<uint32_t>(nt) * (8u * HOP));
        for (int beta = b0; beta <= b1; ++beta) {
            if (prm.use_tma && beta >= 1 && beta * HOP <= n) {
                const int slot = beta % R;
                tma_load_1d(stage + (0 * R + slot) * HOP, far_b + (beta - 1) * HOP, 4u * HOP, mbar);
                tma_load_1d(stage + (1 * R + slot) * HOP, mic_b + (beta - 1) * HOP, 4u * HOP, mbar);
            }
        }
    }
    for (int beta = b0; beta <= b1; ++beta) {
        if (!(prm.use_tma && beta >= 1 && beta * HOP <= n)) {
            const int slot = beta % R;
#pragma unroll
            for (int i = 0; i < HOP / 32; ++i) {
                const int o = lane + 32 * i;
                const int idx = (beta - 1) * HOP + o;
                const bool ok = beta >= 1 && idx < n;
                stage[(0 * R + slot) * HOP + o] = ok ? __ldg(far_b + idx) : 0.f;
                stage[(1 * R + slot) * HOP + o] = ok ? __ldg(mic_b + idx) : 0.f;
            }
        }
    }
}

// a and b summed over the lanes of a warp (OFF = 16) or of each half-warp (OFF = 8)
template <int OFF>
__device__ __forceinline__ void warp_sum2(float& a, float& b) {
#pragma unroll
    for (int o = OFF; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
}

}  // namespace aec
