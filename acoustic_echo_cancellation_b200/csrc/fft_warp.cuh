// Warp-level FFT building blocks for the stage-1 AEC kernels (sm_100a).
//
// A real frame of N = 512 samples is transformed through ONE 256-point complex FFT
// (even samples -> real lane, odd samples -> imaginary lane) executed by a HALF-WARP:
// 16 lanes x 16 complex points in registers, two radix-16 passes, one exchange through
// a 17-pitch padded shared-memory tile (no bank conflicts, immediate addressing).  A warp
// therefore transforms two real frames at once (far-end + microphone on analysis,
// two consecutive frames on synthesis).  The split into the real spectrum
// X[0..256] (and the inverse packing) is done by the per-bin filter threads.
//
// Conventions follow the reference STFT operators (np.fft.rfft sign, periodic Hann):
//   Stage2_lhm/scripts/network/attention_ccrn.py:8-25   (analysis / synthesis kernels)
#pragma once
#include <cuda_runtime.h>

namespace aec {

// Complex helpers are scalar FP32 (FADD / FMUL / FFMA).  The packed FADD2 / FMUL2 / FFMA2
// instructions of sm_100 were tried for all of them (one issue slot per complex add, two per
// complex multiply, +-i rotations as operand modifiers): the FFMA2 probe sustains only
// 58 TFLOP/s against 72 TFLOP/s for scalar FFMA on this B200, register pairs cost extra moves and
// spills, and the fused kernel got 4-6 % SLOWER -- see DESIGN.md "Rejected: packed FP32".
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(fmaf(-a.y, b.y, a.x * b.x), fmaf(a.y, b.x, a.x * b.y));
}
// a * conj(b)
__device__ __forceinline__ float2 cmulc(float2 a, float2 b) {
    return make_float2(fmaf(a.y, b.y, a.x * b.x), fmaf(a.y, b.x, -(a.x * b.y)));
}
// acc + a*b
__device__ __forceinline__ float2 cfma(float2 a, float2 b, float2 acc) {
    return make_float2(fmaf(-a.y, b.y, fmaf(a.x, b.x, acc.x)), fmaf(a.y, b.x, fmaf(a.x, b.y, acc.y)));
}
// acc + conj(a)*b
__device__ __forceinline__ float2 cfmac(float2 a, float2 b, float2 acc) {
    return make_float2(fmaf(a.y, b.y, fmaf(a.x, b.x, acc.x)), fmaf(-a.y, b.x, fmaf(a.x, b.y, acc.y)));
}

// MUFU.SQRT (1 ulp) for spectral magnitudes sqrt(re^2 + im^2 + 1e-9): the arguments are >= 1e-9
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// Real-FFT split and packing, written for frame 512 (the frame-1024 kernels pass 512 - k and exp(-2 pi i k/1024)).
// half-size spectra -> the two real-signal bins of the mirrored pair (k, 256-k).
// fa = Zc[k], fb = Zc[256-k], w = exp(-2 pi i k/512).  The analysis window carries the 1/2.
__device__ __forceinline__ void unpack_pair(float2 fa, float2 fb, float2 w, float2& xk, float2& xm) {
    const float2 a = make_float2(fa.x + fb.x, fa.y - fb.y);          // Zc[k] + conj Zc[256-k]
    const float2 d = make_float2(fa.y + fb.y, fb.x - fa.x);          // (Zc[k] - conj Zc[256-k]) / i
    const float2 t = cmul(w, d);
    xk = make_float2(a.x + t.x, a.y + t.y);
    xm = make_float2(a.x - t.x, t.y - a.y);                          // conj(a - t)
}
// two real-signal bins (k, 256-k) -> half-size inverse spectrum entries G[k], G[256-k]
// (scale 1/512 lives in the synthesis table).
__device__ __forceinline__ void pack_pair(float2 ek, float2 em, float2 w, float2& gk, float2& gm) {
    const float2 a = make_float2(ek.x + em.x, ek.y - em.y);          // E[k] + conj E[256-k]
    const float2 d = make_float2(ek.x - em.x, ek.y + em.y);          // E[k] - conj E[256-k]
    const float2 t = cmulc(d, w);                                    // d * conj(w)
    gk = make_float2(a.x - t.y, a.y + t.x);
    gm = make_float2(a.x + t.y, t.x - a.y);
}

// 4-point DFT in place.  INV=false: e^{-2 pi i jq/4};  INV=true: e^{+2 pi i jq/4}.
template <bool INV>
__device__ __forceinline__ void radix4(float2& a, float2& b, float2& c, float2& d) {
    const float2 s0 = cadd(a, c), d0 = csub(a, c);
    const float2 s1 = cadd(b, d), d1 = csub(b, d);
    // forward: -i*d1 = (d1.y, -d1.x);  inverse: +i*d1 = (-d1.y, d1.x)
    const float2 r = INV ? make_float2(-d1.y, d1.x) : make_float2(d1.y, -d1.x);
    a = cadd(s0, s1);
    c = csub(s0, s1);
    b = cadd(d0, r);
    d = csub(d0, r);
}

// multiply by w16^m (forward) or its conjugate (inverse), m a compile-time constant
template <int M, bool INV>
__device__ __forceinline__ float2 mul_w16(float2 v) {
    constexpr float C1 = 0.92387953251128673848f;   // cos(pi/8)
    constexpr float S1 = 0.38268343236508978178f;   // sin(pi/8)
    constexpr float R2 = 0.70710678118654752440f;   // sqrt(1/2)
    // forward twiddle w = (cr, ci) with ci <= 0 ; inverse uses (cr, -ci)
    if constexpr (M == 0) return v;
    if constexpr (M == 4) return INV ? make_float2(-v.y, v.x) : make_float2(v.y, -v.x);
    if constexpr (M == 2) {
        return INV ? make_float2(R2 * (v.x - v.y), R2 * (v.x + v.y))
                   : make_float2(R2 * (v.x + v.y), R2 * (v.y - v.x));
    }
    if constexpr (M == 6) {
        return INV ? make_float2(-R2 * (v.x + v.y), R2 * (v.x - v.y))
                   : make_float2(R2 * (v.y - v.x), -R2 * (v.x + v.y));
    }
    constexpr float cr = (M == 1) ? C1 : (M == 3) ? S1 : /*M == 9*/ -C1;
    constexpr float cif = (M == 1) ? -S1 : (M == 3) ? -C1 : /*M == 9*/ S1;
    constexpr float ci = INV ? -cif : cif;
    return make_float2(fmaf(-v.y, ci, v.x * cr), fmaf(v.y, cr, v.x * ci));
}

// 16-point DFT in place on registers.  Input v[j], j = 0..15.  On return register
// position p holds output index q = fft16_index(p) (digit reversal, compile time).
__host__ __device__ constexpr int fft16_index(int p) { return (p >> 2) + 4 * (p & 3); }

template <bool INV>
__device__ __forceinline__ void fft16(float2 (&v)[16]) {
#pragma unroll
    for (int j2 = 0; j2 < 4; ++j2) radix4<INV>(v[j2], v[4 + j2], v[8 + j2], v[12 + j2]);
    // position 4*q1 + j2 holds t[j2][q1]; twiddle by w16^(j2*q1)
    v[5] = mul_w16<1, INV>(v[5]);
    v[6] = mul_w16<2, INV>(v[6]);
    v[7] = mul_w16<3, INV>(v[7]);
    v[9] = mul_w16<2, INV>(v[9]);
    v[10] = mul_w16<4, INV>(v[10]);
    v[11] = mul_w16<6, INV>(v[11]);
    v[13] = mul_w16<3, INV>(v[13]);
    v[14] = mul_w16<6, INV>(v[14]);
    v[15] = mul_w16<9, INV>(v[15]);
#pragma unroll
    for (int q1 = 0; q1 < 4; ++q1) radix4<INV>(v[4 * q1], v[4 * q1 + 1], v[4 * q1 + 2], v[4 * q1 + 3]);
}

// Half-warp 256-point complex FFT.
//   h      : lane & 15
//   v[j]   : on entry  z[h + 16 j]                 (j = 0..15)
//            on return Z[h + 16 fft16_index(p)] in register position p
//   tile   : kTilePitch (= 272) float2 of shared memory private to this half-warp, used as the
//            exchange buffer (contents destroyed).  Rows are padded to 17 entries so both the
//            row-wise store and the column-wise load are bank-conflict free with
//            register + immediate addressing (no per-access index arithmetic).  Caller
//            guarantees every lane of the warp has finished reading whatever lived in `tile`
//            (a __syncwarp precedes).
//   tw     : global/L1 table tw[q*16 + h] = exp(-2 pi i h q / 256)
constexpr int kTilePitch = 272;

template <bool INV>
__device__ __forceinline__ void fft256_halfwarp(float2 (&v)[16], float2* tile, const float2* __restrict__ tw,
                                                int h) {
    fft16<INV>(v);
    float2* row = tile + h * 17;
    const float2* twh = tw + h;
#pragma unroll
    for (int p = 0; p < 16; ++p) {
        const int q = fft16_index(p);
        float2 x = v[p];
        if (q != 0) {
            const float2 w = __ldg(twh + q * 16);
            x = INV ? cmulc(x, w) : cmul(x, w);
        }
        row[q] = x;
    }
    __syncwarp();
    const float2* col = tile + h;
#pragma unroll
    for (int l = 0; l < 16; ++l) v[l] = col[l * 17];
    __syncwarp();
    fft16<INV>(v);
}

// Same transform with the inter-pass twiddles generated from four per-lane registers
// (w1, w2, w4, w8 = exp(-2 pi i h {1,2,4,8} / 256)) instead of a table: 11 extra complex
// multiplies per call, no memory traffic and no dependence on L1 residency.
struct TwiddleRegs {
    float2 w1, w2, w4, w8;
    // from the table tw[q*16 + h] = exp(-2 pi i h q / 256)
    static __device__ __forceinline__ TwiddleRegs load(const float2* tw, int h) {
        return {__ldg(&tw[1 * 16 + h]), __ldg(&tw[2 * 16 + h]), __ldg(&tw[4 * 16 + h]), __ldg(&tw[8 * 16 + h])};
    }
};

template <bool INV>
__device__ __forceinline__ void fft256_halfwarp_regs(float2 (&v)[16], float2* tile, const TwiddleRegs& t, int h) {
    fft16<INV>(v);
    float2* row = tile + h * 17;
    // register position of output index q (inverse of fft16_index)
    auto pos = [](int q) constexpr { return ((q & 3) << 2) | (q >> 2); };
    auto tw = [](float2 x, float2 w) { return INV ? cmulc(x, w) : cmul(x, w); };
    // q = low (+8): x_low *= w_low ; x_{low+8} *= w_low * w8.  Only one derived twiddle (w3) stays
    // live, which keeps the register footprint at the four base twiddles plus a temporary.
    row[0] = v[pos(0)];
    row[8] = tw(v[pos(8)], t.w8);
    const float2 w3 = cmul(t.w1, t.w2);
#pragma unroll
    for (int low = 1; low < 8; ++low) {
        const float2 wl = (low == 1) ? t.w1 : (low == 2) ? t.w2 : (low == 3) ? w3 : (low == 4) ? t.w4
                        : (low == 5) ? cmul(t.w1, t.w4) : (low == 6) ? cmul(t.w2, t.w4) : cmul(w3, t.w4);
        row[low] = tw(v[pos(low)], wl);
        row[low + 8] = tw(tw(v[pos(low + 8)], wl), t.w8);
    }
    __syncwarp();
    const float2* col = tile + h;
#pragma unroll
    for (int l = 0; l < 16; ++l) v[l] = col[l * 17];
    __syncwarp();
    fft16<INV>(v);
}

// ------------------------------------------------------------------------------------------
// Full-warp 512-point complex FFT (real frames of N = 1024 samples, 48 kHz configuration).
//   lane l holds z[l + 32 j] (j = 0..15).  512 = 16 (registers) x 2 (lane pair l, l^16) x 16
//   (half-warp transpose):  radix-16 over j, twiddle w512^(l q), radix-2 across the lane pair with
//   one shuffle per value (upper lanes take the difference times w32^(l & 15)), then each half-warp
//   finishes with the transposed radix-16 pass of the 256-point kernel; half-warp b produces the
//   outputs Z[h + 16 (2 s + b)], s = 0..15, in register position p with s = fft16_index(p).
//   tile: 2 * kTilePitch float2 private to the warp (two padded half tiles).
// ------------------------------------------------------------------------------------------
struct TwiddleRegs512 {
    float2 w1, w2, w4, w8;   // exp(-2 pi i l {1,2,4,8} / 512)
    float2 wr;               // lanes 16..31: exp(-2 pi i (l & 15) / 32); lanes 0..15: 1
    float sgn;               // lanes 16..31: -1 (difference); lanes 0..15: +1 (sum)
    // from the table tw[q*32 + l] = exp(-2 pi i l q / 512), q < 16, whose row 16 is exp(-2 pi i a / 32), a < 16
    static __device__ __forceinline__ TwiddleRegs512 load(const float2* tw, int lane) {
        return {__ldg(&tw[1 * 32 + lane]), __ldg(&tw[2 * 32 + lane]), __ldg(&tw[4 * 32 + lane]), __ldg(&tw[8 * 32 + lane]),
                (lane >> 4) ? __ldg(&tw[16 * 32 + (lane & 15)]) : make_float2(1.f, 0.f), (lane >> 4) ? -1.f : 1.f};
    }
};

template <bool INV>
__device__ __forceinline__ void fft512_warp_regs(float2 (&v)[16], float2* tile, const TwiddleRegs512& t, int lane) {
    fft16<INV>(v);
    const int h = lane & 15, b = lane >> 4;
    float2* row = tile + b * kTilePitch + h * 17;
    auto pos = [](int q) constexpr { return ((q & 3) << 2) | (q >> 2); };
    auto tw = [](float2 x, float2 w) { return INV ? cmulc(x, w) : cmul(x, w); };
    auto pair_step = [&](float2 x) {       // radix-2 across lanes l, l^16, then the w32 twiddle
        const float px = __shfl_xor_sync(0xffffffffu, x.x, 16);
        const float py = __shfl_xor_sync(0xffffffffu, x.y, 16);
        return tw(make_float2(fmaf(t.sgn, x.x, px), fmaf(t.sgn, x.y, py)), t.wr);
    };
    row[0] = pair_step(v[pos(0)]);
    row[8] = pair_step(tw(v[pos(8)], t.w8));
    const float2 w3 = cmul(t.w1, t.w2);
#pragma unroll
    for (int low = 1; low < 8; ++low) {
        const float2 wl = (low == 1) ? t.w1 : (low == 2) ? t.w2 : (low == 3) ? w3 : (low == 4) ? t.w4
                        : (low == 5) ? cmul(t.w1, t.w4) : (low == 6) ? cmul(t.w2, t.w4) : cmul(w3, t.w4);
        row[low] = pair_step(tw(v[pos(low)], wl));
        row[low + 8] = pair_step(tw(tw(v[pos(low + 8)], wl), t.w8));
    }
    __syncwarp();
    const float2* col = tile + b * kTilePitch + h;
#pragma unroll
    for (int a = 0; a < 16; ++a) v[a] = col[a * 17];
    __syncwarp();
    fft16<INV>(v);
}

}  // namespace aec
