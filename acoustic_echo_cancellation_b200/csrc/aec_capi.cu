// C ABI of libaec_b200.so: configuration helpers, constant tables, the stage-1 entry points
// (device- and host-buffer variants) and the FP32 peak probe used by bench.py.
// Declarations and the reference seams each entry replaces: include/aec_b200.h.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <type_traits>
#include <vector>

#include "aec_common.cuh"
#include "stage1_launch.cuh"

namespace aec {

// ------------------------------------------------------------------------------------------
// error bookkeeping
// ------------------------------------------------------------------------------------------
static thread_local char g_cuda_err[256] = "";
static thread_local int64_t g_launches = 0;

void set_cuda_error(cudaError_t e, const char* where) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s (%s)", cudaGetErrorName(e), cudaGetErrorString(e), where);
}
void count_launch(int n) { g_launches += n; }

// ------------------------------------------------------------------------------------------
// constant tables (per device)
// ------------------------------------------------------------------------------------------
namespace {
constexpr int kMaxDevices = 64;
struct DeviceTables {
    bool ready = false;
    Tables t{};
};
DeviceTables g_tables[kMaxDevices];
std::mutex g_tables_mu;

int build_tables(DeviceTables* dt) {
    const double pi = 3.14159265358979323846;
    std::vector<float2> tw256(256), tw512(129), win_a(256), win_s(256), win_r(256);
    std::vector<float> hann(512);
    for (int q = 0; q < 16; ++q)
        for (int h = 0; h < 16; ++h) {
            const double a = -2.0 * pi * double(h * q) / 256.0;
            tw256[q * 16 + h] = make_float2((float)cos(a), (float)sin(a));
        }
    for (int k = 0; k <= 128; ++k) {
        const double a = -2.0 * pi * double(k) / 512.0;
        tw512[k] = make_float2((float)cos(a), (float)sin(a));
    }
    std::vector<double> w(512);
    for (int n = 0; n < 512; ++n) {
        w[n] = 0.5 - 0.5 * cos(2.0 * pi * n / 512.0);   // scipy get_window('hann', 512, fftbins=True)
        hann[n] = (float)w[n];
    }
    auto syn = [&](int n) {
        // every kept output sample sums exactly two frames: coff = w[n']^2 + w[n'+256]^2
        const int m = n & 255;
        const double wf = (double)(float)w[m], wb = (double)(float)w[m + 256];
        const double coff = wf * wf + wb * wb;
        return (double)(float)w[n] / (512.0 * (coff + 1e-8));
    };
    for (int m = 0; m < 256; ++m) {
        win_a[m] = make_float2((float)(0.5 * (double)(float)w[2 * m]), (float)(0.5 * (double)(float)w[2 * m + 1]));
        win_s[m] = make_float2((float)syn(2 * m), (float)syn(2 * m + 1));
        win_r[m] = make_float2((float)((double)(float)w[2 * m] / 512.0), (float)((double)(float)w[2 * m + 1] / 512.0));
    }
    // ---- frame 1024 ----
    std::vector<float2> tw512w(17 * 32), tw1024(257), win_a1k(256), win_s1k(512);
    for (int q = 0; q < 16; ++q)
        for (int l = 0; l < 32; ++l) {
            const double a = -2.0 * pi * double(l * q) / 512.0;
            tw512w[q * 32 + l] = make_float2((float)cos(a), (float)sin(a));
        }
    for (int a = 0; a < 32; ++a) {
        const double ang = -2.0 * pi * double(a) / 32.0;
        tw512w[16 * 32 + a] = make_float2((float)cos(ang), (float)sin(ang));
    }
    for (int k = 0; k <= 256; ++k) {
        const double a = -2.0 * pi * double(k) / 1024.0;
        tw1024[k] = make_float2((float)cos(a), (float)sin(a));
    }
    {
        std::vector<double> w1k(1024);
        for (int n = 0; n < 1024; ++n) w1k[n] = 0.5 - 0.5 * cos(2.0 * pi * n / 1024.0);
        auto syn1k = [&](int n) {
            const int m = n & 511;
            const double wf = (double)(float)w1k[m], wb = (double)(float)w1k[m + 512];
            return (double)(float)w1k[n] / (1024.0 * (wf * wf + wb * wb + 1e-8));
        };
        for (int m = 0; m < 256; ++m)
            win_a1k[m] = make_float2((float)(0.5 * (double)(float)w1k[2 * m]), (float)(0.5 * (double)(float)w1k[2 * m + 1]));
        for (int m = 0; m < 512; ++m) win_s1k[m] = make_float2((float)syn1k(2 * m), (float)syn1k(2 * m + 1));
    }
    char* dev = nullptr;
    AEC_CUDA_CHECK(cudaMalloc(&dev, 32768));
    size_t off = 0;
    // (a private blocking-free stream: the legacy default stream would synchronise with -- or, under stream
    //  capture, invalidate -- whatever the caller has in flight; call aec_init() before capturing a graph)
    cudaStream_t ts = nullptr;
    AEC_CUDA_CHECK(cudaStreamCreateWithFlags(&ts, cudaStreamNonBlocking));
    cudaError_t put_err = cudaSuccess;
    auto put = [&](const void* src, size_t n) -> const void* {
        void* dst = dev + off;
        const cudaError_t pe = cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, ts);
        if (put_err == cudaSuccess) put_err = pe;
        off += (n + 255) / 256 * 256;
        return dst;
    };
    dt->t.tw256 = (const float2*)put(tw256.data(), 256 * sizeof(float2));
    dt->t.tw512 = (const float2*)put(tw512.data(), 129 * sizeof(float2));
    dt->t.win_a = (const float2*)put(win_a.data(), 256 * sizeof(float2));
    dt->t.win_s = (const float2*)put(win_s.data(), 256 * sizeof(float2));
    dt->t.win_r = (const float2*)put(win_r.data(), 256 * sizeof(float2));
    dt->t.hann512 = (const float*)put(hann.data(), 512 * sizeof(float));
    dt->t.tw512w = (const float2*)put(tw512w.data(), tw512w.size() * sizeof(float2));
    dt->t.tw1024 = (const float2*)put(tw1024.data(), tw1024.size() * sizeof(float2));
    dt->t.win_a1k = (const float2*)put(win_a1k.data(), win_a1k.size() * sizeof(float2));
    dt->t.win_s1k = (const float2*)put(win_s1k.data(), win_s1k.size() * sizeof(float2));
    if (put_err == cudaSuccess) put_err = cudaStreamSynchronize(ts);    // the host vectors die with this scope
    (void)cudaStreamDestroy(ts);
    if (put_err != cudaSuccess) {
        set_cuda_error(put_err, "constant tables upload");
        (void)cudaFree(dev);
        return AEC_ECUDA;
    }
    dt->ready = true;
    return AEC_OK;
}
}  // namespace

int get_tables(Tables* out) {
    int dev = -1;
    AEC_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices) return AEC_ENODEVICE;
    std::lock_guard<std::mutex> lock(g_tables_mu);
    if (!g_tables[dev].ready) {
        cudaDeviceProp prop{};
        AEC_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
        if (prop.major != 10) {
            snprintf(g_cuda_err, sizeof(g_cuda_err), "device %d is sm_%d%d; this library is built for sm_100a only", dev,
                     prop.major, prop.minor);
            return AEC_ENODEVICE;
        }
        const int rc = build_tables(&g_tables[dev]);
        if (rc != AEC_OK) return rc;
    }
    *out = g_tables[dev].t;
    return AEC_OK;
}

// ------------------------------------------------------------------------------------------
// FP32 peak probe: 8 independent FFMA chains per thread, every SM full
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ffma_peak_kernel(float* out, int iters, float a, float b) {
    float r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = (float)threadIdx.x * 1e-3f + i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = fmaf(r[i], a, b);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += r[i];
    if (s == 123.456f) out[0] = s;   // never true; keeps the chains alive
}

// same probe with the packed FFMA2 instruction (2 FP32 FMAs per issue slot)
__global__ void __launch_bounds__(256) ffma2_peak_kernel(float* out, int iters, float a, float b) {
    float2 r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = make_float2((float)threadIdx.x * 1e-3f + i, (float)threadIdx.x * 2e-3f - i);
    const float2 a2 = make_float2(a, a * 0.999f), b2 = make_float2(b, -b);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = __ffma2_rn(r[i], a2, b2);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += r[i].x + r[i].y;
    if (s == 123.456f) out[0] = s;
}

// int16 PCM -> float32 in [-1, 1): x / 32768, the scaling of librosa / soundfile
__global__ void __launch_bounds__(256) pcm16_to_f32_kernel(const int16_t* __restrict__ src, float* __restrict__ dst,
                                                           long long n_pairs) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += stride) {
        const short2 v = reinterpret_cast<const short2*>(src)[i];
        reinterpret_cast<float2*>(dst)[i] = make_float2((float)v.x * (1.0f / 32768.0f), (float)v.y * (1.0f / 32768.0f));
    }
}

}  // namespace aec

using namespace aec;

// ------------------------------------------------------------------------------------------
// plain helpers
// ------------------------------------------------------------------------------------------
extern "C" int aec_version(void) { return AEC_B200_VERSION; }

extern "C" int aec_init(void) {
    Tables t;
    return get_tables(&t);
}

extern "C" const char* aec_strerror(int code) {
    switch (code) {
        case AEC_OK: return "ok";
        case AEC_EINVAL: return "invalid argument";
        case AEC_EUNSUPPORTED: return "frame/partitions/algo combination not built into libaec_b200";
        case AEC_ECUDA: return "CUDA runtime error (see aec_last_cuda_error)";
        case AEC_ENODEVICE: return "no usable sm_100 CUDA device is current";
        case AEC_ENOMEM: return "out of memory";
        case AEC_EIO: return "file could not be opened or read";
        default: return "unknown aec error";
    }
}

extern "C" const char* aec_last_cuda_error(void) { return g_cuda_err; }

extern "C" int aec_cfg_default(aec_cfg* cfg, int32_t frame) {
    if (!cfg || (frame != 512 && frame != 1024)) return AEC_EINVAL;
    memset(cfg, 0, sizeof(*cfg));
    cfg->frame = frame;
    cfg->partitions = 4;
    cfg->algo = AEC_ALGO_NLMS;
    cfg->mu = 0.5f;
    cfg->delta = 1e-6f * (float)frame;
    cfg->kalman_a = 0.999f;
    cfg->kalman_lambda = 0.9f;
    cfg->kalman_c0 = 1.0f;
    cfg->kalman_eps = 1e-10f;
    cfg->pb_lambda = 0.5f;
    cfg->erle_skip_hops = 0;
    cfg->variant = 0;
    return AEC_OK;
}

extern "C" int64_t aec_num_frames(int64_t n_samples, int32_t frame) {
    if (n_samples < 0 || frame <= 0 || (frame & 1)) return AEC_EINVAL;
    const int64_t hop = frame / 2;
    const int64_t padded = n_samples + 2 * (frame - hop);
    if (padded < frame) return 0;
    return (padded - frame) / hop + 1;
}

extern "C" int64_t aec_out_samples(int64_t n_samples, int32_t frame) {
    const int64_t t = aec_num_frames(n_samples, frame);
    if (t < 0) return t;
    return t > 0 ? (t - 1) * (frame / 2) : 0;
}

extern "C" int64_t aec_launch_count(int reset) {
    const int64_t v = g_launches;
    if (reset) g_launches = 0;
    return v;
}

// ------------------------------------------------------------------------------------------
// stage 1, device buffers
// ------------------------------------------------------------------------------------------
static int validate_cfg(const aec_cfg* cfg) {
    if (!cfg) return AEC_EINVAL;
    if (cfg->frame != 512 && cfg->frame != 1024) return AEC_EUNSUPPORTED;
    if (cfg->partitions < 1) return AEC_EINVAL;
    if (cfg->algo != AEC_ALGO_NLMS && cfg->algo != AEC_ALGO_KALMAN && cfg->algo != AEC_ALGO_PBFDAF && cfg->algo != AEC_ALGO_PBFKF)
        return AEC_EINVAL;
    if (cfg->erle_skip_hops < 0) return AEC_EINVAL;
    return AEC_OK;
}

#ifdef AEC_PHASE_TIMING
// developer build only (tools/phase_timing.py): device buffer [B][NW][12] of per-phase cycle counts
static long long* g_phase_buffer = nullptr;
extern "C" void aec_debug_set_phase_buffer(void* p) { g_phase_buffer = static_cast<long long*>(p); }
#endif

static int stage1_run_impl(const float* far, const float* mic, float* err, float* echo_est, float* erle_db,
                           const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride, int64_t out_stride,
                           const aec_cfg* cfg, void* cuda_stream, float* feat, const float* erb) {
    int rc = validate_cfg(cfg);
    if (rc != AEC_OK) return rc;
    if (B < 0 || L < 0 || in_stride < L || out_stride < L) return AEC_EINVAL;
    if (B == 0) return AEC_OK;
    if (!far || !mic || !err) return AEC_EINVAL;
    if (feat) {
        if (!erb || echo_est) return AEC_EINVAL;
        if (cfg->frame != 512) return AEC_EUNSUPPORTED;      // the reference's ERB configuration is 257 bins
    }
    if (B > 0x7fffffffLL || L > 0x3fffffffLL) return AEC_EINVAL;
    Tables tab;
    rc = get_tables(&tab);
    if (rc != AEC_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);

    Stage1Params p{};
    p.far = far;
    p.mic = mic;
    p.err = err;
    p.echo = echo_est;
    p.erle_db = erle_db;
    p.n_samples = reinterpret_cast<const long long*>(n_samples);
    p.B = B;
    p.L = L;
    p.in_stride = in_stride;
    p.out_stride = out_stride;
    p.mu = cfg->mu;
    p.delta = cfg->delta;
    p.ka = cfg->kalman_a;
    p.ka2 = cfg->kalman_a * cfg->kalman_a;
    p.kq = (float)(1.0 - (double)cfg->kalman_a * (double)cfg->kalman_a);
    p.klam = cfg->kalman_lambda;
    p.koml = 1.0f - cfg->kalman_lambda;
    p.kc0 = cfg->kalman_c0;
    p.keps = cfg->kalman_eps;
    p.pblam = cfg->pb_lambda;
    p.pboml = 1.0f - cfg->pb_lambda;
    p.erle_skip_hops = cfg->erle_skip_hops;
    p.feat = feat;
    p.erb = erb;
    p.feat_frames = aec_num_frames(L, cfg->frame);
#ifdef AEC_PHASE_TIMING
    p.dbg = g_phase_buffer;
#endif
    auto aligned = [](const void* ptr, size_t a) { return (reinterpret_cast<uintptr_t>(ptr) & (a - 1)) == 0; };
    p.use_tma = (aligned(far, 16) && aligned(mic, 16) && (in_stride % 4) == 0) ? 1 : 0;
    p.vec_out = (aligned(err, 8) && (!echo_est || aligned(echo_est, 8)) && (out_stride % 2) == 0) ? 1 : 0;
    {
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        p.num_sms = sms > 0 ? sms : 148;
        p.stagger_ns = cfg->stagger_ns < 0 ? 0 : cfg->stagger_ns;   // off unless a positive skew is asked for
    }
    const bool wide = cfg->frame == 1024;
    p.tw256 = wide ? tab.tw512w : tab.tw256;
    p.tw512 = wide ? tab.tw1024 : tab.tw512;
    p.win_a = wide ? tab.win_a1k : tab.win_a;
    p.win_s = wide ? tab.win_s1k : tab.win_s;

    // The build to run.  A variant (1000 * warps_per_utterance + register cap, e.g. 2168) names one; 0 asks for the
    // default, the first build the unit lists for (P, algo, echo) at the warp count chosen here.  A build that was not
    // compiled is refused before anything is launched, never replaced by another.
    const int P = cfg->partitions;
    const bool ols = cfg->algo == AEC_ALGO_PBFDAF || cfg->algo == AEC_ALGO_PBFKF;
    int nw = 0, regs = 0;
    if (cfg->variant > 0) {
        if (cfg->variant < 1000) return AEC_EUNSUPPORTED;        // a register cap alone names no build
        if (feat || (wide && ols)) return AEC_EUNSUPPORTED;      // these builds follow from P, algo and the batch size
        nw = cfg->variant / 1000;
        regs = cfg->variant % 1000;
    }
    Stage1Launch (*lookup)(int P, int algo, bool echo, int nw, int regs) = nullptr;
    if (feat) {
        lookup = stage1_build_feat;
        // 4-partition NLMS: five utterances per SM (168 registers) win on many-wave batches (4144 x 10 s: 8.79 vs
        // 9.36 ms); for batches of a wave or two the launch ends with a thin last wave either way and four per SM at 200
        // registers are faster (1024 x 10 s: 2.61 vs 2.88 ms).
        if (P == 4 && cfg->algo == AEC_ALGO_NLMS) regs = B >= 20LL * p.num_sms ? 168 : 200;
    } else if (ols) {
        lookup = wide ? stage1_build_ols1024 : stage1_build_ols;
    } else if (wide) {
        lookup = stage1_build_1024;
    } else {
        // measured defaults (DESIGN.md): short filters 2 warps / 2 pairs per thread; 8 partitions and
        // more: 8 warps, one bin per thread (since bin 128 of the ring kernels runs one chunk ahead on the idle
        // synthesis warps this also holds for the 16-partition NLMS filter: 5.71 ms per 2048 x 10 s against 5.95
        // for the 4-warp / 255-register kernel, which remains available as variant 4255)
        if (nw == 0) nw = P <= 4 ? 2 : 8;
        switch (nw) {
            case 1: lookup = stage1_build_nw1; break;
            case 2: lookup = stage1_build_nw2; break;
            case 4: lookup = stage1_build_nw4; break;
            case 8: lookup = stage1_build_nw8; break;
            default: return AEC_EUNSUPPORTED;
        }
    }
    const Stage1Launch launch = lookup(P, cfg->algo, echo_est != nullptr, nw, regs);
    if (!launch) return AEC_EUNSUPPORTED;
    const cudaError_t e = launch(p, s);
    if (e != cudaSuccess) {
        set_cuda_error(e, "stage1 kernel launch");
        return AEC_ECUDA;
    }
    count_launch();
    return AEC_OK;
}

extern "C" int aec_stage1_run(const float* far, const float* mic, float* err, float* echo_est, float* erle_db,
                              const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride, int64_t out_stride,
                              const aec_cfg* cfg, void* cuda_stream) {
    return stage1_run_impl(far, mic, err, echo_est, erle_db, n_samples, B, L, in_stride, out_stride, cfg, cuda_stream,
                           nullptr, nullptr);
}

extern "C" int aec_stage1_run_features(const float* far, const float* mic, float* err, float* erle_db, float* feat,
                                       const float* erb, const int64_t* n_samples, int64_t B, int64_t L,
                                       int64_t in_stride, int64_t out_stride, const aec_cfg* cfg, void* cuda_stream) {
    if (!feat || !erb) return AEC_EINVAL;
    return stage1_run_impl(far, mic, err, nullptr, erle_db, n_samples, B, L, in_stride, out_stride, cfg, cuda_stream, feat,
                           erb);
}

// ------------------------------------------------------------------------------------------
// stage 1, host buffers: H2D -> kernel -> D2H pipeline, several slices in flight
// ------------------------------------------------------------------------------------------
// Every slot is one stream running H2D -> kernel -> D2H for one slice; a slice of 64 utterances keeps the
// GPU busy for ~0.65 ms (the latency of one utterance) between copies of 0.75-1.5 ms per direction, so two
// slots leave both DMA engines idle part of the time; four keep them saturated (profiles/r2_pcie_floor.md).
constexpr int kMaxSlots = 8;
constexpr int kDefaultSlots = 4;

struct aec_host_ctx {
    int device = 0;
    int slots = kDefaultSlots;
    int ramp = 1;            // taper the first slices as well as the last ones
    int64_t slice = 0;       // utterances per slice
    int64_t max_samples = 0;
    int64_t stride = 0;      // device row stride (multiple of 4 floats)
    cudaStream_t stream[kMaxSlots] = {};
    float* d_far[kMaxSlots] = {};
    float* d_mic[kMaxSlots] = {};
    float* d_err[kMaxSlots] = {};
    float* d_echo[kMaxSlots] = {};     // allocated on the first call that asks for the echo estimate
    float* d_erle[kMaxSlots] = {};
    long long* d_n[kMaxSlots] = {};
    int16_t* d_pcm[kMaxSlots] = {};    // [2 signals][slice][stride] int16 staging (allocated on first use)
    float* d_falign[kMaxSlots] = {};   // aligned far end, allocated on the first call that aligns
    int32_t* d_shift[kMaxSlots] = {};  // per-utterance shift / peak of the aligned calls (with d_falign)
    float* d_peak[kMaxSlots] = {};
    // page-locked staging for the small per-utterance arrays: a copy to / from pageable host memory
    // would serialise the multi-stream pipeline
    float* h_erle[kMaxSlots] = {};
    long long* h_n[kMaxSlots] = {};
    int32_t* h_shift[kMaxSlots] = {};  // (with d_falign)
    float* h_peak[kMaxSlots] = {};
    int64_t pending_off[kMaxSlots];    // slice whose ERLE / shift / peak still sit in h_erle[k] .. (-1: none)
    int64_t pending_nb[kMaxSlots] = {};
    float* pending_dst[kMaxSlots] = {}; // ... and the caller's erle_db array it belongs to (calls may overlap: deferred mode)
    int32_t* pending_shift[kMaxSlots] = {};   // ... the caller's shift_out / peak_out arrays
    float* pending_peak[kMaxSlots] = {};
    int deferred = 0;                  // 1: a run call returns without waiting for its last slices (aec_host_ctx_wait does)
    aec_host_ctx() {
        for (int i = 0; i < kMaxSlots; ++i) pending_off[i] = -1;
    }
};

// Utterances of the next slice.  What precedes the first download (upload of the first slice, the 0.65 ms
// latency of one utterance) and what follows the last upload (kernel, download) is pure ramp / tail, so the
// first slices grow (16, 32, 64, ..) and the last ones shrink (.., 64, 32, 16, 16) around full-size slices.
static int64_t host_slice(const aec_host_ctx* ctx, int64_t done, int64_t remaining) {
    int64_t cap = ctx->slice;
    if (ctx->ramp && remaining > 2 * ctx->slice) {
        const int64_t grow = done < 16 ? 16 : done;           // 16, 16 -> 32, 32 -> 64, ...
        if (grow < cap) cap = grow;
    }
    if (remaining > cap) return cap;              // (never more than the context's capacity)
    if (remaining <= 16) return remaining;
    return (remaining + 1) / 2;
}

// drain slot k: wait for its stream, hand the staged ERLE values to the caller (of the call that produced them)
static int host_ctx_drain(aec_host_ctx* ctx, int k) {
    const cudaError_t e = cudaStreamSynchronize(ctx->stream[k]);
    if (e == cudaSuccess && ctx->pending_off[k] >= 0) {
        const int64_t off = ctx->pending_off[k], nb = ctx->pending_nb[k];
        if (ctx->pending_dst[k]) memcpy(ctx->pending_dst[k] + off, ctx->h_erle[k], (size_t)nb * sizeof(float));
        if (ctx->pending_shift[k]) memcpy(ctx->pending_shift[k] + off, ctx->h_shift[k], (size_t)nb * sizeof(int32_t));
        if (ctx->pending_peak[k]) memcpy(ctx->pending_peak[k] + off, ctx->h_peak[k], (size_t)nb * sizeof(float));
    }
    ctx->pending_off[k] = -1;
    ctx->pending_dst[k] = nullptr;
    ctx->pending_shift[k] = nullptr;
    ctx->pending_peak[k] = nullptr;
    if (e != cudaSuccess) {
        set_cuda_error(e, "aec_stage1_run_host: cudaStreamSynchronize");
        return AEC_ECUDA;
    }
    return AEC_OK;
}

// failure path: nothing of this call may still be in flight towards the caller's buffers when it returns,
// and no stale ERLE slice may survive into the next call
static void host_ctx_quiesce(aec_host_ctx* ctx) {
    for (int i = 0; i < ctx->slots; ++i) {
        if (ctx->stream[i]) (void)cudaStreamSynchronize(ctx->stream[i]);
        ctx->pending_off[i] = -1;
        ctx->pending_dst[i] = nullptr;
        ctx->pending_shift[i] = nullptr;
        ctx->pending_peak[i] = nullptr;
    }
    (void)cudaGetLastError();
}

extern "C" int aec_host_ctx_destroy(aec_host_ctx* ctx) {
    if (!ctx) return AEC_OK;
    int prev = -1;
    (void)cudaGetDevice(&prev);
    (void)cudaSetDevice(ctx->device);
    for (int i = 0; i < kMaxSlots; ++i) {
        if (ctx->stream[i]) cudaStreamSynchronize(ctx->stream[i]);
        cudaFree(ctx->d_far[i]);
        cudaFree(ctx->d_mic[i]);
        cudaFree(ctx->d_err[i]);
        cudaFree(ctx->d_echo[i]);
        cudaFree(ctx->d_erle[i]);
        cudaFree(ctx->d_n[i]);
        cudaFree(ctx->d_pcm[i]);
        cudaFree(ctx->d_falign[i]);
        cudaFree(ctx->d_shift[i]);
        cudaFree(ctx->d_peak[i]);
        cudaFreeHost(ctx->h_erle[i]);
        cudaFreeHost(ctx->h_n[i]);
        cudaFreeHost(ctx->h_shift[i]);
        cudaFreeHost(ctx->h_peak[i]);
        if (ctx->stream[i]) cudaStreamDestroy(ctx->stream[i]);
    }
    if (prev >= 0) (void)cudaSetDevice(prev);
    delete ctx;
    return AEC_OK;
}

extern "C" int aec_host_ctx_create_ex(aec_host_ctx** out, int64_t slice_utterances, int64_t max_samples, int32_t slots,
                                      int32_t flags) {
    if (!out || slice_utterances <= 0 || max_samples <= 0 || slots < 0 || slots > kMaxSlots) return AEC_EINVAL;
    aec_host_ctx* ctx = new (std::nothrow) aec_host_ctx();
    if (!ctx) return AEC_ENOMEM;
    ctx->slots = slots == 0 ? kDefaultSlots : slots;
    ctx->ramp = (flags & AEC_HOST_CTX_NO_RAMP) ? 0 : 1;
    ctx->slice = slice_utterances;
    ctx->max_samples = max_samples;
    ctx->stride = (max_samples + 3) / 4 * 4;
    cudaError_t e = cudaGetDevice(&ctx->device);
    const size_t sig = (size_t)ctx->slice * (size_t)ctx->stride * sizeof(float);
    for (int i = 0; i < ctx->slots && e == cudaSuccess; ++i) {
        e = cudaStreamCreateWithFlags(&ctx->stream[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_far[i], sig);
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_mic[i], sig);
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_err[i], sig);
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_erle[i], (size_t)ctx->slice * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_n[i], (size_t)ctx->slice * sizeof(long long));
        if (e == cudaSuccess) e = cudaHostAlloc(&ctx->h_erle[i], (size_t)ctx->slice * sizeof(float), cudaHostAllocDefault);
        if (e == cudaSuccess) e = cudaHostAlloc(&ctx->h_n[i], (size_t)ctx->slice * sizeof(long long), cudaHostAllocDefault);
    }
    if (e != cudaSuccess) {
        set_cuda_error(e, "aec_host_ctx_create");
        aec_host_ctx_destroy(ctx);
        (void)cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? AEC_ENOMEM : AEC_ECUDA;
    }
    *out = ctx;
    return AEC_OK;
}

extern "C" int aec_host_ctx_wait(aec_host_ctx* ctx) {
    if (!ctx) return AEC_EINVAL;
    int rc = AEC_OK;
    for (int i = 0; i < ctx->slots; ++i) {
        const int r = host_ctx_drain(ctx, i);
        if (r != AEC_OK && rc == AEC_OK) rc = r;
    }
    if (rc != AEC_OK) {
        host_ctx_quiesce(ctx);
        return rc;
    }
    AEC_CUDA_CHECK(cudaGetLastError());
    return AEC_OK;
}

extern "C" int aec_host_ctx_set_deferred(aec_host_ctx* ctx, int32_t deferred) {
    if (!ctx) return AEC_EINVAL;
    ctx->deferred = deferred ? 1 : 0;
    return AEC_OK;
}

extern "C" int aec_host_ctx_create(aec_host_ctx** out, int64_t slice_utterances, int64_t max_samples) {
    return aec_host_ctx_create_ex(out, slice_utterances, max_samples, 0, 0);
}

namespace {
// One body for both host entries: In = float (samples as librosa.load returns them) or int16_t (the PCM the wav
// files hold; converted on the GPU).  align = NULL: no delay estimate, no copies or launches beyond stage 1's.
template <typename In>
int run_host_impl(aec_host_ctx* ctx, const In* far, const In* mic, float* err, float* echo_est, float* erle_db,
                  const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride, int64_t out_stride,
                  const aec_cfg* cfg, const aec_delay_cfg* align, int32_t* shift_out, float* peak_out) {
    constexpr bool kPcm = std::is_same<In, int16_t>::value;
    if (!ctx) return AEC_EINVAL;
    int rc = validate_cfg(cfg);
    if (rc != AEC_OK) return rc;
    if (align) {
        rc = validate_delay_cfg(align);
        if (rc != AEC_OK) return rc;
    } else if (shift_out || peak_out) {
        return AEC_EINVAL;
    }
    if (B < 0 || L < 0 || L > ctx->max_samples || in_stride < L || out_stride < L) return AEC_EINVAL;
    if (B == 0) return AEC_OK;
    if (!far || !mic || !err) return AEC_EINVAL;
    int dev = -1;
    AEC_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev != ctx->device) return AEC_EINVAL;     // the context's streams and buffers belong to ctx->device
    const size_t sig_elems = (size_t)ctx->slice * (size_t)ctx->stride;     // elements per signal per slot
    for (int i = 0; i < ctx->slots; ++i) {
        if (echo_est && !ctx->d_echo[i]) AEC_CUDA_CHECK(cudaMalloc(&ctx->d_echo[i], sig_elems * sizeof(float)));
        if (kPcm && !ctx->d_pcm[i]) AEC_CUDA_CHECK(cudaMalloc(&ctx->d_pcm[i], 2 * sig_elems * sizeof(int16_t)));
        if (align && !ctx->d_falign[i]) {
            AEC_CUDA_CHECK(cudaMalloc(&ctx->d_falign[i], sig_elems * sizeof(float)));
            AEC_CUDA_CHECK(cudaMalloc(&ctx->d_shift[i], (size_t)ctx->slice * sizeof(int32_t)));
            AEC_CUDA_CHECK(cudaMalloc(&ctx->d_peak[i], (size_t)ctx->slice * sizeof(float)));
            AEC_CUDA_CHECK(cudaHostAlloc(&ctx->h_shift[i], (size_t)ctx->slice * sizeof(int32_t), cudaHostAllocDefault));
            AEC_CUDA_CHECK(cudaHostAlloc(&ctx->h_peak[i], (size_t)ctx->slice * sizeof(float), cudaHostAllocDefault));
        }
    }
    int sms = 148;
    (void)cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    const size_t in_row = (size_t)L * sizeof(In), out_row = (size_t)L * sizeof(float);
    const size_t in_spitch = (size_t)in_stride * sizeof(In), in_dpitch = (size_t)ctx->stride * sizeof(In);
    const size_t out_pitch = (size_t)out_stride * sizeof(float), dpitch = (size_t)ctx->stride * sizeof(float);
    // contiguous rows on both sides -> one linear copy per signal (the DMA engines run linear copies at full
    // PCIe rate; pitched copies are only used for strided host layouts)
    const bool lin_in = (in_stride == L) && (ctx->stride == L);
    const bool lin_out = (out_stride == L) && (ctx->stride == L);
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) {
        if (e == cudaSuccess && r != cudaSuccess) e = r;
        return e == cudaSuccess;
    };
    int64_t nb = 0;
    for (int64_t off = 0, it = 0; off < B && rc == AEC_OK && e == cudaSuccess; off += nb, ++it) {
        const int k = (int)(it % ctx->slots);
        nb = host_slice(ctx, off, B - off);
        cudaStream_t s = ctx->stream[k];
        rc = host_ctx_drain(ctx, k);                // slot k's previous slice (`slots` slices ago, maybe of the previous call) is done
        if (rc != AEC_OK) break;
        In* up_f = kPcm ? reinterpret_cast<In*>(ctx->d_pcm[k]) : reinterpret_cast<In*>(ctx->d_far[k]);
        In* up_m = kPcm ? reinterpret_cast<In*>(ctx->d_pcm[k]) + sig_elems : reinterpret_cast<In*>(ctx->d_mic[k]);
        if (lin_in) {
            ok(cudaMemcpyAsync(up_f, far + off * in_stride, in_row * (size_t)nb, cudaMemcpyHostToDevice, s));
            ok(cudaMemcpyAsync(up_m, mic + off * in_stride, in_row * (size_t)nb, cudaMemcpyHostToDevice, s));
        } else {
            ok(cudaMemcpy2DAsync(up_f, in_dpitch, far + off * in_stride, in_spitch, in_row, (size_t)nb,
                                 cudaMemcpyHostToDevice, s));
            ok(cudaMemcpy2DAsync(up_m, in_dpitch, mic + off * in_stride, in_spitch, in_row, (size_t)nb,
                                 cudaMemcpyHostToDevice, s));
        }
        if (!ok(cudaSuccess)) break;
        if (kPcm) {
            const long long pairs = (long long)nb * ctx->stride / 2;          // stride is a multiple of 4
            pcm16_to_f32_kernel<<<sms * 4, 256, 0, s>>>(ctx->d_pcm[k], ctx->d_far[k], pairs);
            pcm16_to_f32_kernel<<<sms * 4, 256, 0, s>>>(ctx->d_pcm[k] + sig_elems, ctx->d_mic[k], pairs);
            count_launch(2);
        }
        if (n_samples) {
            memcpy(ctx->h_n[k], n_samples + off, (size_t)nb * sizeof(int64_t));
            if (!ok(cudaMemcpyAsync(ctx->d_n[k], ctx->h_n[k], (size_t)nb * sizeof(int64_t), cudaMemcpyHostToDevice, s)))
                break;
        }
        const int64_t* d_n = n_samples ? reinterpret_cast<const int64_t*>(ctx->d_n[k]) : nullptr;
        const float* far_s1 = ctx->d_far[k];
        if (align) {
            rc = aec_delay_estimate(ctx->d_far[k], ctx->d_mic[k], d_n, nb, L, ctx->stride, align, nullptr,
                                    ctx->d_shift[k], ctx->d_peak[k], nullptr, s);
            if (rc == AEC_OK)
                rc = aec_delay_align(ctx->d_far[k], ctx->d_falign[k], ctx->d_shift[k], nb, L, ctx->stride, ctx->stride, s);
            if (rc != AEC_OK) break;
            far_s1 = ctx->d_falign[k];
        }
        rc = aec_stage1_run(far_s1, ctx->d_mic[k], ctx->d_err[k], echo_est ? ctx->d_echo[k] : nullptr,
                            erle_db ? ctx->d_erle[k] : nullptr, d_n, nb, L, ctx->stride, ctx->stride, cfg, s);
        if (rc != AEC_OK) break;
        if (lin_out) {
            ok(cudaMemcpyAsync(err + off * out_stride, ctx->d_err[k], out_row * (size_t)nb, cudaMemcpyDeviceToHost, s));
            if (echo_est)
                ok(cudaMemcpyAsync(echo_est + off * out_stride, ctx->d_echo[k], out_row * (size_t)nb,
                                   cudaMemcpyDeviceToHost, s));
        } else {
            ok(cudaMemcpy2DAsync(err + off * out_stride, out_pitch, ctx->d_err[k], dpitch, out_row, (size_t)nb,
                                 cudaMemcpyDeviceToHost, s));
            if (echo_est)
                ok(cudaMemcpy2DAsync(echo_est + off * out_stride, out_pitch, ctx->d_echo[k], dpitch, out_row, (size_t)nb,
                                     cudaMemcpyDeviceToHost, s));
        }
        if (erle_db) {
            ok(cudaMemcpyAsync(ctx->h_erle[k], ctx->d_erle[k], (size_t)nb * sizeof(float), cudaMemcpyDeviceToHost, s));
            ctx->pending_dst[k] = erle_db;
        }
        if (shift_out) {
            ok(cudaMemcpyAsync(ctx->h_shift[k], ctx->d_shift[k], (size_t)nb * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
            ctx->pending_shift[k] = shift_out;
        }
        if (peak_out) {
            ok(cudaMemcpyAsync(ctx->h_peak[k], ctx->d_peak[k], (size_t)nb * sizeof(float), cudaMemcpyDeviceToHost, s));
            ctx->pending_peak[k] = peak_out;
        }
        if (erle_db || shift_out || peak_out) {
            ctx->pending_off[k] = off;
            ctx->pending_nb[k] = nb;
        }
    }
    if (e != cudaSuccess) {
        set_cuda_error(e, "aec_stage1_run_host: copy / launch");
        rc = AEC_ECUDA;
    }
    if (rc != AEC_OK) {
        host_ctx_quiesce(ctx);
        return rc;
    }
    if (ctx->deferred) return AEC_OK;               // the last slices land under the next call / aec_host_ctx_wait
    return aec_host_ctx_wait(ctx);
}
}  // namespace

extern "C" int aec_stage1_run_host(aec_host_ctx* ctx, const float* far, const float* mic, float* err, float* echo_est,
                                   float* erle_db, const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride,
                                   int64_t out_stride, const aec_cfg* cfg) {
    return run_host_impl<float>(ctx, far, mic, err, echo_est, erle_db, n_samples, B, L, in_stride, out_stride, cfg,
                                nullptr, nullptr, nullptr);
}

extern "C" int aec_stage1_run_host_ex(aec_host_ctx* ctx, const float* far, const float* mic, float* err,
                                      float* echo_est, float* erle_db, const int64_t* n_samples, int64_t B, int64_t L,
                                      int64_t in_stride, int64_t out_stride, const aec_cfg* cfg,
                                      const aec_delay_cfg* align, int32_t* shift_out, float* peak_out) {
    return run_host_impl<float>(ctx, far, mic, err, echo_est, erle_db, n_samples, B, L, in_stride, out_stride, cfg,
                                align, shift_out, peak_out);
}

extern "C" int aec_stage1_run_host_pcm16(aec_host_ctx* ctx, const int16_t* far, const int16_t* mic, float* err,
                                         float* echo_est, float* erle_db, const int64_t* n_samples, int64_t B,
                                         int64_t L, int64_t in_stride, int64_t out_stride, const aec_cfg* cfg) {
    return run_host_impl<int16_t>(ctx, far, mic, err, echo_est, erle_db, n_samples, B, L, in_stride, out_stride, cfg,
                                  nullptr, nullptr, nullptr);
}

extern "C" int aec_stage1_run_host_pcm16_ex(aec_host_ctx* ctx, const int16_t* far, const int16_t* mic, float* err,
                                            float* echo_est, float* erle_db, const int64_t* n_samples, int64_t B,
                                            int64_t L, int64_t in_stride, int64_t out_stride, const aec_cfg* cfg,
                                            const aec_delay_cfg* align, int32_t* shift_out, float* peak_out) {
    return run_host_impl<int16_t>(ctx, far, mic, err, echo_est, erle_db, n_samples, B, L, in_stride, out_stride, cfg,
                                  align, shift_out, peak_out);
}

extern "C" int aec_host_alloc_ex(void** ptr, int64_t bytes, int32_t flags) {
    if (!ptr || bytes <= 0) return AEC_EINVAL;
    unsigned f = cudaHostAllocDefault;
    if (flags & AEC_HOST_WRITE_COMBINED) f |= cudaHostAllocWriteCombined;
    if (flags & AEC_HOST_PORTABLE) f |= cudaHostAllocPortable;
    AEC_CUDA_CHECK(cudaHostAlloc(ptr, (size_t)bytes, f));
    return AEC_OK;
}

extern "C" int aec_host_alloc(void** ptr, int64_t bytes) { return aec_host_alloc_ex(ptr, bytes, 0); }

extern "C" int aec_host_free(void* ptr) {
    if (!ptr) return AEC_OK;
    AEC_CUDA_CHECK(cudaFreeHost(ptr));
    return AEC_OK;
}

extern "C" int aec_host_is_pinned(const void* ptr) {
    if (!ptr) return AEC_EINVAL;
    cudaPointerAttributes a{};
    const cudaError_t e = cudaPointerGetAttributes(&a, ptr);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return a.type == cudaMemoryTypeHost ? 1 : 0;
}

// ------------------------------------------------------------------------------------------
// FP32 peak probe
// ------------------------------------------------------------------------------------------
extern "C" int aec_bench_fp32_peak(int iters, double* tflops, void* cuda_stream) {
    if (iters <= 0 || !tflops) return AEC_EINVAL;
    cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
    int dev = 0, sms = 0;
    AEC_CUDA_CHECK(cudaGetDevice(&dev));
    AEC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    float* d = nullptr;
    AEC_CUDA_CHECK(cudaMalloc(&d, 256));
    cudaEvent_t a, b;
    AEC_CUDA_CHECK(cudaEventCreate(&a));
    AEC_CUDA_CHECK(cudaEventCreate(&b));
    const int blocks = sms * 8;
    ffma_peak_kernel<<<blocks, 256, 0, s>>>(d, iters / 4 + 1, 0.999f, 1e-3f);   // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        AEC_CUDA_CHECK(cudaEventRecord(a, s));
        ffma_peak_kernel<<<blocks, 256, 0, s>>>(d, iters, 0.999f, 1e-3f);
        AEC_CUDA_CHECK(cudaEventRecord(b, s));
        AEC_CUDA_CHECK(cudaEventSynchronize(b));
        float ms = 0.f;
        AEC_CUDA_CHECK(cudaEventElapsedTime(&ms, a, b));
        const double flops = 2.0 * 64.0 * (double)iters * 256.0 * (double)blocks;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    // packed probe: FFMA2 does 2 FMAs per lane per issue; report the larger of the two rates
    for (int rep = 0; rep < 3; ++rep) {
        AEC_CUDA_CHECK(cudaEventRecord(a, s));
        ffma2_peak_kernel<<<blocks, 256, 0, s>>>(d, iters, 0.999f, 1e-3f);
        AEC_CUDA_CHECK(cudaEventRecord(b, s));
        AEC_CUDA_CHECK(cudaEventSynchronize(b));
        float ms = 0.f;
        AEC_CUDA_CHECK(cudaEventElapsedTime(&ms, a, b));
        const double flops = 2.0 * 128.0 * (double)iters * 256.0 * (double)blocks;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (getenv("AEC_PEAK_VERBOSE")) fprintf(stderr, "[aec] FFMA2 probe %.2f TFLOP/s, FFMA probe best %.2f\n", tf, best);
        if (tf > best) best = tf;
    }
    count_launch(9);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(d);
    AEC_CUDA_CHECK(cudaGetLastError());
    *tflops = best;
    return AEC_OK;
}
