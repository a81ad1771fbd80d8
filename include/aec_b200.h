/* aec_b200 -- C ABI of the B200-native stage-1 linear acoustic echo canceller.
 *
 * Drop-in boundary for the data-parallel hot path named by BASELINE.json's north_star:
 * batched STFT framing/windowing -> partitioned frequency-domain adaptive filter (NLMS or
 * Kalman step size) -> iSTFT -> residual / feature output for the Stage-2 model of
 * SZU-Speech/Acoustic-Echo-Cancellation.
 *
 * The reference is plain Python calling torch.nn.functional; it has NO plugin / FFI
 * interface.  Each entry point below cites the reference seam it replaces (paths relative
 * to the reference root).  The reference contains no stage-1 filter at all: the FDAF entry
 * points replace the (missing) step between `librosa.load` and `h5py.create_dataset` in
 * Stage2_lhm/generate_h5files/train_wav2h5.py:20-42, and their arithmetic is the
 * builder-authored recurrence frozen in DESIGN.md (parity unpinned by the reference).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types.
 *   - `*_run` / `aec_stft` / `aec_istft` / `aec_features` take DEVICE pointers and launch on
 *     the caller's CUDA stream (`cuda_stream` is a cudaStream_t cast to void*, NULL = default
 *     stream) on the CURRENT device, without synchronising.  The caller owns every buffer.
 *   - `aec_stage1_run_host` takes HOST pointers, stages through an `aec_host_ctx`, and returns
 *     when the outputs are in host memory.
 *   - return 0 on success, a negative AEC_E* code otherwise; never throws, never falls
 *     back to a CPU implementation.
 */
#ifndef AEC_B200_H_
#define AEC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AEC_B200_VERSION 100 /* 0.1.0 */

enum {
    AEC_OK = 0,
    AEC_EINVAL = -1,      /* bad argument (null pointer, negative size, ...) */
    AEC_EUNSUPPORTED = -2, /* frame / partitions / algo combination not built */
    AEC_ECUDA = -3,       /* a CUDA runtime call failed; see aec_last_cuda_error() */
    AEC_ENODEVICE = -4,   /* no sm_100 device is current */
    AEC_ENOMEM = -5,
    AEC_EIO = -6          /* a file could not be opened / read (wav ingest) */
};

/* 0, 1: the STFT-domain recurrence (Hann-windowed STFT, one complex tap per bin and past hop) with an NLMS / Kalman step;
 * 2, 3: overlap-save partitioned-block FDAF with the alternated gradient constraint -- time-domain blocks of hop new
 *    samples, FFT length frame, exact linear convolution (no analysis window; ~25 dB more ERLE on the single-talk set,
 *    DESIGN.md section 2b).  2 = NLMS step on a smoothed input power (pb_lambda), 3 = the diagonal Kalman step of algo 1
 *    (kalman_*; holds ~15 dB through double talk where the NLMS step drops to 2).  Frame 512: partitions 1 / 2 / 4 / 8 / 16;
 *    frame 1024: partitions 4 / 8;
 *    outputs cover the whole blocks only ((n / hop) * hop samples, the same count as (frames - 1) * hop of algos 0 / 1);
 *    no fused feature epilogue.  All four recurrences are builder-authored: the reference has no stage-1 filter. */
enum { AEC_ALGO_NLMS = 0, AEC_ALGO_KALMAN = 1, AEC_ALGO_PBFDAF = 2, AEC_ALGO_PBFKF = 3 };

/* Parameter block of the stage-1 filter.  frame / hop follow the reference's
 * speech_conf (Stage2_lhm/scripts/configs.py:1-8: win_size 512, hop_size 256) and the window is
 * the periodic Hann hard-coded at Stage2_lhm/scripts/network/ERB.py:210.  hop = frame / 2. */
typedef struct aec_cfg {
    int32_t frame;          /* N: 512 (16 kHz) or 1024 (48 kHz) */
    int32_t partitions;     /* P: taps per bin, one per past hop */
    int32_t algo;           /* AEC_ALGO_NLMS | AEC_ALGO_KALMAN | AEC_ALGO_PBFDAF | AEC_ALGO_PBFKF */
    float mu;               /* NLMS step size                      (default 0.5) */
    float delta;            /* NLMS regulariser                    (default 1e-6 * frame) */
    float kalman_a;         /* Kalman transition factor A          (default 0.999) */
    float kalman_lambda;    /* observation-noise smoothing         (default 0.9) */
    float kalman_c0;        /* initial covariance                  (default 1) */
    float kalman_eps;       /* floor added to the innovation power (default 1e-10) */
    int32_t erle_skip_hops; /* hops excluded from the ERLE sums at the start of each utterance */
    int32_t variant;        /* 0 = library default; otherwise 1000*warps_per_utterance + register cap of one built kernel
                             * (DESIGN.md; e.g. 2168).  A warp count or cap that (frame, partitions, algo, echo) was not
                             * built with returns AEC_EUNSUPPORTED: the overlap-save kernels take 2 warps up to 4
                             * partitions and P / 2 above, the frame-1024 STFT-domain kernel 8; the frame-1024 overlap-save
                             * path and aec_stage1_run_features (build chosen from the batch size) take no variant. */
    int32_t stagger_ns;     /* tuning: start-up skew (ns per resident slot) between co-resident utterances; <= 0 = off (default) */
    float pb_lambda;        /* algo 2: smoothing of the per-bin input power (default 0.5) */
    int32_t reserved[3];
} aec_cfg;

int aec_version(void);
const char* aec_strerror(int code);
/* text of the last CUDA error seen by the calling thread ("" if none) */
const char* aec_last_cuda_error(void);

/* Optional: builds the constant tables (windows, twiddles) of the CURRENT device now instead of on the first
 * launch.  Call it once per device before capturing a CUDA graph around the `*_run` entries (the first-use
 * path allocates and copies, which a capture does not allow). */
int aec_init(void);

/* fills *cfg with the frozen defaults for the given frame length */
int aec_cfg_default(aec_cfg* cfg, int32_t frame);

/* Frame count of ConvSTFT.forward (Stage2_lhm/scripts/network/attention_ccrn.py:48-49):
 * (n + 2*(frame-hop) - frame) / hop + 1.   Replaces the off-by-one helper
 * countFrames (Stage2_lhm/scripts/utils/tools.py:30-32) for buffer sizing. */
int64_t aec_num_frames(int64_t n_samples, int32_t frame);
/* Output length of ConviSTFT.forward (attention_ccrn.py:99): (frames - 1) * hop. */
int64_t aec_out_samples(int64_t n_samples, int32_t frame);

/* Stage-1 canceller on DEVICE buffers.
 *   far, mic   [B][in_stride]  float32, the first n_samples[b] (or L) samples are used
 *   err        [B][out_stride] float32  time-domain error signal e = iSTFT(Y - Yhat); zero
 *              beyond aec_out_samples(n_b) up to L
 *   echo_est   nullable, like err: yhat = iSTFT(Yhat)
 *   erle_db    nullable [B]: 10 log10(sum mic^2 / sum err^2) over output hops >= erle_skip_hops
 *   n_samples  nullable DEVICE int64 [B] (ragged batch, values clamped to [0, L])
 * in_stride, out_stride >= L.  Fast paths need 16-byte aligned rows (stride % 4 == 0 and
 * aligned base); other layouts are handled by a slower in-kernel path, never on the CPU. */
int aec_stage1_run(const float* far, const float* mic, float* err, float* echo_est, float* erle_db,
                   const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride, int64_t out_stride,
                   const aec_cfg* cfg, void* cuda_stream);

/* Stage 1 WITH the Stage-2 feature front end fused into the kernel (SURVEY 8f rank 2; replaces, for the two-stage
 * pipeline, the three dense-conv STFTs + magnitude + ERB matmul + cat of Little_net.forward,
 * Stage2_lhm/scripts/network/ERB.py:262-290, applied to (stage-1 error, far end)):
 *   feat [B][aec_num_frames(L)][64] = cat[err_erb, |err_erb - far_erb|], err_erb = sqrt(re^2+im^2+1e-9)(STFT(err)) @ erb,
 *   far_erb likewise from the far end.  STFT(err) is the re-analysis of the SYNTHESISED error signal (parity with
 *   aec_features(err, far, erb, shift 0)), computed on chip one frame behind the synthesis; the far-end spectrum is the
 *   one the filter already has.  The batch-global shift of ERB.py:254-256 is NOT applied (it needs the whole error
 *   batch first): this is the `in_norm = False` form; use aec_batch_shift + aec_features_dev for the shifted one.
 *   erb: dense [257][32] float32 bank on the DEVICE (ERB.py:10-71; at most 512 coefficients inside the bands' non-zero
 *   ranges -- the reference's bank has 483).  Rows of a ragged utterance beyond its own frames hold the front end's
 *   response to silence.  Built for frame 512, partitions 4 (NLMS, Kalman), 2 and 1 (NLMS); no echo-estimate output. */
int aec_stage1_run_features(const float* far, const float* mic, float* err, float* erle_db, float* feat, const float* erb,
                            const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride, int64_t out_stride,
                            const aec_cfg* cfg, void* cuda_stream);

/* Streaming stage 1 (online use: a chunk of every live stream per call) for the frame-512 overlap-save filters
 * (algos 2 / 3, partitions 1 / 2 / 4 / 8 / 16, variant 0).  Each stream's filter state lives in caller-owned DEVICE
 * memory, row b at state + b * state_stride (16-byte aligned; state_stride >= aec_stage1_state_bytes, a multiple of 16).
 * Chunked calls give bit for bit the outputs of one aec_stage1_run over the whole signal.
 * State of one stream after T blocks (the quantities of oracle/aec_oracle.py:pbfdaf_ols in its rfft units, K = 257 bins,
 * little-endian, every array starting on a 16-byte boundary, the gaps zero):
 *   offset 0                  int64 blocks = T (+ 8 reserved bytes, zero)
 *   16                        float prev[256]: the far-end samples of block T - 1 (zeros at T = 0)
 *   1040                      complex64 W[P][K]: taps by partition p, after the update with E_{T-1}
 *   1040 + a16(8 P K)         complex64 X[P][K]: X[p] = rfft([x_{T-2-p}, x_{T-1-p}])
 *   1040 + 2 a16(8 P K)       algo 2: float Pw[K] (smoothed input power); algo 3: float Psi[K] (observation-noise power),
 *   ... + a16(4 K)            then (algo 3) float C[P][K] (covariances)                    a16(n) = n rounded up to 16
 * After aec_stage1_state_init: T = 0 and every other byte zero, except C = kalman_c0.
 * aec_stage1_state_bytes: bytes of one stream's state for cfg, or AEC_EUNSUPPORTED for algos 0 / 1, frame 1024, a
 *   variant or an unbuilt P (a negative AEC_E* code).
 * aec_stage1_state_init: (re)initialises rows b with reset_mask == NULL or reset_mask[b] != 0 (nullable DEVICE uint8 [B]);
 *   the other rows are left untouched.  One launch on the caller's stream.
 * aec_stage1_run_stream: aec_stage1_run's arguments for one chunk per stream.  Row b consumes n_b / 256 whole blocks
 *   (n_b = n_samples[b] or L): it writes that many blocks of err / echo_est, zeros beyond them up to L, and the caller
 *   keeps its remaining n_b mod 256 samples for the next call.  erle_db covers this call's blocks whose index in the
 *   stream is >= erle_skip_hops (0 dB without any).  A row without a whole block leaves its state untouched. */
int64_t aec_stage1_state_bytes(const aec_cfg* cfg);
int aec_stage1_state_init(void* state, int64_t B, int64_t state_stride, const uint8_t* reset_mask, const aec_cfg* cfg,
                          void* cuda_stream);
int aec_stage1_run_stream(const float* far, const float* mic, float* err, float* echo_est, float* erle_db,
                          const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride, int64_t out_stride,
                          const aec_cfg* cfg, void* state, int64_t state_stride, void* cuda_stream);

/* Host-buffer variant: the call a data-prep script makes with arrays that came out of
 * `librosa.load` (Stage2_lhm/generate_h5files/train_wav2h5.py:20-23) and whose results go to
 * `create_dataset` (train_wav2h5.py:39-42).  Copies are pipelined against the kernel in
 * slices of `ctx`'s capacity, four slices in flight (one stream each: H2D -> kernel -> D2H);
 * pinned host memory (aec_host_alloc) gives full PCIe rate.
 * n_samples is a HOST int64 [B] or NULL. */
typedef struct aec_host_ctx aec_host_ctx;
/* A context belongs to the device that was current when it was created (calls made with another device current
 * return AEC_EINVAL) and is NOT re-entrant: one `aec_stage1_run_host*` call at a time per context; use one
 * context per thread.  On any failure the call returns only after every copy it started has finished, so the
 * caller's buffers are never written after the return.
 * aec_host_ctx_create == aec_host_ctx_create_ex(.., slots = 0, flags = 0). */
int aec_host_ctx_create(aec_host_ctx** ctx, int64_t slice_utterances, int64_t max_samples);
/* slots: slices in flight, 1..8 (0 = default 4).  flags: AEC_HOST_CTX_NO_RAMP keeps the first slices full-size
 * (by default the first slices grow 16, 16, 32, 64, .. so that the first download starts early). */
enum { AEC_HOST_CTX_NO_RAMP = 1 };
int aec_host_ctx_create_ex(aec_host_ctx** ctx, int64_t slice_utterances, int64_t max_samples, int32_t slots,
                           int32_t flags);
int aec_host_ctx_destroy(aec_host_ctx* ctx);
/* Streaming use (batch after batch through one context): with deferred = 1 a run call returns as soon as its last
 * slice has been ENQUEUED, so that the tail of batch k (last kernel + download, ~1 ms) runs under the first uploads of
 * batch k+1.  The outputs (and erle_db) of a deferred call are complete after aec_host_ctx_wait(ctx) -- or once the
 * next call has returned, for slices whose slot it has reused; the caller keeps every buffer of a call alive and
 * unread until then, and gives consecutive calls DIFFERENT output buffers.  deferred = 0 (default): every call
 * returns with its outputs in host memory. */
int aec_host_ctx_set_deferred(aec_host_ctx* ctx, int32_t deferred);
int aec_host_ctx_wait(aec_host_ctx* ctx);
int aec_stage1_run_host(aec_host_ctx* ctx, const float* far, const float* mic, float* err, float* echo_est,
                        float* erle_db, const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride,
                        int64_t out_stride, const aec_cfg* cfg);
/* Same call for 16-bit PCM inputs (what the wav files hold before `librosa.load` turns them into
 * float32 = sample / 32768, train_wav2h5.py:20-23): the int16 -> float32 conversion runs on the GPU,
 * which halves the host-to-device bytes of a PCIe-bound pipeline.  Outputs stay float32. */
int aec_stage1_run_host_pcm16(aec_host_ctx* ctx, const int16_t* far, const int16_t* mic, float* err,
                              float* echo_est, float* erle_db, const int64_t* n_samples, int64_t B, int64_t L,
                              int64_t in_stride, int64_t out_stride, const aec_cfg* cfg);
/* Far-end bulk delay (GCC-PHAT over the whole utterance) and far-end alignment before stage 1.  The stage-1 filters
 * model echo paths that start at lag 0 and end before their tail (P * hop samples); a device's playback / capture
 * latency delays the echo by tens to hundreds of milliseconds, past that tail.  Per utterance, with D = max_delay:
 *   r[l] = PHAT-weighted cross-correlation of mic and far end at lag l = 0..D (|r| <= 1; DC and Nyquist dropped),
 *   delay = smallest l maximising |r[l]|, peak = |r[delay]|,
 *   shift = peak >= min_peak ? max(0, delay - margin) : 0,   far_aligned[n] = far[n - shift] (0 for n < shift).
 * Exact definition: DESIGN.md "Far-end delay estimation" and oracle/delay_oracle.py.  Whole samples; lags are
 * non-negative (the microphone never leads the far end); an empty utterance or a silent far end gives 0, 0, 0. */
typedef struct aec_delay_cfg {
    int32_t max_delay;    /* D: largest lag searched, a power of two in [256, 8192]   (default 8192: 512 ms at 16 kHz) */
    int32_t margin;       /* samples of echo path kept in front of the estimated delay, >= 0  (default 128) */
    float min_peak;       /* peak below which no shift is applied                       (default 0.1) */
    int32_t reserved[5];
} aec_delay_cfg;
int aec_delay_cfg_default(aec_delay_cfg* dcfg);
/* DEVICE buffers, caller's stream.  far, mic [B][in_stride] (first n_samples[b] or L samples; n_samples nullable
 * DEVICE int64 [B], clamped to [0, L]); outputs [B]: delay (nullable), shift, peak (nullable); corr nullable
 * [B][max_delay + 1] = r.  One CTA per utterance: a row's outputs are bit-identical alone or in any batch. */
int aec_delay_estimate(const float* far, const float* mic, const int64_t* n_samples, int64_t B, int64_t L,
                       int64_t in_stride, const aec_delay_cfg* dcfg, int32_t* delay, int32_t* shift, float* peak,
                       float* corr, void* cuda_stream);
/* far_out[b][n] = far[b][n - shift[b]] for shift[b] <= n < L, 0 below (a negative shift counts as 0).  DEVICE
 * buffers; far_out [B][out_stride] must not overlap far. */
int aec_delay_align(const float* far, float* far_out, const int32_t* shift, int64_t B, int64_t L, int64_t in_stride,
                    int64_t out_stride, void* cuda_stream);
/* aec_stage1_run_host[_pcm16] with the far end aligned first: each slice runs H2D, (PCM16 conversion), estimate,
 * align, stage 1 on the aligned far end, D2H.  align = NULL is exactly aec_stage1_run_host[_pcm16].  shift_out /
 * peak_out: nullable HOST [B], delivered like erle_db (after aec_host_ctx_wait in deferred mode); non-NULL only with
 * align.  The outputs are those of aec_delay_estimate + aec_delay_align + aec_stage1_run on the device buffers. */
int aec_stage1_run_host_ex(aec_host_ctx* ctx, const float* far, const float* mic, float* err, float* echo_est,
                           float* erle_db, const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride,
                           int64_t out_stride, const aec_cfg* cfg, const aec_delay_cfg* align, int32_t* shift_out,
                           float* peak_out);
int aec_stage1_run_host_pcm16_ex(aec_host_ctx* ctx, const int16_t* far, const int16_t* mic, float* err,
                                 float* echo_est, float* erle_db, const int64_t* n_samples, int64_t B, int64_t L,
                                 int64_t in_stride, int64_t out_stride, const aec_cfg* cfg, const aec_delay_cfg* align,
                                 int32_t* shift_out, float* peak_out);
/* page-locked host memory helpers (cudaHostAlloc / cudaFreeHost).  Pageable buffers work with the host entries
 * but every copy is then staged by the driver and serialises the slices -- allocate the arrays that
 * `librosa.load` results are gathered into with these.  AEC_HOST_WRITE_COMBINED: for buffers the CPU only
 * writes (inputs); AEC_HOST_PORTABLE: usable from every CUDA context of the process. */
enum { AEC_HOST_WRITE_COMBINED = 1, AEC_HOST_PORTABLE = 2 };
int aec_host_alloc(void** ptr, int64_t bytes);
int aec_host_alloc_ex(void** ptr, int64_t bytes, int32_t flags);
int aec_host_free(void* ptr);
/* 1 if ptr lies in page-locked host memory known to CUDA, 0 if not (pageable / unknown) */
int aec_host_is_pinned(const void* ptr);

/* Batched wav ingest (host code): what replaces the four serial `librosa.load(path, sr=args.sr)` calls per
 * utterance of the generators (Stage2_lhm/generate_h5files/train_wav2h5.py:20-23, test_wav2h5.py:29-32,
 * val_wav2h5.py:33-36) for the format those corpora are in -- 16-bit PCM, mono, already at the target rate.
 * aec_wav_probe parses the RIFF chunk list (no samples read).  aec_wav_read_pcm16_batch reads n files with
 * `threads` threads into rows of an int16 batch buffer (row i at dst + i * row_stride; the first
 * min(frames, row_samples) samples, zero-filled up to row_samples), storing the true frame counts in frames[]
 * (nullable).  Files that are not 16-bit mono PCM at expect_rate (expect_rate <= 0: any rate) make the call return
 * AEC_EUNSUPPORTED -- the caller decodes that batch with a general loader; the samples are never touched here
 * (int16 in, int16 out; `x / 32768`, librosa's scaling, is applied on the GPU by aec_stage1_run_host_pcm16). */
typedef struct aec_wav_info {
    int32_t rate, channels, bits;
    int32_t format;      /* 1 = integer PCM, 3 = IEEE float (WAVE_FORMAT_EXTENSIBLE resolved to its sub-format) */
    int64_t frames;      /* samples per channel in the data chunk */
    int64_t data_offset; /* byte offset of the first sample */
} aec_wav_info;
int aec_wav_probe(const char* path, aec_wav_info* info);
int aec_wav_probe_batch(const char* const* paths, int64_t n, aec_wav_info* infos, int32_t threads);
int aec_wav_read_pcm16_batch(const char* const* paths, int64_t n, int16_t* dst, int64_t row_stride,
                             int64_t row_samples, int64_t* frames, int32_t expect_rate, int32_t threads);

/* Batched writer of the per-utterance training files (host code): replaces, for a whole batch, the
 * `h5py.File(tr_filename, 'w')` / `create_dataset(key, data=x.astype(np.float32), shape=x.shape, chunks=True)` x 4 /
 * `close()` block of Stage2_lhm/generate_h5files/train_wav2h5.py:35-44.  File f (paths[f]) becomes an HDF5 file whose
 * root group holds n_datasets (<= 8) one-dimensional float32 datasets names[d] of lens[f * n_datasets + d] samples
 * taken from data[f * n_datasets + d]; formats[d] (nullable = all 0) says what the source is: 0 = float32, stored as it
 * is; 1 = 16-bit PCM, stored as float32 = sample / 32768 (librosa's scaling, train_wav2h5.py:20-23).  `threads` C++
 * threads share the files.  Format: superblock v0, symbol-table root group, contiguous storage -- byte-identical to
 * acoustic_echo_cancellation_b200/h5lite.py (which documents it and reads it back); every libhdf5 / h5py opens it.
 * Returns AEC_EINVAL for bad arguments (duplicate / empty / '/'-containing names, > 8 datasets), AEC_EIO when a file
 * cannot be created or written (the other files of the batch are still attempted). */
int aec_ex_write_batch(const char* const* paths, int64_t n_files, int32_t n_datasets, const char* const* names,
                       const void* const* data, const int64_t* lens, const int32_t* formats, int32_t threads);

/* STFT analysis on DEVICE buffers: replaces ConvSTFT(frame, frame/2, frame, 'hann', 'complex')
 * .forward (Stage2_lhm/scripts/network/attention_ccrn.py:45-52).
 *   x [B][in_stride] -> spec [B][2K][T], K = frame/2+1, T = aec_num_frames(L): channels
 *   0..K-1 real, K..2K-1 imaginary (the reference's real-over-imag layout). */
int aec_stft(const float* x, float* spec, int64_t B, int64_t L, int64_t in_stride, int32_t frame,
             void* cuda_stream);
/* iSTFT synthesis: replaces ConviSTFT(...).forward (attention_ccrn.py:82-101).
 *   spec [B][2K][T] -> y [B][out_stride], (T-1)*hop samples written per row. */
int aec_istft(const float* spec, float* y, int64_t B, int64_t T, int64_t out_stride, int32_t frame,
              void* cuda_stream);

/* Stage-2 feature front end: replaces Little_net.forward lines
 * Stage2_lhm/scripts/network/ERB.py:262-290 (complex STFT of mic and ref, magnitude
 * sqrt(re^2+im^2+1e-9), @ erb, cat[mic_erb, |mic_erb - ref_erb|]).
 *   mic, ref [B][in_stride]; erb [K][bands] row-major float32 (ERB.py:10-71);
 *   shift_mic / shift_ref: the batch-global scalar mean/std subtracted at ERB.py:254-255
 *   (computed by the caller; pass 0 to skip);  feat [B][T][2*bands]. */
int aec_features(const float* mic, const float* ref, const float* erb, float* feat, int64_t B, int64_t L,
                 int64_t in_stride, int32_t frame, int32_t bands, float shift_mic, float shift_ref,
                 void* cuda_stream);

/* The batch-global scalar of ERB.py:254-256, mean(x) / std(x) over ALL B*L samples (unbiased std, torch.std),
 * computed on the device and left there: shift_dev[0] feeds aec_features_dev / aec_stage2_synth_dev without a host
 * round trip.  `workspace`: caller-owned device memory of at least aec_batch_shift_workspace_bytes() bytes (8-byte
 * aligned); partial sums are accumulated in double in a fixed order (deterministic). */
int64_t aec_batch_shift_workspace_bytes(void);
int aec_batch_shift(const float* x, int64_t B, int64_t L, int64_t stride, float* shift_dev, void* workspace,
                    int64_t workspace_bytes, void* cuda_stream);
/* aec_features with the two shifts read from DEVICE memory (NULL = 0) */
int aec_features_dev(const float* mic, const float* ref, const float* erb, float* feat, int64_t B, int64_t L,
                     int64_t in_stride, int32_t frame, int32_t bands, const float* shift_mic_dev,
                     const float* shift_ref_dev, void* cuda_stream);

/* Stage-2 residual-echo suppressor inference (the consumer of the stage-1 output), for the
 * reference's live model Little_net (Stage2_lhm/scripts/network/ERB.py:203-334, 32 ERB bands):
 *   feat = aec_features(stage1_error or mic, far, erb)                          ERB.py:254-290
 *   aec_stage2_mask : GRU(64->32) + Linear(64->32)+ReLU + Linear(32->32)+sigmoid, est_erb = mask*mic_erb
 *                     feat [B][T][64] -> est_erb [B][T][32]                       ERB.py:293-304
 *   aec_stage2_synth: out = iSTFT((est_erb @ erb^T) * STFT(mic - shift_mic)) + 1e-9 -> out [B][out_stride]
 *                                                                                 ERB.py:306-316
 * Weights are the module's state_dict tensors (row-major, PyTorch layouts, gate order r,z,n), on the device. */
typedef struct aec_stage2_weights {
    const float* gru_w_ih; /* gru1.weight_ih_l0 [96][64] */
    const float* gru_w_hh; /* gru1.weight_hh_l0 [96][32] */
    const float* gru_b_ih; /* gru1.bias_ih_l0   [96]     */
    const float* gru_b_hh; /* gru1.bias_hh_l0   [96]     */
    const float* lin1_w;   /* linear1.weight    [32][64] */
    const float* lin1_b;   /* linear1.bias      [32]     */
    const float* lin2_w;   /* linear2.weight    [32][32] */
    const float* lin2_b;   /* linear2.bias      [32]     */
} aec_stage2_weights;
int aec_stage2_mask(const float* feat, const aec_stage2_weights* w, float* est_erb, int64_t B, int64_t T,
                    int32_t bands, void* cuda_stream);
int aec_stage2_synth(const float* mic, const float* est_erb, const float* erb, float* out, int64_t B, int64_t L,
                     int64_t in_stride, int64_t out_stride, int32_t frame, int32_t bands, float shift_mic,
                     void* cuda_stream);

/* aec_stage2_synth with the shift read from DEVICE memory (NULL = 0) */
int aec_stage2_synth_dev(const float* mic, const float* est_erb, const float* erb, float* out, int64_t B, int64_t L,
                         int64_t in_stride, int64_t out_stride, int32_t frame, int32_t bands, const float* shift_mic_dev,
                         void* cuda_stream);

/* Streaming Stage 2 (online use: the new hops of every live stream per call): features, GRU, mask, gain, inverse STFT
 * and overlap-add of Little_net in one launch, without the batch-global input shift (in_norm off, ERB.py:254-256 needs
 * the whole signal).  Frame 512, hop 256, 32 bands.  Each stream's state lives in caller-owned DEVICE memory, row b at
 * state + b * state_stride (16-byte aligned; state_stride >= aec_stage2_state_bytes(), a multiple of 16).
 * State of one stream after T frames (little-endian, 3216 bytes):
 *   offset 0      int64 frames = T (+ 8 reserved bytes, zero)
 *   16            float h[32]: the GRU state after frame T - 1
 *   144           float mic_prev[256]: hop T - 1 of the mic input (zeros at T = 0)
 *   1168          float ref_prev[256]: hop T - 1 of the ref input
 *   2192          float ola[256]: the windowed second half of frame T - 1 (without the + 1e-9)
 * After aec_stage2_state_init every byte is zero.
 * aec_stage2_state_init: (re)initialises rows b with reset_mask == NULL or reset_mask[b] != 0 (nullable DEVICE uint8
 *   [B]); the other rows and the bytes past aec_stage2_state_bytes() are left untouched.  One launch.
 * aec_stage2_run_stream: mic (the stage-1 error or the microphone), ref (the far end) [B][in_stride]; row b consumes
 *   n_b / 256 whole hops (n_b = n_samples[b] or L; n_samples a nullable DEVICE int64 [B]) and computes frames
 *   T0 .. T0+n-1; it writes output blocks T0-1 .. T0+n-2 to out [B][out_stride] from column 0 (block -1 is not part of
 *   the signal: a stream's first call with hops writes one block fewer) and zeros after them up to L.  The caller keeps
 *   the remaining n_b mod 256 samples for the next call.  A row without a whole hop leaves its state untouched.  Chunked
 *   calls give bit for bit the output of one call over the whole stream; fed one more hop (the last samples zero-padded),
 *   the concatenated output is the (T-1) * 256 samples of the whole-utterance path with in_norm off (to rounding).
 *   bands != 32: AEC_EUNSUPPORTED; a null or misaligned state or weight pointer, a bad stride or B < 0: AEC_EINVAL.
 *   Every refusal launches nothing. */
int64_t aec_stage2_state_bytes(void);
int aec_stage2_state_init(void* state, int64_t B, int64_t state_stride, const uint8_t* reset_mask, void* cuda_stream);
int aec_stage2_run_stream(const float* mic, const float* ref, const float* erb, const aec_stage2_weights* w, float* out,
                          const int64_t* n_samples, int64_t B, int64_t L, int64_t in_stride, int64_t out_stride,
                          void* state, int64_t state_stride, int32_t bands, void* cuda_stream);

/* Measurement helpers used by bench.py (not part of the reference-facing surface).
 * aec_bench_fp32_peak: dependent-free FFMA loop on every SM; returns achieved FP32 TFLOP/s. */
int aec_bench_fp32_peak(int iters, double* tflops, void* cuda_stream);
/* number of kernels this library has launched on the calling thread since the last reset */
int64_t aec_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* AEC_B200_H_ */
