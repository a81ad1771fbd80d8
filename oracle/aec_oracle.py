"""CPU oracle for the stage-1 linear echo canceller path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product path
(``acoustic_echo_cancellation_b200``) never imports it and has no CPU fallback.

Parity status (see DESIGN.md, SURVEY.md section 8c)
---------------------------------------------------
* ``stft`` / ``istft`` / ``count_frames_reference`` / ``erb_filterbank`` /
  ``stage2_features`` / ``stage2_little_net`` restate code that EXISTS in the reference and are pinned
  by golden vectors produced by importing the reference modules
  (``tests/golden/make_golden.py``):
    - STFT analysis      Stage2_lhm/scripts/network/attention_ccrn.py:8-25,45-52
    - iSTFT synthesis    Stage2_lhm/scripts/network/attention_ccrn.py:20-23,82-101
    - frame constants    Stage2_lhm/scripts/configs.py:1-8, network/ERB.py:210,223-224
    - countFrames        Stage2_lhm/scripts/utils/tools.py:30-32
    - ERB filterbank     Stage2_lhm/scripts/network/ERB.py:10-71
    - feature front end  Stage2_lhm/scripts/network/ERB.py:254-290
* ``fdaf_nlms`` / ``fdaf_kalman`` / ``erle_db``: **PARITY UNPINNED**.  The reference
  repository contains no stage-1 adaptive filter at all (no FDAF/NLMS/Kalman/ERLE
  code).  The recurrences below are BUILDER-AUTHORED, frozen in DESIGN.md
  ("Frozen recurrence"), and must never be described as "the reference
  implementation".  They are instances of published filters (DESIGN.md section 2, "Lineage":
  Avargel & Cohen 2007 for the cross-band-free STFT-domain model, Enzner & Vary 2006 / Kuech et al.
  2014 for the diagonal frequency-domain Kalman step, Soo & Pang 1990 with the alternated constraint
  of Joho & Moschytz 2000 for ``pbfdaf_ols``), written out here with fixed constants; no code of
  theirs was available to check against.

All functions are plain numpy.  ``dtype=np.float64`` is the arbiter for parity
tests (the CUDA path computes in float32; tolerance 1e-4 max-abs on the
time-domain error signal, 0.05 dB on ERLE).  ``dtype=np.float32`` runs the same
operation order in single precision and is used to measure drift.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

# --------------------------------------------------------------------------------------
# constants the reference fixes (Stage2_lhm/scripts/configs.py:1-8, network/ERB.py:210)
# --------------------------------------------------------------------------------------
SAMPLE_RATE = 16000
WIN_SIZE = 512
HOP_SIZE = 256

ALGO_NLMS = 0
ALGO_KALMAN = 1
ALGO_PBFDAF = 2       # overlap-save constrained PBFDAF, NLMS step (round 2; time-domain blocks, no STFT framing)
ALGO_PBFKF = 3        # the same filter with the diagonal Kalman step of algo 1


@dataclass(frozen=True)
class AecConfig:
    """Builder-authored parameter block of the stage-1 filter (frozen defaults)."""

    frame: int = WIN_SIZE          # N, also the FFT length
    partitions: int = 4            # P, taps per bin (one per past hop)
    algo: int = ALGO_NLMS
    mu: float = 0.5                # NLMS step size
    delta: float = 1e-6 * WIN_SIZE  # NLMS regulariser (added to the sliding power)
    kalman_a: float = 0.999        # Kalman transition factor A
    kalman_lambda: float = 0.9     # smoothing of the observation-noise estimate
    kalman_c0: float = 1.0         # initial state covariance
    kalman_eps: float = 1e-10      # keeps D > 0 on digital silence
    pb_lambda: float = 0.5         # PBFDAF: smoothing of the per-bin input power

    @property
    def hop(self) -> int:
        return self.frame // 2

    @property
    def bins(self) -> int:
        return self.frame // 2 + 1


# --------------------------------------------------------------------------------------
# STFT / iSTFT  (pinned by the reference)
# --------------------------------------------------------------------------------------
def hann_periodic(n: int, dtype=np.float64) -> np.ndarray:
    """``scipy.signal.get_window('hann', n, fftbins=True)`` in closed form
    (attention_ccrn.py:12).  The reference builds it in float64 and casts the
    window-times-basis product to float32 (attention_ccrn.py:25)."""
    k = np.arange(n, dtype=np.float64)
    return (0.5 - 0.5 * np.cos(2.0 * np.pi * k / n)).astype(dtype)


def n_frames(n_samples: int, frame: int = WIN_SIZE, hop: int = HOP_SIZE) -> int:
    """Frame count of ``ConvSTFT.forward`` (attention_ccrn.py:48-49): pad
    ``frame-hop`` zeros on both sides, stride-``hop`` valid convolution."""
    padded = n_samples + 2 * (frame - hop)
    if padded < frame:
        return 0
    return (padded - frame) // hop + 1


def count_frames_reference(n_samples: int, win_size: int, hop_size: int) -> int:
    """The reference's loss-weighting helper (utils/tools.py:30-32).  It is one
    short of the true STFT frame count for 10 s inputs (625 vs 626) and must not
    be used to size buffers; restated only so the discrepancy is tested."""
    n_overlap = win_size // hop_size
    return int((n_samples - n_overlap) // hop_size + 1)


def _frames(x: np.ndarray, frame: int, hop: int) -> np.ndarray:
    """[B, L] -> [B, T, frame] view of the zero-padded signal."""
    pad = frame - hop
    xp = np.pad(x, ((0, 0), (pad, pad)))
    t = (xp.shape[1] - frame) // hop + 1
    idx = np.arange(frame)[None, :] + hop * np.arange(t)[:, None]
    return xp[:, idx]


def stft_complex(x: np.ndarray, frame: int = WIN_SIZE, hop: int = HOP_SIZE,
                 dtype=np.float64) -> np.ndarray:
    """Complex spectra [B, T, K].  Sign convention of ``np.fft.rfft``
    (imag = -sum x sin), as the reference's conv kernel (attention_ccrn.py:15-18)."""
    x = np.atleast_2d(np.asarray(x, dtype=dtype))
    w = hann_periodic(frame, dtype)
    fr = _frames(x, frame, hop) * w
    spec = np.fft.rfft(fr, axis=-1)
    return spec.astype(np.complex128 if dtype == np.float64 else np.complex64)


def stft(x: np.ndarray, frame: int = WIN_SIZE, hop: int = HOP_SIZE,
         dtype=np.float64) -> np.ndarray:
    """``ConvSTFT(frame, hop, frame, 'hann', 'complex')(x)`` layout:
    [B, 2K, T], channels 0..K-1 real, K..2K-1 imaginary (attention_ccrn.py:49-52)."""
    s = stft_complex(x, frame, hop, dtype)
    return np.concatenate([s.real, s.imag], axis=-1).transpose(0, 2, 1).astype(dtype)


def istft_complex(spec: np.ndarray, frame: int = WIN_SIZE, hop: int = HOP_SIZE,
                  dtype=np.float64) -> np.ndarray:
    """Inverse of :func:`stft_complex` with the reference's normalisation
    (attention_ccrn.py:92-99): irfft * window, overlap-add, divide by the
    overlap-added squared window + 1e-8, trim ``frame-hop`` samples at both ends.
    [B, T, K] -> [B, (T-1)*hop].  Imaginary parts of the DC / Nyquist bins do not
    contribute (their rows of the pinv synthesis kernel are zero)."""
    spec = np.asarray(spec)
    b, t, k = spec.shape
    assert k == frame // 2 + 1
    w = hann_periodic(frame, dtype)
    fr = np.fft.irfft(spec, n=frame, axis=-1).astype(dtype) * w
    total = (t - 1) * hop + frame
    out = np.zeros((b, total), dtype=dtype)
    coff = np.zeros(total, dtype=dtype)
    w2 = w * w
    for i in range(t):
        out[:, i * hop:i * hop + frame] += fr[:, i]
        coff[i * hop:i * hop + frame] += w2
    out = out / (coff + dtype(1e-8))
    pad = frame - hop
    return out[:, pad:total - pad]


def istft(spec_ri: np.ndarray, frame: int = WIN_SIZE, hop: int = HOP_SIZE,
          dtype=np.float64) -> np.ndarray:
    """``ConviSTFT(...)(spec)`` for the [B, 2K, T] real-over-imag layout; returns
    [B, 1, (T-1)*hop] like the reference (attention_ccrn.py:82-101)."""
    spec_ri = np.asarray(spec_ri, dtype=dtype)
    k = frame // 2 + 1
    s = spec_ri[:, :k, :] + 1j * spec_ri[:, k:, :]
    y = istft_complex(s.transpose(0, 2, 1), frame, hop, dtype)
    return y[:, None, :]


# --------------------------------------------------------------------------------------
# FDAF recurrences  (BUILDER-AUTHORED -- parity unpinned by the reference)
# --------------------------------------------------------------------------------------
def _cdtype(dtype):
    return np.complex128 if dtype == np.float64 else np.complex64


def fdaf_nlms(X: np.ndarray, Y: np.ndarray, cfg: AecConfig, dtype=np.float64):
    """STFT-domain partitioned NLMS.  X, Y: [T, K] complex spectra of far-end and
    microphone.  Returns (E, Yhat), both [T, K].

    per frame t, per bin k (X[t<0] = 0, W_p = 0 initially):
        Yhat = sum_p W_p * X[t-p]
        E    = Y - Yhat
        Pw   = sum_p |X[t-p]|^2
        W_p += (mu / (Pw + delta)) * conj(X[t-p]) * E
    """
    cd = _cdtype(dtype)
    X = np.asarray(X, dtype=cd)
    Y = np.asarray(Y, dtype=cd)
    T, K = X.shape
    P = cfg.partitions
    W = np.zeros((P, K), dtype=cd)
    hist = np.zeros((P, K), dtype=cd)          # hist[p] = X[t-p]
    E = np.zeros((T, K), dtype=cd)
    Yh = np.zeros((T, K), dtype=cd)
    mu = dtype(cfg.mu)
    delta = dtype(cfg.delta)
    for t in range(T):
        hist[1:] = hist[:-1].copy()
        hist[0] = X[t]
        yh = (W * hist).sum(axis=0)
        e = Y[t] - yh
        pw = (hist.real ** 2 + hist.imag ** 2).sum(axis=0).astype(dtype)
        g = (mu / (pw + delta)).astype(dtype)
        W = W + np.conj(hist) * (g * e)[None, :]
        E[t] = e
        Yh[t] = yh
    return E, Yh


def fdaf_kalman(X: np.ndarray, Y: np.ndarray, cfg: AecConfig, dtype=np.float64):
    """Diagonal frequency-domain Kalman filter, partitioned over P past hops.
    Returns (E, Yhat).

    per frame t, per bin k (W_p = 0, C_p = c0, Psi = 0 initially):
        Yhat = sum_p W_p * X[t-p]
        E    = Y - Yhat
        Psi  = lambda * Psi + (1 - lambda) * |E|^2
        D    = sum_p C_p * |X[t-p]|^2 + Psi + eps
        G_p  = C_p * conj(X[t-p]) / D
        W_p  = A * (W_p + G_p * E)
        C_p  = A^2 * (1 - C_p |X[t-p]|^2 / D) * C_p + (1 - A^2) * |W_p|^2   (new W_p)
    """
    cd = _cdtype(dtype)
    X = np.asarray(X, dtype=cd)
    Y = np.asarray(Y, dtype=cd)
    T, K = X.shape
    P = cfg.partitions
    W = np.zeros((P, K), dtype=cd)
    C = np.full((P, K), cfg.kalman_c0, dtype=dtype)
    psi = np.zeros(K, dtype=dtype)
    hist = np.zeros((P, K), dtype=cd)
    E = np.zeros((T, K), dtype=cd)
    Yh = np.zeros((T, K), dtype=cd)
    A = dtype(cfg.kalman_a)
    A2 = dtype(cfg.kalman_a * cfg.kalman_a)
    Q = dtype(1.0 - cfg.kalman_a * cfg.kalman_a)
    lam = dtype(cfg.kalman_lambda)
    oml = dtype(1.0 - cfg.kalman_lambda)
    eps = dtype(cfg.kalman_eps)
    one = dtype(1.0)
    for t in range(T):
        hist[1:] = hist[:-1].copy()
        hist[0] = X[t]
        yh = (W * hist).sum(axis=0)
        e = Y[t] - yh
        e2 = (e.real ** 2 + e.imag ** 2).astype(dtype)
        psi = lam * psi + oml * e2
        x2 = (hist.real ** 2 + hist.imag ** 2).astype(dtype)
        cx2 = C * x2
        D = cx2.sum(axis=0) + psi + eps
        rD = one / D
        G = (C * rD[None, :]) * np.conj(hist)
        W = A * (W + G * e[None, :])
        w2 = (W.real ** 2 + W.imag ** 2).astype(dtype)
        C = A2 * (one - cx2 * rD[None, :]) * C + Q * w2
        E[t] = e
        Yh[t] = yh
    return E, Yh


def pbfdaf_ols(far: np.ndarray, mic: np.ndarray, cfg: AecConfig, dtype=np.float64):
    """Overlap-save partitioned-block FDAF with the alternated gradient constraint (algo = 2: NLMS step, algo = 3:
    the diagonal Kalman step of ``fdaf_kalman``; BUILDER-AUTHORED, parity unpinned like the other recurrences).  One
    utterance, time-domain in, time-domain out: blocks of H = frame / 2 new samples, FFT length 2H = frame,
    P partitions -> the same P*H-sample tail as algos 0 / 1, but as an exact linear convolution (no analysis window,
    no cross-band leakage).

    per block t, c = t mod P (W_p = 0, Xh_p = 0, Pw = 0 / C_p = c0, Psi = 0, x_{-1} = 0 initially):
        Xh_p   = Xh_{p-1} (shift);  Xh_0 = rfft([x_{t-1}, x_t])
        y      = irfft(sum_p W_p Xh_p)[H:]           e = d_t - y            E = rfft([0_H, e])
        W_c    = rfft(g),  g = irfft(W_c),  g[H:] = 0      (one partition constrained per block, AS IT ENTERED the
                                                            block: the constraint does not wait for E, so a kernel
                                                            runs its two transforms beside the two of the error path)
      algo 2:
        Pw     = lam Pw + (1 - lam) sum_p |Xh_p|^2
        W_p   += mu / (Pw + delta) * conj(Xh_p) * E
      algo 3:
        Psi    = lambda Psi + (1 - lambda) |E|^2
        D      = sum_p C_p |Xh_p|^2 + Psi + eps          G_p = C_p conj(Xh_p) / D
        W_p    = A (W_p + G_p E)
        C_p    = A^2 (1 - C_p |Xh_p|^2 / D) C_p + (1 - A^2) |W_p|^2        (new W_p)
    Returns (err, yhat), each (n // H) * H samples."""
    cd = _cdtype(dtype)
    far = np.asarray(far, dtype=dtype)
    mic = np.asarray(mic, dtype=dtype)
    N, H, P = cfg.frame, cfg.hop, cfg.partitions
    K = H + 1
    kalman = cfg.algo == ALGO_PBFKF
    nblk = min(len(far), len(mic)) // H
    W = np.zeros((P, K), dtype=cd)
    Xh = np.zeros((P, K), dtype=cd)
    pw = np.zeros(K, dtype=dtype)
    C = np.full((P, K), cfg.kalman_c0, dtype=dtype)
    psi = np.zeros(K, dtype=dtype)
    prev = np.zeros(H, dtype=dtype)
    mu, delta, lam = dtype(cfg.mu), dtype(cfg.delta), dtype(cfg.pb_lambda)
    A = dtype(cfg.kalman_a)
    A2 = dtype(cfg.kalman_a * cfg.kalman_a)
    Q = dtype(1.0 - cfg.kalman_a * cfg.kalman_a)
    klam = dtype(cfg.kalman_lambda)
    koml = dtype(1.0 - cfg.kalman_lambda)
    eps = dtype(cfg.kalman_eps)
    one = dtype(1.0)
    err = np.zeros(nblk * H, dtype=dtype)
    yh = np.zeros(nblk * H, dtype=dtype)
    zeros = np.zeros(H, dtype=dtype)
    for t in range(nblk):
        cur = far[t * H:(t + 1) * H]
        Xh[1:] = Xh[:-1].copy()
        Xh[0] = np.fft.rfft(np.concatenate([prev, cur])).astype(cd)
        prev = cur
        y = np.fft.irfft((W * Xh).sum(axis=0), n=N)[H:].astype(dtype)
        e = mic[t * H:(t + 1) * H] - y
        err[t * H:(t + 1) * H] = e
        yh[t * H:(t + 1) * H] = y
        E = np.fft.rfft(np.concatenate([zeros, e])).astype(cd)
        c = t % P
        gt = np.fft.irfft(W[c], n=N).astype(dtype)
        gt[H:] = 0
        W[c] = np.fft.rfft(gt).astype(cd)
        x2 = (Xh.real ** 2 + Xh.imag ** 2).astype(dtype)
        if not kalman:
            pw = lam * pw + (one - lam) * x2.sum(axis=0)
            g = (mu / (pw + delta)).astype(dtype)
            W = W + np.conj(Xh) * (g * E)[None, :]
        else:
            psi = klam * psi + koml * (E.real ** 2 + E.imag ** 2).astype(dtype)
            cx2 = C * x2
            rD = one / (cx2.sum(axis=0) + psi + eps)
            G = (C * rD[None, :]) * np.conj(Xh)
            W = A * (W + G * E[None, :])
            w2 = (W.real ** 2 + W.imag ** 2).astype(dtype)
            C = A2 * (one - cx2 * rD[None, :]) * C + Q * w2
    return err, yh


def erle_db(num_sig: np.ndarray, den_sig: np.ndarray, skip: int = 0) -> np.ndarray:
    """ERLE in dB per utterance over samples [skip:]: 10 log10(sum num^2 / sum den^2).
    Single-talk: num = mic, den = error.  Double-talk: num = echo, den = echo - echo_est.
    Energies are floored at 1e-20 so digital silence is finite."""
    num = np.atleast_2d(np.asarray(num_sig, dtype=np.float64))[:, skip:]
    den = np.atleast_2d(np.asarray(den_sig, dtype=np.float64))[:, skip:]
    pn = np.maximum((num * num).sum(axis=1), 1e-20)
    pd = np.maximum((den * den).sum(axis=1), 1e-20)
    return 10.0 * np.log10(pn / pd)


def stage1(far: np.ndarray, mic: np.ndarray, cfg: AecConfig = AecConfig(),
           dtype=np.float64, n_samples=None, erle_skip: int = 0):
    """Whole stage-1 path for a batch: STFT -> FDAF -> iSTFT.

    far, mic: [B, L].  ``n_samples`` (optional, [B]) gives ragged lengths: each
    utterance is processed as if it were alone with that length and its outputs
    are zero beyond ``(T_b - 1) * hop``.
    Returns dict(err [B, L_out], echo [B, L_out], erle_db [B]) with
    L_out = (T_max - 1) * hop.
    """
    far = np.atleast_2d(np.asarray(far, dtype=dtype))
    mic = np.atleast_2d(np.asarray(mic, dtype=dtype))
    B, L = far.shape
    N, H = cfg.frame, cfg.hop
    if n_samples is None:
        n_samples = [L] * B
    l_out = max((n_frames(int(n), N, H) - 1) * H for n in n_samples)
    l_out = max(l_out, 0)
    err = np.zeros((B, l_out), dtype=dtype)
    echo = np.zeros((B, l_out), dtype=dtype)
    erle = np.zeros(B, dtype=np.float64)
    run = fdaf_nlms if cfg.algo == ALGO_NLMS else fdaf_kalman
    for b in range(B):
        n = int(n_samples[b])
        if cfg.algo in (ALGO_PBFDAF, ALGO_PBFKF):   # time-domain blocks: (n // H) * H output samples, like (T - 1) * H
            e, yh = pbfdaf_ols(far[b, :n], mic[b, :n], cfg, dtype)
            err[b, :e.shape[0]] = e
            echo[b, :yh.shape[0]] = yh
            m = e.shape[0]
            erle[b] = erle_db(mic[b, :m], e, erle_skip)[0] if m > erle_skip else 0.0
            continue
        X = stft_complex(far[b:b + 1, :n], N, H, dtype)[0]
        Y = stft_complex(mic[b:b + 1, :n], N, H, dtype)[0]
        E, Yh = run(X, Y, cfg, dtype)
        e = istft_complex(E[None], N, H, dtype)[0]
        yh = istft_complex(Yh[None], N, H, dtype)[0]
        err[b, :e.shape[0]] = e
        echo[b, :yh.shape[0]] = yh
        m = e.shape[0]
        erle[b] = erle_db(mic[b, :m], e, erle_skip)[0] if m > erle_skip else 0.0
    return {"err": err, "echo": echo, "erle_db": erle}


# --------------------------------------------------------------------------------------
# Stage-2 feature front end  (pinned by the reference)
# --------------------------------------------------------------------------------------
def erb_filterbank(nfreqs: int = 257, sample_rate: int = 16000, bands: int = 32,
                   low_freq: float = 0, max_freq: float = 8000) -> np.ndarray:
    """Cosine ERB bands [nfreqs, bands] as returned by
    ``EquivalentRectangularBandwidth(...).filters`` (network/ERB.py:10-71): only
    the cosine columns are returned; the low/high-pass columns the reference
    builds are dropped at ERB.py:71.  ``low_freq``/``max_freq`` of ``None``
    default to 20 Hz / Nyquist (ERB.py:12-15); the live config passes 0 / 8000
    (configs.py:21-27)."""
    if low_freq is None:
        low_freq = 20
    if max_freq is None:
        max_freq = sample_rate // 2
    ear_q, min_bw = 9.265, 24.7

    def hz_to_erb(f):
        return ear_q * np.log(1 + f / (min_bw * ear_q))

    def erb_to_hz(e):
        return (np.exp(e / ear_q) - 1) * min_bw * ear_q

    hz = np.linspace(0, max_freq, nfreqs)
    edges = erb_to_hz(np.linspace(hz_to_erb(low_freq), hz_to_erb(max_freq), bands + 2))
    bank = np.zeros((nfreqs, bands))
    for b in range(bands):
        lo, hi = edges[b], edges[b + 2]
        first = int(np.nonzero(hz > lo)[0].min())
        last = int(np.nonzero(hz < hi)[0].max())
        centre = 0.5 * (hz_to_erb(lo) + hz_to_erb(hi))
        width = hz_to_erb(hi) - hz_to_erb(lo)
        sl = slice(first, last + 1)
        bank[sl, b] = np.cos((hz_to_erb(hz[sl]) - centre) / width * np.pi)
    return bank


def stage2_features(mic: np.ndarray, ref: np.ndarray, erb: np.ndarray,
                    frame: int = WIN_SIZE, hop: int = HOP_SIZE, dtype=np.float64,
                    in_norm: bool = True) -> np.ndarray:
    """Feature tensor the Stage-2 net is fed (network/ERB.py:254-290), [B, T, 2*bands]:
    batch-global shift ``x - mean(x)/std(x)`` (unbiased std, torch default; ERB.py:254-255),
    complex STFT (ERB.py:263-264), ``sqrt(re^2 + im^2 + 1e-9)`` (ERB.py:277-278),
    ``@ erb`` (ERB.py:282-283), ``cat[mic_erb, |mic_erb - ref_erb|]`` (ERB.py:287-290)."""
    mic = np.atleast_2d(np.asarray(mic, dtype=dtype))
    ref = np.atleast_2d(np.asarray(ref, dtype=dtype))
    erb = np.asarray(erb, dtype=dtype)
    if in_norm:
        mic = mic - mic.mean() / mic.std(ddof=1)
        ref = ref - ref.mean() / ref.std(ddof=1)
    out = []
    for x in (mic, ref):
        s = stft_complex(x, frame, hop, dtype)
        mag = np.sqrt(s.real ** 2 + s.imag ** 2 + dtype(1e-9))
        out.append(mag.astype(dtype) @ erb)
    mic_erb, ref_erb = out
    return np.concatenate([mic_erb, np.abs(mic_erb - ref_erb)], axis=2)


def stage2_little_net(mic: np.ndarray, ref: np.ndarray, erb: np.ndarray, w: dict,
                      frame: int = WIN_SIZE, hop: int = HOP_SIZE, dtype=np.float64,
                      in_norm: bool = True) -> np.ndarray:
    """Inference path of the reference's live Stage-2 model ``Little_net.forward``
    (network/ERB.py:252-316; pinned by tests/golden/reference_stage2.npz, produced by running the
    reference module itself).  ``w`` holds the state_dict arrays ``gru1_weight_ih_l0`` [96,64],
    ``gru1_weight_hh_l0`` [96,32], ``gru1_bias_ih_l0``, ``gru1_bias_hh_l0`` (PyTorch gate order r, z, n),
    ``linear1_weight`` [32,64], ``linear1_bias``, ``linear2_weight`` [32,32], ``linear2_bias``.
    ``in_norm=False`` skips the batch-global shift (as ``stage2_features`` does): each row is then independent of the
    others.  Returns ``out_wav`` [B, (T-1)*hop]."""
    mic = np.atleast_2d(np.asarray(mic, dtype=dtype))
    ref = np.atleast_2d(np.asarray(ref, dtype=dtype))
    erb = np.asarray(erb, dtype=dtype)
    g = {k: np.asarray(v, dtype=dtype) for k, v in w.items()}
    if in_norm:
        mic = mic - mic.mean() / mic.std(ddof=1)                           # ERB.py:254
        ref = ref - ref.mean() / ref.std(ddof=1)                           # ERB.py:255
    M = stft_complex(mic, frame, hop, dtype)                               # ERB.py:263
    R = stft_complex(ref, frame, hop, dtype)                               # ERB.py:264
    merb = np.sqrt(M.real ** 2 + M.imag ** 2 + 1e-9) @ erb                 # ERB.py:277, 282
    rerb = np.sqrt(R.real ** 2 + R.imag ** 2 + 1e-9) @ erb                 # ERB.py:278, 283
    x = np.concatenate([merb, np.abs(merb - rerb)], axis=2)                # ERB.py:287-290
    B, T, _ = x.shape
    nh = g["gru1_weight_hh_l0"].shape[1]
    sig = lambda v: 1.0 / (1.0 + np.exp(-v))                               # noqa: E731
    h = np.zeros((B, nh), dtype=dtype)
    out1 = np.zeros((B, T, nh), dtype=dtype)
    for t in range(T):                                                     # ERB.py:293 (torch.nn.GRU cell)
        gi = x[:, t] @ g["gru1_weight_ih_l0"].T + g["gru1_bias_ih_l0"]
        gh = h @ g["gru1_weight_hh_l0"].T + g["gru1_bias_hh_l0"]
        r = sig(gi[:, :nh] + gh[:, :nh])
        z = sig(gi[:, nh:2 * nh] + gh[:, nh:2 * nh])
        n = np.tanh(gi[:, 2 * nh:] + r * gh[:, 2 * nh:])
        h = (1.0 - z) * n + z * h
        out1[:, t] = h
    outcat = np.concatenate([out1, merb], axis=2)                          # ERB.py:295
    out2 = np.maximum(outcat @ g["linear1_weight"].T + g["linear1_bias"], 0.0)   # ERB.py:298
    mask = sig(out2 @ g["linear2_weight"].T + g["linear2_bias"])           # ERB.py:301
    est_erb = mask * merb                                                  # ERB.py:304
    gain = est_erb @ erb.T                                                 # ERB.py:306-307
    est = gain * M                                                         # ERB.py:309-310
    return istft_complex(est, frame, hop, dtype) + dtype(1e-9)             # ERB.py:315-316


# --------------------------------------------------------------------------------------
# algorithmic work (SURVEY.md section 8d) -- used by bench.py for the roofline
# --------------------------------------------------------------------------------------
def flops_per_frame(cfg: AecConfig) -> float:
    n, k, p = cfg.frame, cfg.bins, cfg.partitions
    if cfg.algo in (ALGO_PBFDAF, ALGO_PBFKF):     # per block: five real transforms (X, y, E, two of the constraint), no windows
        common = 12.5 * n * math.log2(n) + 2 * n
    else:
        common = 7.5 * n * math.log2(n) + 5 * n
    if cfg.algo in (ALGO_NLMS, ALGO_PBFDAF):
        return common + 16 * k * p + 12 * k
    return common + 31 * k * p + 11 * k


def bytes_per_audio_second(sample_rate: int, with_echo: bool = False) -> float:
    return (4 if with_echo else 3) * 4.0 * sample_rate
