"""Float64 numpy oracle of the far-end delay estimator and the far-end shift (builder-authored; frozen here).

Per utterance b with n = n_b samples, D = ``max_delay`` (a power of two, 256 <= D <= 8192), M = 2D, and the far end
x~ / microphone y~ zero outside [0, n):

    blocks s = 0 .. ceil(n / D) - 1
    X_s = rfft_M( x~[(s-1)D : (s+1)D] )          previous and current far-end block
    Y_s = rfft_M( [0_D, y~[sD : (s+1)D]] )        current mic block, zero first half
    S[k] = sum_s Y_s[k] conj(X_s[k])              k = 0 .. D
          -> irfft_M(S)[l] = sum_n y~[n] x~[n-l] exactly, l = 0 .. D   (linear cross-correlation)
    G[k] = S[k] / |S[k]|  (0 where S[k] = 0);  G[0] = G[D] = 0       (PHAT weighting, DC and Nyquist dropped)
    r[l] = irfft_M(G)[l],  l = 0 .. D                                  (|r| <= 1)
    delay = smallest l with |r[l]| = max |r|      peak = |r[delay]|
    shift = peak >= min_peak ? max(0, delay - margin) : 0
    far_aligned[n] = far[n - shift] for n >= shift, 0 below

The blocking is that of the overlap-save filter (``aec_oracle.pbfdaf_ols``: previous and current block in, a block
zero-padded at the front out): with the mic block in the second half of the window, every product x~[m] y~[n] with
0 <= n - m <= D lands in exactly one block's circular correlation at lag n - m, and no other product reaches lags
0..D, so r[0..D] of S is the linear cross-correlation.

``dtype=np.float32`` runs the same arithmetic in float32 (scipy.fft keeps single precision), to measure how far
float32 rounding alone moves the outputs on a given row.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import scipy.fft as sfft


@dataclass(frozen=True)
class DelayConfig:
    max_delay: int = 8192      # D: largest lag searched, a power of two in [256, 8192]
    margin: int = 128          # samples of the echo path left before the estimated delay
    min_peak: float = 0.1      # normalised PHAT peak below which no shift is applied


def _blocks(far: np.ndarray, mic: np.ndarray, D: int, dtype):
    n = far.shape[0]
    nblk = -(-n // D)
    xp = np.zeros((nblk + 1) * D, dtype=dtype)
    xp[D:D + n] = far
    yp = np.zeros(nblk * D, dtype=dtype)
    yp[:n] = mic
    xw = np.lib.stride_tricks.sliding_window_view(xp, 2 * D)[::D][:nblk]
    yw = np.zeros((nblk, 2 * D), dtype=dtype)
    yw[:, D:] = yp.reshape(nblk, D)
    return xw, yw


def cross_spectrum(far: np.ndarray, mic: np.ndarray, D: int, dtype=np.float64) -> np.ndarray:
    """S[0..D] of one utterance (1-D arrays of its n samples)."""
    far = np.asarray(far, dtype=dtype)
    mic = np.asarray(mic, dtype=dtype)
    if far.shape[0] == 0:
        return np.zeros(D + 1, dtype=np.complex128 if dtype == np.float64 else np.complex64)
    xw, yw = _blocks(far, mic, D, dtype)
    X = sfft.rfft(xw, axis=1)
    Y = sfft.rfft(yw, axis=1)
    return (Y * np.conj(X)).sum(axis=0)


def phat_correlation(S: np.ndarray, D: int) -> np.ndarray:
    """r[0..D] of the PHAT-weighted cross-spectrum."""
    a = np.abs(S)
    G = np.zeros_like(S)
    nz = a > 0
    G[nz] = S[nz] / a[nz]
    G[0] = 0
    G[D] = 0
    return sfft.irfft(G, 2 * D)[:D + 1]


def estimate(far: np.ndarray, mic: np.ndarray, cfg: DelayConfig = DelayConfig(), n_samples=None,
             dtype=np.float64):
    """far, mic: [B, L] (or [L]).  Returns dict(delay int32 [B], shift int32 [B], peak [B], corr [B][D+1])."""
    far = np.atleast_2d(np.asarray(far))
    mic = np.atleast_2d(np.asarray(mic))
    B, L = far.shape
    D = int(cfg.max_delay)
    if n_samples is None:
        n_samples = [L] * B
    delay = np.zeros(B, dtype=np.int32)
    shift = np.zeros(B, dtype=np.int32)
    peak = np.zeros(B, dtype=np.float64)
    corr = np.zeros((B, D + 1), dtype=np.float64)
    for b in range(B):
        n = min(max(int(n_samples[b]), 0), L)
        r = phat_correlation(cross_spectrum(far[b, :n], mic[b, :n], D, dtype), D)
        a = np.abs(r)
        d = int(np.argmax(a))                 # first index of the maximum: ties go to the smaller lag
        delay[b] = d
        peak[b] = a[d]
        corr[b] = r
        shift[b] = max(0, d - int(cfg.margin)) if a[d] >= cfg.min_peak else 0
    return {"delay": delay, "shift": shift, "peak": peak, "corr": corr}


def align(far: np.ndarray, shift) -> np.ndarray:
    """far_aligned[b, n] = far[b, n - shift[b]] for n >= shift[b], 0 below (rows keep their length)."""
    far = np.atleast_2d(np.asarray(far))
    out = np.zeros_like(far)
    L = far.shape[1]
    for b, s in enumerate(np.asarray(shift).reshape(-1)):
        s = max(int(s), 0)
        if s < L:
            out[b, s:] = far[b, :L - s]
    return out


def linear_xcorr(far: np.ndarray, mic: np.ndarray, D: int) -> np.ndarray:
    """sum_n y[n] x[n-l], l = 0..D, by the direct time-domain sum (what irfft_M(S)[0..D] must equal)."""
    x = np.asarray(far, dtype=np.float64)
    y = np.asarray(mic, dtype=np.float64)
    n = x.shape[0]
    return np.array([np.dot(y[l:], x[:n - l]) if l < n else 0.0 for l in range(D + 1)])
