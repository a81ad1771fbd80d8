"""Seeded synthetic far-end / RIR / near-end / microphone signals (SURVEY.md section 8d).

The reference ships no audio (only filelists of absolute paths on the authors'
machine, Stage2_lhm/examples/filelists/tr_list.txt), so every measurement and
parity test runs on these signals.  numpy's PCG64 generator is used (bit-stable
across machines) so the CPU box and the GPU box see identical inputs.

far-end : white Gaussian -> one-pole low-pass y[n] = 0.9 y[n-1] + x[n] -> 4 Hz raised-cosine
          amplitude modulation -> peak-scaled to 0.5                      (seed 1000 + u)
RIR     : g[n] exp(-n / tau), g ~ N(0,1), length = P*H, tau = length / 6.9, ||h||_2 = 0.5
                                                                          (seed 2000 + u)
echo    : far * h truncated to L; with bulk_delay = d the response starts after d zeros (the playback and
          capture latency of a real device), so the echo arrives d samples late
near-end: zero (single talk) or the far-end generator gated on [0.4 L, 0.7 L], SER = 0 dB
                                                                          (seed 3000 + u)
mic     : echo + near + white noise at -40 dB re echo                     (seed 4000 + u)
"""
from __future__ import annotations

import numpy as np
from scipy.signal import fftconvolve, lfilter


def _speechlike(rng: np.random.Generator, n: int, sample_rate: int) -> np.ndarray:
    x = rng.standard_normal(n)
    y = lfilter([1.0], [1.0, -0.9], x)
    t = np.arange(n) / float(sample_rate)
    env = 0.5 - 0.5 * np.cos(2.0 * np.pi * 4.0 * t)
    y = y * env
    return 0.5 * y / (np.abs(y).max() + 1e-12)


def make_rir(u: int, length: int) -> np.ndarray:
    rng = np.random.default_rng(2000 + u)
    tau = length / 6.9
    h = rng.standard_normal(length) * np.exp(-np.arange(length) / tau)
    return 0.5 * h / np.linalg.norm(h)


def make_utterance(u: int, n_samples: int, sample_rate: int = 16000, rir_len: int = 1024,
                   double_talk: bool = False, bulk_delay: int = 0):
    """Returns dict of float32 arrays: far, mic, echo, near (all [n_samples])."""
    far = _speechlike(np.random.default_rng(1000 + u), n_samples, sample_rate)
    h = make_rir(u, rir_len)
    if bulk_delay:
        h = np.concatenate([np.zeros(int(bulk_delay)), h])
    echo = fftconvolve(far, h)[:n_samples]
    near = np.zeros(n_samples)
    if double_talk:
        s = _speechlike(np.random.default_rng(3000 + u), n_samples, sample_rate)
        gate = np.zeros(n_samples)
        gate[int(0.4 * n_samples):int(0.7 * n_samples)] = 1.0
        s = s * gate
        pe = float((echo ** 2).mean())
        ps = float((s ** 2).sum() / max(gate.sum(), 1.0))
        near = s * np.sqrt(pe / (ps + 1e-20))
    noise = np.random.default_rng(4000 + u).standard_normal(n_samples)
    noise *= np.sqrt((echo ** 2).mean()) * 10.0 ** (-40.0 / 20.0)
    mic = echo + near + noise
    # keep |x| < 1 as wav-derived float32 data would be
    peak = max(np.abs(mic).max(), 1e-12)
    if peak >= 1.0:
        s = 0.99 / peak
        mic, echo, near = mic * s, echo * s, near * s
    f32 = np.float32
    return {"far": far.astype(f32), "mic": mic.astype(f32), "echo": echo.astype(f32),
            "near": near.astype(f32)}


def make_batch(first_u: int, batch: int, n_samples: int, sample_rate: int = 16000,
               rir_len: int = 1024, double_talk: bool = False, bulk_delay: int = 0):
    """Stacked [batch, n_samples] float32 arrays for utterances first_u .. first_u+batch-1."""
    keys = ("far", "mic", "echo", "near")
    out = {k: np.empty((batch, n_samples), dtype=np.float32) for k in keys}
    for i in range(batch):
        utt = make_utterance(first_u + i, n_samples, sample_rate, rir_len, double_talk, bulk_delay)
        for k in keys:
            out[k][i] = utt[k]
    return out
