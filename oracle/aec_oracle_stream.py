"""Stateful form of ``aec_oracle.pbfdaf_ols``: the overlap-save filter run chunk by chunk.  TEST INFRASTRUCTURE ONLY.

``pbfdaf_ols_stream(far, mic, cfg, state)`` consumes the whole blocks of one chunk (``len // hop``; the caller keeps
the rest) and returns ``(err, yhat, state)``.  The state holds the quantities of ``pbfdaf_ols`` after the last
block consumed, in its rfft convention (the layout the streaming kernels keep, include/aec_b200.h):

    blocks  T, blocks consumed since init
    prev    x_{T-1}, the far-end samples of the last consumed block (zeros at T = 0)
    W       [P, K] taps by partition, after the update with E_{T-1}
    X       [P, K] X[p] = rfft([x_{T-2-p}, x_{T-1-p}])
    Pw      [K] (algo 2)        Psi [K], C [P, K] (algo 3)

The block loop is ``pbfdaf_ols``'s, operation for operation, with the block index T = blocks + t where the partition
constrained in a block depends on it; chunked runs therefore equal one run over the whole signal exactly.
"""
from __future__ import annotations

import numpy as np

from .aec_oracle import ALGO_PBFKF, AecConfig, _cdtype


def init_state(cfg: AecConfig, dtype=np.float64) -> dict:
    cd = _cdtype(dtype)
    P, H = cfg.partitions, cfg.hop
    K = H + 1
    st = {"blocks": 0, "prev": np.zeros(H, dtype=dtype), "W": np.zeros((P, K), dtype=cd),
          "X": np.zeros((P, K), dtype=cd)}
    if cfg.algo == ALGO_PBFKF:
        st["Psi"] = np.zeros(K, dtype=dtype)
        st["C"] = np.full((P, K), cfg.kalman_c0, dtype=dtype)
    else:
        st["Pw"] = np.zeros(K, dtype=dtype)
    return st


def pbfdaf_ols_stream(far: np.ndarray, mic: np.ndarray, cfg: AecConfig, state: dict = None, dtype=np.float64):
    """One chunk of one stream.  ``state=None`` starts a stream; the state passed in is not modified."""
    cd = _cdtype(dtype)
    far = np.asarray(far, dtype=dtype)
    mic = np.asarray(mic, dtype=dtype)
    N, H, P = cfg.frame, cfg.hop, cfg.partitions
    kalman = cfg.algo == ALGO_PBFKF
    st = init_state(cfg, dtype) if state is None else state
    T0 = int(st["blocks"])
    W = np.array(st["W"], dtype=cd)
    Xh = np.array(st["X"], dtype=cd)
    prev = np.array(st["prev"], dtype=dtype)
    if kalman:
        psi = np.array(st["Psi"], dtype=dtype)
        C = np.array(st["C"], dtype=dtype)
    else:
        pw = np.array(st["Pw"], dtype=dtype)
    nblk = min(len(far), len(mic)) // H
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
        c = (T0 + t) % P
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
    out = {"blocks": T0 + nblk, "prev": np.array(prev, dtype=dtype), "W": W, "X": Xh}
    if kalman:
        out["Psi"], out["C"] = psi, C
    else:
        out["Pw"] = pw
    return err, yh, out
