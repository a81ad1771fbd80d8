"""Stateful form of ``aec_oracle.stage2_little_net(in_norm=False)``: Little_net run hop by hop.  TEST INFRASTRUCTURE
ONLY.

``little_net_stream(mic, ref, erb, w, state)`` consumes the whole hops of one chunk of ONE stream (``len // 256``; the
caller keeps the rest) and returns ``(out, state)``.  Frame t of the reference STFT covers hops t - 1 and t (hop -1 is
zero); output block g is the second half of frame g plus the first half of frame g + 1.  A chunk of n hops computes
frames T0 .. T0+n-1 and returns blocks T0-1 .. T0+n-2 (block -1 is not part of the signal).  The state holds, after
T frames (the layout the streaming kernel keeps, include/aec_b200.h):

    frames    T
    h         [32] the GRU state after frame T - 1
    mic_prev  [256] hop T - 1 of mic (zeros at T = 0)
    ref_prev  [256] hop T - 1 of ref
    ola       [256] the second half of frame T - 1 after the synthesis window and the overlap normalisation of
              ``istft_complex`` (divided by coff + 1e-8), without the + 1e-9

Each frame goes through the numpy calls of ``stage2_little_net`` on a one-row batch; fed one more hop after the end (the
last samples zero-padded), the concatenated output equals the whole-signal oracle to rounding (1e-12 relative).
"""
from __future__ import annotations

import numpy as np

from .aec_oracle import HOP_SIZE, WIN_SIZE, hann_periodic

H = HOP_SIZE
NH = 32


def init_state(dtype=np.float64) -> dict:
    return {"frames": 0, "h": np.zeros(NH, dtype=dtype), "mic_prev": np.zeros(H, dtype=dtype),
            "ref_prev": np.zeros(H, dtype=dtype), "ola": np.zeros(H, dtype=dtype)}


def little_net_stream(mic: np.ndarray, ref: np.ndarray, erb: np.ndarray, w: dict, state: dict = None,
                      dtype=np.float64):
    """One chunk of one stream.  ``w``: the state_dict arrays of ``stage2_little_net``.  ``state=None`` starts a stream;
    the state passed in is not modified."""
    mic = np.asarray(mic, dtype=dtype).reshape(-1)
    ref = np.asarray(ref, dtype=dtype).reshape(-1)
    erb = np.asarray(erb, dtype=dtype)
    g = {k: np.asarray(v, dtype=dtype) for k, v in w.items()}
    st = init_state(dtype) if state is None else {k: (np.array(v, dtype=dtype) if k != "frames" else int(v))
                                                 for k, v in state.items()}
    win = hann_periodic(WIN_SIZE, dtype)
    w2 = win * win
    coff = (np.zeros(H, dtype=dtype) + w2[H:]) + w2[:H]          # istft_complex's overlap sum at every kept sample
    norm = coff + dtype(1e-8)
    sig = lambda v: 1.0 / (1.0 + np.exp(-v))                      # noqa: E731
    h = st["h"][None, :]
    out = []
    for i in range(len(mic) // H):
        m_hop, r_hop = mic[i * H:(i + 1) * H], ref[i * H:(i + 1) * H]
        M = np.fft.rfft((np.concatenate([st["mic_prev"], m_hop]) * win)[None, :], axis=-1)
        R = np.fft.rfft((np.concatenate([st["ref_prev"], r_hop]) * win)[None, :], axis=-1)
        merb = np.sqrt(M.real ** 2 + M.imag ** 2 + 1e-9) @ erb
        rerb = np.sqrt(R.real ** 2 + R.imag ** 2 + 1e-9) @ erb
        x = np.concatenate([merb, np.abs(merb - rerb)], axis=1)
        gi = x @ g["gru1_weight_ih_l0"].T + g["gru1_bias_ih_l0"]
        gh = h @ g["gru1_weight_hh_l0"].T + g["gru1_bias_hh_l0"]
        r = sig(gi[:, :NH] + gh[:, :NH])
        z = sig(gi[:, NH:2 * NH] + gh[:, NH:2 * NH])
        n = np.tanh(gi[:, 2 * NH:] + r * gh[:, 2 * NH:])
        h = (1.0 - z) * n + z * h
        out2 = np.maximum(np.concatenate([h, merb], axis=1) @ g["linear1_weight"].T + g["linear1_bias"], 0.0)
        mask = sig(out2 @ g["linear2_weight"].T + g["linear2_bias"])
        est = ((mask * merb) @ erb.T) * M
        fr = (np.fft.irfft(est, n=WIN_SIZE, axis=-1).astype(dtype) * win)[0]
        if st["frames"] > 0:
            out.append(st["ola"] + fr[:H] / norm + dtype(1e-9))
        st["ola"] = fr[H:] / norm
        st["mic_prev"], st["ref_prev"] = m_hop.copy(), r_hop.copy()
        st["frames"] += 1
    st["h"] = h[0].copy()
    return (np.concatenate(out) if out else np.zeros(0, dtype=dtype)), st
