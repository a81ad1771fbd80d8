"""Drop-in operators for the reference's STFT / iSTFT modules and Stage-2 feature front end.

    ConvSTFT   <-> Stage2_lhm/scripts/network/attention_ccrn.py:28-59
    ConviSTFT  <-> Stage2_lhm/scripts/network/attention_ccrn.py:62-101
    stage2_features <-> Stage2_lhm/scripts/network/ERB.py:254-290
    batch_shift     <-> the scalar mean/std of ERB.py:254-256 (device-side reduction, no host sync)
    erb_filterbank  <-> Stage2_lhm/scripts/network/ERB.py:10-71 (host-side table, numpy)

Same constructor arguments, same tensor layouts ([B, 2K, T] real-over-imag; [B, 1, L']),
but the transform is the FFT kernel in ``libaec_b200.so`` instead of a dense
[2K x N] convolution.  Only what the live reference path uses is built: periodic Hann,
``fft_len == win_len``, ``win_inc == win_len // 2``, ``feature_type='complex'``; anything else
raises (no silent fallback to a torch implementation).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .stage1 import _disjoint_rows, _require_cuda_f32, _stream_ptr, num_frames


def _check_ctor(win_len, win_inc, fft_len, win_type, feature_type):
    if fft_len is None:
        fft_len = int(2 ** np.ceil(np.log2(win_len)))      # attention_ccrn.py:33 (np.int is gone)
    if win_type != "hann":
        raise NotImplementedError("libaec_b200 builds the reference's live window only: 'hann' (ERB.py:210)")
    if fft_len != win_len or win_inc * 2 != win_len:
        raise NotImplementedError("libaec_b200 needs fft_len == win_len and win_inc == win_len // 2 "
                                  "(the reference's live setting, configs.py:1-8)")
    if win_len not in (512, 1024):
        raise NotImplementedError("frame must be 512 or 1024")
    if feature_type != "complex":
        raise NotImplementedError("only feature_type='complex' is built (ERB.py:223-224)")
    return fft_len


class ConvSTFT(torch.nn.Module):
    """``ConvSTFT(win_len, win_inc, fft_len, 'hann', 'complex')``; forward [B, L] or [B, 1, L]
    float32 CUDA -> [B, 2K, T]."""

    def __init__(self, win_len, win_inc, fft_len=None, win_type="hann", feature_type="complex", fix=True):
        super().__init__()
        self.fft_len = _check_ctor(win_len, win_inc, fft_len, win_type, feature_type)
        self.win_len, self.stride, self.dim, self.feature_type = win_len, win_inc, self.fft_len, feature_type

    def forward(self, inputs: torch.Tensor) -> torch.Tensor:
        if inputs.dim() == 3:
            if inputs.shape[1] != 1:
                raise ValueError("expected [B, 1, L]")
            inputs = inputs[:, 0]
        _require_cuda_f32("inputs", inputs)
        if inputs.dim() != 2:
            raise ValueError("expected [B, L] or [B, 1, L]")
        x, stride = _disjoint_rows(inputs)
        B, L = x.shape
        T = num_frames(L, self.win_len)
        K = self.win_len // 2 + 1
        with torch.cuda.device(x.device):
            spec = torch.empty((B, 2 * K, T), dtype=torch.float32, device=x.device)
            rc = _lib.load().aec_stft(x.data_ptr(), spec.data_ptr(), B, L, stride, self.win_len, _stream_ptr(x))
        _lib.check(rc, "aec_stft")
        return spec


class ConviSTFT(torch.nn.Module):
    """``ConviSTFT(win_len, win_inc, fft_len, 'hann', 'complex')``; forward [B, 2K, T] -> [B, 1, (T-1)*hop]."""

    def __init__(self, win_len, win_inc, fft_len=None, win_type="hann", feature_type="complex", fix=True):
        super().__init__()
        self.fft_len = _check_ctor(win_len, win_inc, fft_len, win_type, feature_type)
        self.win_len, self.stride, self.dim, self.feature_type = win_len, win_inc, self.fft_len, feature_type

    def forward(self, inputs: torch.Tensor, phase=None) -> torch.Tensor:
        if phase is not None:
            raise NotImplementedError("magnitude/phase input is not used by the live reference path")
        _require_cuda_f32("inputs", inputs)
        K = self.win_len // 2 + 1
        if inputs.dim() != 3 or inputs.shape[1] != 2 * K:
            raise ValueError(f"expected [B, {2 * K}, T]")
        s = inputs.contiguous()
        B, _, T = s.shape
        n_out = max(T - 1, 0) * self.stride
        with torch.cuda.device(s.device):
            y = torch.empty((B, 1, n_out), dtype=torch.float32, device=s.device)
            if n_out > 0:
                rc = _lib.load().aec_istft(s.data_ptr(), y.data_ptr(), B, T, n_out, self.win_len, _stream_ptr(s))
                _lib.check(rc, "aec_istft")
        return y


def erb_filterbank(nfreqs=257, sample_rate=16000, total_erb_bands=32, low_freq=0, max_freq=8000) -> np.ndarray:
    """Cosine ERB bank [nfreqs, bands] (float64) -- the array ``EquivalentRectangularBandwidth(...).filters``
    holds (ERB.py:10-71; only the cosine columns survive ERB.py:71).  A host-side constant table,
    built once per run like the reference does in train1.py:145-148."""
    low_freq = 20 if low_freq is None else low_freq
    max_freq = sample_rate // 2 if max_freq is None else max_freq
    q, bw = 9.265, 24.7
    to_erb = lambda f: q * np.log(1 + f / (bw * q))          # noqa: E731
    to_hz = lambda e: (np.exp(e / q) - 1) * bw * q            # noqa: E731
    grid = np.linspace(0, max_freq, nfreqs)
    cut = to_hz(np.linspace(to_erb(low_freq), to_erb(max_freq), total_erb_bands + 2))
    bank = np.zeros((nfreqs, total_erb_bands))
    for i in range(total_erb_bands):
        lo, hi = cut[i], cut[i + 2]
        a = int(np.flatnonzero(grid > lo)[0])
        z = int(np.flatnonzero(grid < hi)[-1])
        mid = (to_erb(lo) + to_erb(hi)) / 2
        span = to_erb(hi) - to_erb(lo)
        bank[a:z + 1, i] = np.cos((to_erb(grid[a:z + 1]) - mid) / span * np.pi)
    return bank


def batch_shift(x: torch.Tensor, out: torch.Tensor = None) -> torch.Tensor:
    """The scalar ``x.mean() / x.std()`` over the WHOLE batch tensor that ERB.py:254-256 subtracts, computed by
    ``aec_batch_shift`` and left on the device (a 1-element float32 CUDA tensor): no host synchronisation."""
    _require_cuda_f32("x", x)
    if x.dim() != 2 or x.stride(1) != 1:
        raise ValueError("x must be [B, L] with unit inner stride")
    x, stride = _disjoint_rows(x)
    lib = _lib.load()
    with torch.cuda.device(x.device):
        if out is None:
            out = torch.empty(1, dtype=torch.float32, device=x.device)
        nbytes = int(lib.aec_batch_shift_workspace_bytes())
        ws = torch.empty(nbytes // 8, dtype=torch.float64, device=x.device)
        B, L = x.shape
        rc = lib.aec_batch_shift(x.data_ptr(), B, L, stride, out.data_ptr(), ws.data_ptr(), nbytes, _stream_ptr(x))
    _lib.check(rc, "aec_batch_shift")
    return out


def stage2_features(mic: torch.Tensor, ref: torch.Tensor, erb: torch.Tensor, frame: int = 512,
                    in_norm: bool = True, shifts=None) -> torch.Tensor:
    """Feature tensor fed to the Stage-2 GRU: ``cat[mic_erb, |mic_erb - ref_erb|]`` [B, T, 2*bands]
    (ERB.py:254-290) in ONE kernel: no [B, 514, T] spectra are materialised.  ``mic`` would be the
    stage-1 error signal in a two-stage pipeline; ``erb`` is [257, bands] float32 on the device."""
    _require_cuda_f32("mic", mic)
    _require_cuda_f32("ref", ref)
    _require_cuda_f32("erb", erb)
    if mic.shape != ref.shape or mic.dim() != 2:
        raise ValueError("mic and ref must be [B, L]")
    mic, ref, erb = mic.contiguous(), ref.contiguous(), erb.contiguous()
    B, L = mic.shape
    K = frame // 2 + 1
    if erb.shape[0] != K:
        raise ValueError(f"erb must be [{K}, bands]")
    bands = erb.shape[1]
    # ERB.py:254-255 subtract the batch-global scalar mean/std (torch.std is unbiased): reduced on the device and
    # handed to the feature kernel by device pointer -- the call stays asynchronous (``shifts`` = precomputed pair)
    if shifts is not None:
        sm, sr = shifts
    elif in_norm:
        sm, sr = batch_shift(mic), batch_shift(ref)
    else:
        sm = sr = None
    T = num_frames(L, frame)
    with torch.cuda.device(mic.device):
        feat = torch.empty((B, T, 2 * bands), dtype=torch.float32, device=mic.device)
        rc = _lib.load().aec_features_dev(mic.data_ptr(), ref.data_ptr(), erb.data_ptr(), feat.data_ptr(), B, L, L,
                                          frame, bands, sm.data_ptr() if sm is not None else None,
                                          sr.data_ptr() if sr is not None else None, _stream_ptr(mic))
    _lib.check(rc, "aec_features_dev")
    return feat
